"""The float64 forced alignment (tests/ctc_align_oracle.py) against brute force over every valid CTC alignment, the exact CTC
likelihood and torchaudio's ``forced_align``.  CPU only."""
import numpy as np
import pytest

from ctc_align_oracle import align_batch, ctc_viterbi, lattice, min_frames
from oracle import nsd_oracle as O


def log_probs(rng, T, C, scale=2.0):
    return O.log_softmax(rng.standard_normal((T, C)) * scale)


def valid_alignments(T, C, target, blank):
    """Every frame-label sequence of length T whose CTC collapse (merge repeats, drop blanks) is ``target``."""
    L = len(target)
    out = []

    def walk(prefix, n, last):
        if len(prefix) == T:
            if n == L:
                out.append(tuple(prefix))
            return
        for c in range(C):
            if c == blank:
                walk(prefix + [c], n, c)
            elif c == last:
                walk(prefix + [c], n, c)
            elif n < L and c == target[n]:
                walk(prefix + [c], n + 1, c)
    walk([], 0, None)
    return out


def collapse(labels, blank):
    out, prev = [], None
    for c in labels:
        if c != prev and c != blank:
            out.append(int(c))
        prev = c
    return out


def check_path(states, ext, skip, il):
    S = len(ext)
    assert len(states) == il and states[0] in (0, 1) and states[-1] in (S - 1, S - 2)
    for a, b in zip(states[:-1], states[1:]):
        assert b - a in (0, 1) or (b - a == 2 and skip[b]), (a, b)


# (C, T, target): repeats, L = 0, il exactly at the minimum, blank at 0 and elsewhere
TARGETS = {(3, 0): ([], [1], [1, 1], [1, 2], [1, 1, 1], [2, 1, 2]),
           (4, 0): ([], [1], [1, 1], [1, 3], [1, 1, 1], [3, 1, 3]),
           (4, 2): ([], [1], [1, 1], [1, 3], [3, 3, 1], [3, 1, 3])}
BRUTE = [(C, T, tg, blank) for (C, blank), tgs in TARGETS.items() for tg in tgs
         for T in range(max(1, min_frames(np.array(tg), len(tg))), 9 if C == 3 else 8)]


@pytest.mark.parametrize("C,T,target,blank", BRUTE)
def test_brute_force(C, T, target, blank):
    rng = np.random.default_rng([C, T, blank] + target)
    for trial in range(3):
        lp = log_probs(rng, T, C, scale=[2.0, 0.5, 4.0][trial])
        if trial == 1:
            lp = np.round(lp, 1)                          # coarse values: exact ties between paths
        tg = np.array(target, dtype=np.int64)
        score, states, margin = ctc_viterbi(lp, tg, T, len(tg), blank)
        paths = valid_alignments(T, C, target, blank)
        assert paths
        scores = np.array([lp[np.arange(T), list(p)].sum() for p in paths])
        best = scores.max()
        assert abs(score - best) < 1e-12
        ext, skip = lattice(tg, len(tg), blank)
        check_path(states, ext, skip, T)
        labels = ext[states]
        assert collapse(labels, blank) == list(target)
        assert abs(lp[np.arange(T), labels].sum() - score) < 1e-12
        if (scores > best - 1e-9).sum() == 1:
            assert tuple(labels.tolist()) == paths[int(scores.argmax())]
            assert margin > 0
        else:
            assert margin < 1e-9                           # a tie somewhere on the path


def test_infeasible_and_empty():
    lp = log_probs(np.random.default_rng(0), 5, 4)
    assert ctc_viterbi(lp, np.array([1, 1, 1]), 4, 3)[:2] == (-np.inf, None)     # needs 5 frames
    s, st, _ = ctc_viterbi(lp, np.array([1, 1, 1]), 5, 3)
    assert st.tolist() == [1, 2, 3, 4, 5]
    assert ctc_viterbi(lp, np.zeros(0), 0, 0)[0] == 0.0
    s, st, _ = ctc_viterbi(lp, np.zeros(0), 5, 0)
    assert st.tolist() == [0] * 5 and abs(s - lp[:, 0].sum()) < 1e-12


@pytest.mark.parametrize("seed", range(6))
def test_batch_outputs_and_alpha_beta_bound(seed):
    rng = np.random.default_rng(seed)
    T, B, C = 40, 6, 7
    lp = np.stack([log_probs(rng, T, C) for _ in range(B)], axis=1)
    targets = rng.integers(1, C, (B, 12))
    targets[0, 1] = targets[0, 0]
    in_lens = np.array([40, 0, 1, 33, 25, 40])
    tgt_lens = np.array([12, 0, 1, 10, 0, 30])              # the last one is clamped to 12
    out = align_batch(lp, targets, in_lens, tgt_lens)
    for b in range(B):
        il, L = in_lens[b], min(tgt_lens[b], 12)
        lab = out["labels"][b]
        if out["score"][b] == -np.inf:
            assert (lab == -1).all() and (out["spans"][b] == -1).all()
            continue
        assert collapse(lab[:il], 0) == targets[b, :L].tolist() and (lab[il:] == -1).all()
        assert abs(out["frame_logp"][b].sum() - out["score"][b]) < 1e-10
        for k in range(L):
            f0, f1 = out["spans"][b, k]
            assert 0 <= f0 <= f1 < il and (lab[f0:f1 + 1] == targets[b, k]).all()
            assert abs(out["token_logp"][b, k] - out["frame_logp"][b, f0:f1 + 1].sum()) < 1e-12
        assert (out["spans"][b, L:] == -1).all() and (out["token_logp"][b, L:] == 0).all()
        nll, _, _ = O.ctc_alpha_beta(lp[:, b], targets[b], int(il), int(L), 0)
        assert out["score"][b] <= -nll + 1e-12
    assert out["score"][1] == 0.0 and (out["labels"][1] == -1).all()


def test_bad_target():
    lp = log_probs(np.random.default_rng(1), 10, 5)[:, None, :]
    for bad in (0, 5, -1):
        out = align_batch(lp, np.array([[1, bad, 2]]), [10], [3])
        assert out["bad"][0] and out["score"][0] == -np.inf and (out["labels"] == -1).all()
    assert not align_batch(lp, np.array([[1, 2, 5]]), [10], [2])["bad"][0]       # only the first L targets count


# ---------------------------------------------------------------------------------------------------- torchaudio
@pytest.mark.parametrize("seed", range(8))
def test_against_torchaudio(seed):
    torch = pytest.importorskip("torch")
    F = pytest.importorskip("torchaudio.functional")
    rng = np.random.default_rng(50 + seed)
    C = [5, 41][seed % 2]
    T = int(rng.integers(20, 120))
    L = int(rng.integers(1, T // 3))                  # torchaudio takes no empty target
    tg = rng.integers(1, C, L)
    if L > 2:
        tg[1] = tg[0]
    logits = rng.standard_normal((T, C)) * 6.0
    logits[:, 0] += 2.0
    lp = O.log_softmax(logits)
    score, states, margin = ctc_viterbi(lp, tg, T, L, 0)
    ta_lab, ta_sc = F.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(tg).int()[None], torch.tensor([T]), torch.tensor([L]), blank=0)
    assert abs(ta_sc.sum().item() - score) < 1e-12
    if margin > 1e-9:
        ext, _ = lattice(tg, L, 0)
        assert ext[states].tolist() == ta_lab[0].tolist()
