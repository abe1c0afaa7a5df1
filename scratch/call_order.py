"""Records which library entry points GRUDecoder's paths call, in order, with their non-pointer arguments.

    python scratch/call_order.py OUT.json [OUTPUTS.json]

The loaded library is swapped for a recorder that forwards every call.  Per section (fp32 / bf16, bi- and unidirectional:
train_step padded and packed with dropout and input noise, eval_batch, input_attribution; bf16 unidirectional: a
StreamingDecoder run through its exact form into its fast form, once on fresh bf16 weight copies and once on current ones)
OUT.json gets [name, args...] per call, a pointer argument written as "p" (null: None).  OUTPUTS.json (optional) gets a
SHA-1 of the bytes of what each section returned.  Two commits that call the same kernels the same way give identical files.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import neural_speech_decoder_b200 as nsd  # noqa: E402
from neural_speech_decoder_b200 import _lib  # noqa: E402
from neural_speech_decoder_b200.synthetic import fill_trained_like_, make_batch  # noqa: E402


class Recorder:
    def __init__(self, lib):
        self._lib = lib
        self.calls = []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        types = _lib.SIGNATURES.get(name, (None, []))[1]

        def rec(*args):
            row = [name]
            for t, a in zip(types, args):
                if t is _lib.vp or not isinstance(a, (int, float)) or a is None:
                    row.append(None if a is None else "p")
                else:
                    row.append(round(a, 7) if isinstance(a, float) else a)
            self.calls.append(row)
            return fn(*args)
        return rec


def digest(*ts):
    h = hashlib.sha1()
    for t in ts:
        if isinstance(t, torch.Tensor):
            h.update(t.detach().float().cpu().contiguous().numpy().tobytes())
        else:
            h.update(repr(t).encode())
    return h.hexdigest()


def main():
    out, outputs = sys.argv[1], (sys.argv[2] if len(sys.argv) > 2 else None)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rec = Recorder(_lib.lib())
    _lib._lib = rec
    calls, hashes = {}, {}

    def section(key, fn):
        torch.cuda.synchronize()
        rec.calls = []
        res = fn()
        torch.cuda.synchronize()
        calls[key] = rec.calls
        hashes[key] = digest(*(res if isinstance(res, tuple) else (res,)))

    kw = dict(neural_dim=32, n_classes=10, hidden_dim=64, layer_dim=3, nDays=4, dropout=0.3, strideLen=4, kernelLen=16,
              gaussianSmoothWidth=2.0)
    args = dict(lrStart=0.02, lrEnd=0.02, nBatch=10, l2_decay=1e-5)
    X, y, X_len, y_len, day = [t.to(dev) for t in make_batch(4, 72, n_feat=32, n_days=4, n_classes=10, seed=5, ragged=True,
                                                             min_tgt=2, max_tgt=6, kernel_len=16, stride_len=4)]
    for precision in ("fp32", "bf16"):
        for bi in (True, False):
            nsd.set_default_precision(precision)
            torch.manual_seed(0)
            m = nsd.GRUDecoder(device="cuda", bidirectional=bi, **kw)
            nsd.set_default_precision("fp32")
            fill_trained_like_(m, seed=3)
            m = m.to(dev).train()
            opt, sched = nsd.make_optimizer(m, args)
            tag = f"{precision}-{'bi' if bi else 'uni'}"
            for packed in (False, True):
                def step():
                    loss = nsd.train_step(m, opt, X, y, X_len, y_len, day, sched, white_noise_sd=0.1, constant_offset_sd=0.05,
                                          packed=packed)
                    return (loss,) + tuple(p for p in m.parameters())
                section(f"{tag}/train_step packed={packed}", step)
            m.eval()
            section(f"{tag}/eval_batch", lambda: nsd.eval_batch(m, X, y, X_len, y_len, day))
            section(f"{tag}/input_attribution", lambda: nsd.input_attribution(m, X, y, X_len, y_len, day))

    skw = dict(neural_dim=32, n_classes=10, hidden_dim=512, layer_dim=2, nDays=4, dropout=0.0, strideLen=4, kernelLen=16,
               gaussianSmoothWidth=2.0, bidirectional=False)
    nsd.set_default_precision("bf16")
    torch.manual_seed(0)
    sm = nsd.GRUDecoder(device="cuda", **skw)
    nsd.set_default_precision("fp32")
    fill_trained_like_(sm, seed=4)
    sm = sm.to(dev).eval()
    Xs, _, _, _, ds = make_batch(2, 120, n_feat=32, n_days=4, n_classes=10, seed=7, kernel_len=16, stride_len=4)
    Xs, ds = Xs.to(dev), ds.to(dev)
    for copies in ("fresh", "current"):          # fresh: the model's bf16 weight copies are made by the first exact-form call
        def stream():
            sd = nsd.StreamingDecoder(sm, 2, ds)
            outs = [sd.push(Xs[:, :37])]             # exact form, several frames
            for pos in range(37, 117, 4):            # one stride per push: enters the fast form
                outs.append(sd.push(Xs[:, pos:pos + 4]))
            outs.append(sd.push(Xs[:, 117:]))
            outs.append(sd.finish())
            assert sd.fast and sd._graph is not None
            return tuple(o for o in outs if o is not None)
        section(f"stream ({copies} weight copies)", stream)

    json.dump(calls, open(out, "w"), indent=0)
    if outputs:
        json.dump(hashes, open(outputs, "w"), indent=1)
    print(json.dumps({k: len(v) for k, v in calls.items()}))


if __name__ == "__main__":
    main()
