"""Record tests/golden/reference_init.json: the state dicts the reference's ``GRUDecoder`` (unidirectional and
bidirectional, torch seed 3) and ``NeuralTransformerCTCModel`` (torch seed 0) hold right after construction on the CPU,
each as [name, shape, dtype, SHA-256 of the bytes] in state-dict order, plus the parameter names.

tests/test_host.py checks that this package's modules, constructed under the same seeds, reproduce them bit for bit:
same constructor, same parameter and buffer names, same order of RNG draws, so that a reference checkpoint loads with
``strict=True`` and a seeded run starts from the reference's weights.  The file was recorded from this package's own
modules at a commit whose tests compared them with the reference's modules directly, tensor by tensor, in one process.
Rerun it only for a deliberate change of that contract:

    python tests/golden/make_golden_init.py
"""
from __future__ import annotations

import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import neural_speech_decoder_b200 as nsd  # noqa: E402
from test_host import CONFORMER_KW, KW, state_record  # noqa: E402


def record(seed, make):
    torch.manual_seed(seed)
    return state_record(make())


def main():
    out = {
        "gru_uni": record(3, lambda: nsd.GRUDecoder(device="cpu", **dict(KW, bidirectional=False))),
        "gru_bi": record(3, lambda: nsd.GRUDecoder(device="cpu", **dict(KW, bidirectional=True))),
        "conformer": record(0, lambda: nsd.NeuralTransformerCTCModel(device="cpu", **CONFORMER_KW)),
    }
    path = os.path.join(HERE, "reference_init.json")
    with open(path, "w") as f:                              # one line per tensor
        f.write("{\n" + ",\n".join(
            f'"{name}": {{"state": [\n' + ",\n".join(json.dumps(e) for e in rec["state"]) + f'\n], "parameters": {json.dumps(rec["parameters"])}}}'
            for name, rec in out.items()) + "\n}\n")
    print(f"wrote {path}: " + ", ".join(f"{k} {len(v['state'])} tensors" for k, v in out.items()))


if __name__ == "__main__":
    main()
