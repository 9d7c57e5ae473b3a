#!/usr/bin/env python
"""Writes tests/golden/parsing_checkpoint.npz from the face-parsing checkpoint the reference ships.

    python oracle/make_golden_parsing_checkpoint.py <reference checkout>

The checkpoint (pretrained_ckpts/auxiliray/model.pth, 7.8 MB) is too large to keep in the repository.  What the tests need
from it is stored instead: the key / shape layout of all 136 entries (what a strict state-dict load checks) and the values of
the encoder's first two stages, `conv1` and `conv2` (17 k numbers).  The parsing features at those two depths depend on
nothing else, so they are compared with the reference's own features in tests/golden/loss_vectors.npz (written by
oracle/make_golden_losses.py with the whole checkpoint); this script asserts that they agree before it writes the file.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import loss_oracle as LO  # noqa: E402

STORED_STAGES = ("conv1.", "conv2.")
TOL = 2e-5


def main(ref: str) -> None:
    sd = torch.load(os.path.join(ref, "pretrained_ckpts", "auxiliray", "model.pth"), map_location="cpu")
    out = {}
    for k, v in sd.items():
        out["shape/" + k] = np.asarray(v.shape, dtype=np.int64)
        if k.startswith(STORED_STAGES):
            out["value/" + k] = v.numpy()

    # the stages not stored take the seeded stand-in values the tests use; the features at the stored depths do not see them
    seeded = LO.loss_states(11)["parsing"]
    partial = {"G." + k: (v if k.startswith(STORED_STAGES) else seeded["G." + k]) for k, v in sd.items()}
    gold = np.load(os.path.join(ROOT, "tests", "golden", "loss_vectors.npz"))
    img, _, _ = LO.golden_inputs()
    with torch.no_grad():
        feats = LO.parsing_extract_feats(partial, img)
    for i in range(len(STORED_STAGES)):
        ref_f = torch.from_numpy(gold[f"parsing_shipped/feats{i}"]).double()
        e = float((feats[i][:, :4096].double() - ref_f).abs().max() / ref_f.abs().max())
        print(f"parsing feats {i} with the stored stages vs the reference with the whole checkpoint: {e:.2e}")
        assert e <= TOL, (i, e)

    dst = os.path.join(ROOT, "tests", "golden", "parsing_checkpoint.npz")
    np.savez_compressed(dst, **out)
    print(f"wrote {dst} ({os.path.getsize(dst) / 1e3:.0f} kB, {len(out)} arrays)")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
