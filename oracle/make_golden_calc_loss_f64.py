#!/usr/bin/env python
"""Writes tests/golden/calc_loss_f64.npz: the reference's calc_loss and its gradient with respect to the reconstruction, in
float64.

    python oracle/make_golden_calc_loss_f64.py <reference checkout>

The loss networks and the unmodified source text of Optimizer.calc_loss (scripts/optimization.py:88-122) are set up as in
oracle/make_golden_losses.py, then run in float64.  The losses are 1 - cosine of nearly parallel feature vectors, so in fp32
their gradient depends on the host's summation order.  The script prints the oracle's fp32 gradient at 1, 8 and 64 CPU
threads against this float64 one and against the fp32 gradient of loss_vectors.npz (max-norm, on an 8-core host: with
AVX-512 kernels 5.7e-4 from float64 at every count and 8e-8 / 0 / 1.5e-4 from loss_vectors.npz, which was made there at 8
threads; with AVX2 kernels 7e-6 from float64 and 5.7e-4 from loss_vectors.npz).  In float64 the host does not matter, so
the oracle's gradient is compared with this one.  Stored: the loss, its terms, and every 4th pixel of the
gradient (rounded to float32).
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TOL = 1e-9


def main(ref: str) -> None:
    sys.path.insert(0, ref)
    from oracle import loss_oracle as LO, make_golden_losses as MG
    MG.REF = ref
    torch.manual_seed(0)
    states = LO.loss_states(salt=11)
    lp, idl, fp_seed, _, _ = MG.build_reference(states)
    calc = MG.reference_calc_loss()
    stub = types.SimpleNamespace(opts=types.SimpleNamespace(id_lambda=0.1, l2_lambda=1.0, lpips_lambda=0.8, face_parsing_lambda=0.1),
                                 id_loss=idl.double(), lpips_loss=lp.double(), face_parsing_loss=fp_seed.double())
    img, recon, _ = LO.golden_inputs()
    img, recon = img[:1].double(), recon[:1].double()
    r_ref = recon.clone().requires_grad_(True)
    loss_ref, dict_ref, _ = calc(stub, img, r_ref, None)
    loss_ref.backward()

    st64 = {n: {k: v.double() if v.is_floating_point() else v for k, v in d.items()} for n, d in states.items()}
    r_or = recon.clone().requires_grad_(True)
    loss_or, terms = LO.calc_loss(st64, img, r_or)
    loss_or.backward()

    def rel(a, b):
        a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
        return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))

    out = {"loss": np.float64(loss_ref.item())}
    checks = [("loss", loss_or, loss_ref.detach())]
    for k in ("loss_id", "loss_l2", "loss_lpips", "loss_face_parsing"):
        out[k] = np.float64(dict_ref[k])
        checks.append((k, terms[k].detach(), torch.tensor(dict_ref[k], dtype=torch.float64)))
    checks.append(("grad_recon", r_or.grad, r_ref.grad))
    for name, a, b in checks:
        e = rel(a, b)
        print(f"{name:20s} oracle vs reference (float64): {e:.2e}")
        assert e <= TOL, (name, e)
    out["grad_recon"] = r_ref.grad[:, :, ::4, ::4].float().numpy()

    # why the comparison is made in float64: the oracle's fp32 gradient against this one and against the fp32 gradient of
    # loss_vectors.npz, at three CPU thread counts
    g32 = np.load(os.path.join(ROOT, "tests", "golden", "loss_vectors.npz"))["calc_loss/grad_recon"]
    threads = torch.get_num_threads()
    for n in (1, 8, 64):
        torch.set_num_threads(n)
        r32 = recon.float().requires_grad_(True)
        loss32, _ = LO.calc_loss(states, img.float(), r32)
        loss32.backward()
        g = r32.grad[:, :, ::4, ::4]
        print(f"fp32 gradient at {n:2d} CPU threads: max-rel {rel(g, out['grad_recon']):.2e} vs float64, "
              f"{rel(g, g32):.2e} vs loss_vectors.npz")
    torch.set_num_threads(threads)

    dst = os.path.join(ROOT, "tests", "golden", "calc_loss_f64.npz")
    np.savez_compressed(dst, **out)
    print(f"wrote {dst} ({os.path.getsize(dst) / 1e3:.0f} kB, {len(out)} arrays)")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
