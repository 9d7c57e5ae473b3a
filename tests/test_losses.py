"""Loss networks of the inversion loop (SURVEY.md section 8 f1; scripts/optimization.py:88-122): the CPU oracle against the
reference-generated golden vectors (oracle/make_golden_losses.py), the product modules (e4s_b200.criteria) against both, and
the 3-step loss trajectory of the full-loss inversion loop against the oracle's loop."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import e4s_oracle as O
from oracle import loss_oracle as LO
from conftest import ROOT, assert_close

DEV = "cuda:0"
SALT = 11                                             # the salt oracle/make_golden_losses.py used


@pytest.fixture(scope="module")
def gold():
    d = np.load(os.path.join(ROOT, "tests", "golden", "loss_vectors.npz"))
    return {k: d[k] for k in d.files}


def _close(a, b, tol=2e-5, atol=0.0):
    a, b = float(a), float(b)
    assert abs(a - b) <= tol * max(abs(b), 1e-30) + atol, (a, b)


# The identity and parsing losses are sums over 5 scales of (1 - cosine) with cosines near 1 for a good reconstruction: a loss
# of 0.086 is a difference of numbers of size 5, so the 1e-3 bar is applied to that natural scale (absolute 2e-4 on the GPU,
# whose cuDNN fp32 convolutions may use Winograd transforms); the features themselves are compared at 1e-3.
COS_ATOL = 2e-4


# ------------------------------------------------------------------------------------------------- CPU: the oracle
def test_loss_oracle_matches_reference_vectors(gold):
    st = LO.loss_states(SALT)
    img, recon, far = LO.golden_inputs()
    with torch.no_grad():
        for tag, r in (("near", recon), ("far", far)):
            _close(LO.lpips(st["lpips"], r, img), gold[f"lpips/{tag}"])
            _close(LO.id_loss(st["id"], r, img), gold[f"id/{tag}"])
            _close(LO.parsing_loss(st["parsing"], r, img), gold[f"parsing_seeded/{tag}"])
        for i, f in enumerate(LO.id_extract_feats(st["id"], img)):
            assert_close(f[:, :4096], gold[f"id/feats{i}"], 2e-5, f"id feats {i}")


def test_shipped_parsing_checkpoint_layout_and_first_stages(gold):
    """The one loss network whose weights ship with the reference: its checkpoint's key / shape layout (which the seeded
    stand-in shares) loads strictly into the product module, and with the checkpoint's first two encoder stages
    (tests/golden/parsing_checkpoint.npz) the oracle's and the product module's features at those depths equal the
    reference's features with the whole checkpoint."""
    from e4s_b200.criteria import FaceParsingLoss
    ck = np.load(os.path.join(ROOT, "tests", "golden", "parsing_checkpoint.npz"))
    shapes = {k[len("shape/"):]: tuple(int(s) for s in ck[k]) for k in ck.files if k.startswith("shape/")}
    seeded = LO.loss_states(SALT)["parsing"]
    assert shapes == {k[len("G."):]: tuple(v.shape) for k, v in seeded.items()}
    sd = {k: torch.from_numpy(ck["value/" + k]) if "value/" + k in ck.files else seeded["G." + k] for k in shapes}
    m = FaceParsingLoss(types.SimpleNamespace())
    m.G.load_state_dict(sd, strict=True)
    img, _, _ = LO.golden_inputs()
    with torch.no_grad():
        oracle = LO.parsing_extract_feats({"G." + k: v for k, v in sd.items()}, img)
        ours = m.extract_feats(img)
    for i in range(2):
        assert_close(oracle[i][:, :4096], gold[f"parsing_shipped/feats{i}"], 2e-5, f"oracle parsing feats {i}")
        assert_close(ours[i][:, :4096], gold[f"parsing_shipped/feats{i}"], 2e-5, f"product parsing feats {i}")


def test_loss_oracle_calc_loss_matches_reference(gold):
    """calc_loss at the reference's own scales (1024 / 512 / 256): value, terms and the gradient the generator receives."""
    st = LO.loss_states(SALT)
    img, recon, _ = LO.golden_inputs()
    with torch.no_grad():
        loss, terms = LO.calc_loss(st, img[:1], recon[:1])
    _close(loss, gold["calc_loss/loss"])
    for k in ("loss_id", "loss_l2", "loss_lpips", "loss_face_parsing"):
        _close(terms[k], gold[f"calc_loss/{k}"])
    # the fp32 gradient (1 - cosine of nearly parallel features) moves with the host CPU's thread count and vector ISA: the
    # one in loss_vectors.npz is 5.7e-4 (max-norm) from the float64 gradient, another host's lands 1.5e-4 from it.  So it is
    # compared in float64 with the reference's float64 gradient (oracle/make_golden_calc_loss_f64.py prints these distances)
    g64 = np.load(os.path.join(ROOT, "tests", "golden", "calc_loss_f64.npz"))
    st64 = {n: {k: v.double() if v.is_floating_point() else v for k, v in d.items()} for n, d in st.items()}
    r64 = recon[:1].double().requires_grad_(True)
    loss64, terms64 = LO.calc_loss(st64, img[:1].double(), r64)
    loss64.backward()
    _close(loss64, g64["loss"], 1e-9)
    for k in ("loss_id", "loss_l2", "loss_lpips", "loss_face_parsing"):
        _close(terms64[k], g64[k], 1e-9)
    assert_close(r64.grad[:, :, ::4, ::4], g64["grad_recon"], 1e-6, "d calc_loss / d recon (float64)")


def test_product_loss_modules_state_dict_contract():
    """e4s_b200.criteria modules take the reference modules' state dicts (same keys and shapes), and the product's seeded
    stand-in weights equal the oracle's (with which the golden vectors were made)."""
    from e4s_b200.criteria import InversionLoss
    from e4s_b200.synthetic import synthetic_loss_state
    m = InversionLoss()
    st = LO.loss_states(SALT)
    for off, (name, key) in enumerate((("lpips_loss", "lpips"), ("id_loss", "id"), ("face_parsing_loss", "parsing"))):
        sub = getattr(m, name)
        sub.load_state_dict(st[key], strict=True)
        ours = synthetic_loss_state(sub, SALT + off)
        assert set(ours) == set(st[key])
        for k in ours:
            assert torch.equal(ours[k], st[key][k]), k


# ---------------------------------------------------------------------------------------------- GPU: the product
def conv_precision(exact):
    from e4s_b200.criteria.inversion_loss import conv_precision as cp
    return cp(exact)


def _criterion(**kw):
    from e4s_b200.criteria import InversionLoss
    from e4s_b200.synthetic import load_synthetic_losses
    m = InversionLoss(**kw)
    load_synthetic_losses(m, SALT)
    return m.to(DEV)


@pytest.mark.gpu
def test_pool_pyramid_kernel():
    from e4s_b200 import kernels as K
    g = torch.Generator().manual_seed(2)
    x = torch.randn(2, 3, 64, 96, generator=g).to(DEV).requires_grad_(True)
    y2, y4 = K.avgpool_pyramid(x.detach())
    assert_close(y2, torch.nn.functional.adaptive_avg_pool2d(x.detach(), (32, 48)), 1e-6, "2x2 means")
    assert_close(y4, torch.nn.functional.adaptive_avg_pool2d(x.detach(), (16, 24)), 1e-6, "4x4 means")
    from e4s_b200.criteria.inversion_loss import pyramid
    xs = torch.randn(1, 3, 128, 128, generator=g).to(DEV)
    a = xs.clone().requires_grad_(True)
    b = xs.clone().requires_grad_(True)
    w = [torch.randn(1, 3, s, s, generator=g).to(DEV) for s in (128, 64, 32)]
    sum((t * wi).sum() for t, wi in zip(pyramid(a, (128, 64, 32)), w)).backward()
    sum((torch.nn.functional.adaptive_avg_pool2d(b, (s, s)) * wi).sum() for s, wi in zip((128, 64, 32), w)).backward()
    assert_close(a.grad, b.grad, 1e-6, "pyramid backward")


@pytest.mark.gpu
def test_loss_modules_match_reference_vectors(gold):
    m = _criterion()
    img, recon, far = (t.to(DEV) for t in LO.golden_inputs())
    with torch.no_grad(), conv_precision(True):
        for tag, r in (("near", recon), ("far", far)):
            _close(m.lpips_loss(r, img), gold[f"lpips/{tag}"], 1e-3)
            _close(m.id_loss(r, img)[0], gold[f"id/{tag}"], 1e-3, COS_ATOL)
            _close(m.face_parsing_loss(r, img)[0], gold[f"parsing_seeded/{tag}"], 1e-3, COS_ATOL)
        for i, f in enumerate(m.face_parsing_loss.extract_feats(img)):
            ref = LO.parsing_extract_feats(LO.loss_states(SALT)["parsing"], img.cpu())[i]
            assert_close(f[:, :65536], ref[:, :65536], 1e-3, f"parsing feats {i}")
        for i, f in enumerate(m.id_loss.extract_feats(img)):
            assert_close(f[:, :4096], gold[f"id/feats{i}"], 1e-3, f"id feats {i}")


@pytest.mark.gpu
def test_inversion_loss_matches_reference_calc_loss(gold):
    """InversionLoss with the cached target == the reference's calc_loss (value, terms, gradient wrt the reconstruction)."""
    m = _criterion()
    img, recon, _ = (t.to(DEV) for t in LO.golden_inputs())
    m.set_target(img[:1])
    r = recon[:1].clone().requires_grad_(True)
    loss, terms = m(r, return_terms=True)
    loss.backward()
    _close(loss, gold["calc_loss/loss"], 1e-3)
    for k in ("loss_id", "loss_l2", "loss_lpips", "loss_face_parsing"):
        _close(terms[k], gold[f"calc_loss/{k}"], 1e-3, COS_ATOL if k in ("loss_id", "loss_face_parsing") else 0.0)
    assert_close(r.grad[:, :, ::4, ::4], gold["calc_loss/grad_recon"], 1e-3, "d loss / d recon")
    # 1024x1024 input: the fused pooling pyramid feeds all three networks; same numbers as the module-by-module evaluation
    g = torch.Generator().manual_seed(9)
    big = (torch.rand(1, 3, 1024, 1024, generator=g) * 2 - 1).to(DEV)
    big_r = (big + 0.1 * torch.randn(1, 3, 1024, 1024, generator=g).to(DEV)).clamp(-1, 1)
    with torch.no_grad(), conv_precision(True):
        fused = m(big_r, big)
        lp = sum(m.lpips_loss(torch.nn.functional.adaptive_avg_pool2d(big_r, (s, s)), torch.nn.functional.adaptive_avg_pool2d(big, (s, s)))
                 for s in (1024, 512, 256))
        plain = 0.1 * m.id_loss(big_r, big)[0] + torch.nn.functional.mse_loss(big_r, big) + 0.8 * lp + 0.1 * m.face_parsing_loss(big_r, big)[0]
    _close(fused, plain, 1e-4)


@pytest.mark.gpu
def test_full_loss_inversion_trajectory_matches_oracle(monkeypatch):
    """Three Adam steps of the inversion loop with the reference's default loss (0.1 ID + 1.0 l2 + 0.8 LPIPS x3 + 0.1 parsing,
    scripts/optimization.py:88-122, 209-232) on a 32x32 generator, fixed noise: loss trajectory against the same loop through
    the CPU oracle (generator + loss networks), eager and as a replayed CUDA graph."""
    from e4s_b200.networks import Net3
    from e4s_b200.optimization import invert
    monkeypatch.setenv("E4S_B200_CONV", "simt")
    monkeypatch.setenv("E4S_B200_BWD", "simt")
    size, ncls, K = 32, 12, 13
    opts = types.SimpleNamespace(fsencoder_type="psp", remaining_layer_idx=K, num_seg_cls=ncls, out_size=size,
                                 train_G=False, start_from_latent_avg=True, learn_in_w=False)
    net = Net3(opts).eval()
    st = O.synthetic_state({k: tuple(v.shape) for k, v in net.state_dict().items()}, salt=5)
    net.load_state_dict(st)
    for p in net.parameters():
        p.requires_grad = False
    net = net.to(DEV)
    lat = 0.1 * torch.randn(18, 512, generator=torch.Generator().manual_seed(77))
    net.latent_avg = lat.to(DEV)
    g = torch.Generator().manual_seed(8)
    sv0 = 0.5 * torch.randn(1, ncls, 1280, generator=g)
    _, mask, _, noise = O.synthetic_inputs(1, ncls, size, 64, seed=12)
    gst = {k[2:]: v for k, v in st.items() if k.startswith("G.")}
    with torch.no_grad():
        target, _ = O.generator_forward(gst, O.cal_style_codes(st, 0.5 * torch.randn(1, ncls, 1280, generator=g), lat, K), mask, noise, size, K)
    lst = LO.loss_states(SALT)
    latent = sv0.clone().requires_grad_(True)
    opt = torch.optim.Adam([latent], lr=1e-2)
    ref_losses = []
    for _ in range(3):
        opt.zero_grad()
        rec, _ = O.generator_forward(gst, O.cal_style_codes(st, latent, lat, K), mask, noise, size, K)
        loss, _ = LO.calc_loss(lst, target, rec)
        loss.backward()
        opt.step()
        ref_losses.append(float(loss.detach()))
    crit = _criterion()
    for graphed in (False, True):
        _, _, hist = invert(net, target.to(DEV), mask.to(DEV), style_vectors=sv0.to(DEV), steps=3 if not graphed else 4, lr=1e-2,
                            noise=[n.to(DEV) for n in noise], criterion=crit, cuda_graph=graphed)
        ours = [float(h) for h in hist][:3]
        for a, b in zip(ours, ref_losses):
            assert abs(a - b) <= 1e-3 * abs(b), (graphed, ours, ref_losses)
        assert ours[-1] < ours[0]
