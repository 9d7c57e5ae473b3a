"""GPU parity: the sm_100a kernels (through the C ABI) against the committed reference vectors and the CPU oracle.

Bar: max|ours - ref| / max|ref| <= 1e-3 for floating point (north_star), bit-exact for mask / index ops.
"""
import math
import types

import numpy as np
import pytest
import torch

from oracle import e4s_oracle as O
from conftest import REL_TOL, assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(t):
    return t.to(DEV)


# ------------------------------------------------------------------------------------ upfirdn2d
def test_upfirdn2d_golden(golden):
    from e4s_b200.stylegan2.op import upfirdn2d
    for tag in ("blur_up", "skip_up", "blur_dn", "down2", "ragged", "crop"):
        up, down, p0, p1, gain = golden[f"upfirdn2d/{tag}/cfg"]
        fir = O.make_fir((1, 3, 3, 1), float(round(gain)))
        x = torch.from_numpy(golden[f"upfirdn2d/{tag}/x"])
        y = upfirdn2d(cu(x), cu(fir), up=int(up), down=int(down), pad=(int(p0), int(p1)))
        assert_close(y, golden[f"upfirdn2d/{tag}/y"], 1e-5, tag)
    x = torch.from_numpy(golden["upfirdn2d/asym/x"])
    y = upfirdn2d(cu(x), cu(torch.from_numpy(golden["upfirdn2d/asym/fir"])), up=2, down=1, pad=(2, 1))
    assert_close(y, golden["upfirdn2d/asym/y"], 1e-5, "asym (kernel flip)")


@pytest.mark.parametrize("shape,up,down,pad", [
    ((2, 3, 33, 33), 1, 1, (1, 1)),      # hot path, odd input (2H+1 -> 2H), narrow tile variant
    ((1, 2, 257, 257), 1, 1, (1, 1)),    # hot path, wide tile variant, partial tiles
    ((1, 2, 130, 70), 1, 1, (2, 2)),     # its gradient configuration, non-square
    ((2, 3, 40, 24), 2, 1, (2, 1)),
    ((1, 1, 31, 17), 1, 2, (1, 1)),
    ((1, 2, 5, 5), 1, 1, (1, 1)),        # tiny
])
def test_upfirdn2d_vs_oracle(shape, up, down, pad):
    from e4s_b200.stylegan2.op import upfirdn2d
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(*shape, generator=g)
    fir = torch.rand(4, 4, generator=g) - 0.3            # arbitrary, non-separable, asymmetric
    y = upfirdn2d(cu(x), cu(fir), up=up, down=down, pad=pad)
    assert_close(y, O.upfirdn2d(x, fir, up, down, pad), 1e-5)


def test_upfirdn2d_gradients():
    from e4s_b200.stylegan2.op import upfirdn2d
    g = torch.Generator().manual_seed(5)
    for up, down, pad in [(1, 1, (1, 1)), (2, 1, (2, 1)), (1, 2, (1, 1))]:
        x = torch.randn(2, 3, 12, 10, generator=g)
        fir = torch.rand(4, 4, generator=g)
        xr = x.clone().requires_grad_(True)
        yr = O.upfirdn2d(xr, fir, up, down, pad)
        go = torch.randn(yr.shape, generator=g)
        yr.backward(go)
        xg = cu(x).requires_grad_(True)
        gog = cu(go).requires_grad_(True)
        y = upfirdn2d(xg, cu(fir), up=up, down=down, pad=pad)
        (gx,) = torch.autograd.grad(y, xg, gog, create_graph=True)
        assert_close(gx, xr.grad, 1e-5, f"grad up{up} down{down}")
        # second order (upfirdn2d.py:61-82): d<gx, v>/d(grad_output) is the forward op applied to v
        v = torch.randn(x.shape, generator=g)
        (gg,) = torch.autograd.grad((gx * cu(v)).sum(), gog)
        assert_close(gg, O.upfirdn2d(v, fir, up, down, pad), 1e-5, f"double-backward up{up} down{down}")


def test_upfirdn2d_full_size_properties():
    """At BASELINE config-1 size the oracle is too slow; check size-independent properties instead:
    linearity, DC gain (sum of taps) away from the border, and agreement of the tiled hot kernel with the
    gather kernel (forced by an equivalent 5x5 zero-padded FIR)."""
    from e4s_b200.stylegan2.op import upfirdn2d
    fir = cu(O.make_fir((1, 3, 3, 1), 4.0))
    x = torch.randn(4, 32, 1025, 1025, device=DEV)
    z = torch.randn(4, 32, 1025, 1025, device=DEV)
    y = upfirdn2d(x, fir, pad=(1, 1))
    assert y.shape == (4, 32, 1024, 1024)
    lin = upfirdn2d(2.0 * x - 3.0 * z, fir, pad=(1, 1))
    assert_close(lin, 2.0 * y - 3.0 * upfirdn2d(z, fir, pad=(1, 1)), 1e-5, "linearity")
    ones = upfirdn2d(torch.ones(1, 1, 1025, 1025, device=DEV), fir, pad=(1, 1))
    assert torch.allclose(ones[:, :, 2:-2, 2:-2], torch.full_like(ones[:, :, 2:-2, 2:-2], 4.0), atol=1e-5)
    fir5 = torch.zeros(5, 5, device=DEV)
    fir5[1:, 1:] = fir                                    # same filter, but kh=kw=5 -> gather kernel
    sub = x[:1, :4]
    assert_close(upfirdn2d(sub, fir, pad=(1, 1)), upfirdn2d(sub, fir5, pad=(1, 2)), 1e-5, "tiled vs gather")


# ------------------------------------------------------------------------------ fused_leaky_relu
def test_fused_leaky_relu_golden(golden):
    from e4s_b200.stylegan2.op import fused_leaky_relu
    x = cu(torch.from_numpy(golden["flrelu/x"])).requires_grad_(True)
    b = cu(torch.from_numpy(golden["flrelu/b"])).requires_grad_(True)
    y = fused_leaky_relu(x, b)
    assert_close(y, golden["flrelu/y"], 1e-6)
    y.backward(cu(torch.from_numpy(golden["flrelu/go"])))
    assert_close(x.grad, golden["flrelu/gx"], 1e-6)
    assert_close(b.grad, golden["flrelu/gb"], 1e-5)


def test_fused_leaky_relu_layouts_and_shapes():
    from e4s_b200.stylegan2.op import fused_leaky_relu, FusedLeakyReLU
    g = torch.Generator().manual_seed(2)
    for shape in [(3, 8), (2, 8, 5, 7), (1, 12, 16, 16), (2, 5, 3, 3)]:
        x = torch.randn(*shape, generator=g)
        b = torch.randn(shape[1], generator=g)
        ref = O.fused_leaky_relu(x, b)
        assert_close(fused_leaky_relu(cu(x), cu(b)), ref, 1e-6, f"planar {shape}")
        if len(shape) == 4:
            xcl = cu(x).contiguous(memory_format=torch.channels_last)
            assert_close(fused_leaky_relu(xcl, cu(b)), ref, 1e-6, f"channels_last {shape}")
    m = FusedLeakyReLU(8).to(DEV)
    assert list(dict(m.named_parameters())) == ["bias"]
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        fused_leaky_relu(torch.zeros(2, 3), torch.zeros(3))


# ------------------------------------------------------------------------------------- mask ops
def test_mask_ops_bit_exact(golden):
    from e4s_b200 import kernels as K
    from e4s_b200.masks import labelMap2OneHot, celeba19_to_12
    from e4s_b200.stylegan2.modconv import LabelPyramid
    g = torch.Generator().manual_seed(3)
    lab = torch.randint(0, 12, (2, 1, 37, 53), generator=g)
    oh = labelMap2OneHot(cu(lab), 12)
    assert torch.equal(oh.cpu(), O.label_to_onehot(lab, 12))
    label, flag = K.onehot_to_label(oh)
    assert int(flag.item()) == 0 and torch.equal(label.cpu().long(), lab[:, 0])
    bad = oh.clone()
    bad[0, :, 0, 0] = 0.5
    assert int(K.onehot_to_label(bad)[1].item()) == 1
    with pytest.raises(RuntimeError, match="not one-hot"):
        LabelPyramid.from_mask(bad)
    # nearest resize, down and up, power-of-two and ragged ratios
    oh512 = labelMap2OneHot(cu(torch.randint(0, 12, (1, 1, 96, 96), generator=g)), 12)
    pyr = LabelPyramid.from_mask(oh512)
    for s in (4, 8, 16, 32, 48, 96, 192, 100, 7):
        ref = torch.nn.functional.interpolate(oh512.cpu(), size=(s, s), mode="nearest").argmax(1)
        assert torch.equal(pyr.at(s, s).cpu().long(), ref), s
    for who in ("source", "target"):
        raw = cu(torch.from_numpy(golden[f"mask/{who}_raw19"]))
        assert np.array_equal(celeba19_to_12(raw).cpu().numpy(), golden[f"mask/{who}_cls12"])


def test_region_mean(golden):
    from e4s_b200.encoders.psp_encoders import FSEncoder_PSP
    feats, m5 = O.region_mean_case()                       # classes 3 and 4 are empty regions
    enc = FSEncoder_PSP.__new__(FSEncoder_PSP)
    out = FSEncoder_PSP.get_per_comp_styleCode(enc, cu(feats), cu(m5))
    assert_close(out, golden["region_mean/y"], 1e-5)
    assert float(out[:, 3:].abs().max()) == 0.0


# ------------------------------------------------------------- modulated conv building blocks
def _load(module, salt):
    st = O.synthetic_state({k: tuple(v.shape) for k, v in module.state_dict().items()}, salt)
    module.load_state_dict(st)
    return st


def test_modulated_conv_golden(golden):
    from e4s_b200.stylegan2.model import ModulatedConv2d
    for tag, (cin, cout, k, demod, up, hw) in O.MODCONV_CASES.items():
        m = ModulatedConv2d(cin, cout, k, 512, demodulate=demod, upsample=up)
        _load(m, len(tag))
        x, w = O.modconv_case(tag)
        with torch.no_grad():
            y = m.to(DEV)(cu(x), cu(w))
        assert_close(y, golden[f"modconv/{tag}/y"], 1e-5, tag)


def test_styled_conv_and_torgb_golden(golden):
    from e4s_b200.stylegan2.model import StyledConv, ToRGB
    for tag, (cin, cout, up, hw) in O.STYLEDCONV_CASES.items():
        m = StyledConv(cin, cout, 3, 512, upsample=up, mask_op=True)
        _load(m, 7 + len(tag))
        x, nz, codes, mask = O.styledconv_case(tag)
        with torch.no_grad():
            y = m.to(DEV)(cu(x), cu(codes[:, :, 0]), cu(mask), noise=cu(nz))
        assert_close(y, golden[f"styledconv/{tag}/y"], 1e-5, tag)
    m = ToRGB(24, 512, upsample=True, mask_op=True)
    _load(m, 11)
    x, skip, codes, mask = O.torgb_case()
    with torch.no_grad():
        y = m.to(DEV)(cu(x), cu(codes[:, :, 1]), cu(mask), cu(skip))
    assert_close(y, golden["torgb/y"], 1e-5, "torgb")


@pytest.mark.parametrize("kind", ["blobs", "iid"])
def test_styled_conv_and_torgb_vs_oracle(kind):
    """More shapes than the goldens hold: channel counts that do not fill a tile, mixed-class tiles (iid)."""
    from e4s_b200.stylegan2.model import StyledConv, ToRGB
    g = torch.Generator().manual_seed(11)
    ncls = 5
    codes, mask, _, _ = O.synthetic_inputs(2, ncls, 16, 32, seed=3, kind=kind)
    for tag, cin, cout, up, hw in [("plain", 16, 24, False, 8), ("up", 24, 16, True, 8), ("wide", 72, 40, False, 20),
                                   ("tiny", 8, 8, True, 4)]:
        m = StyledConv(cin, cout, 3, 512, upsample=up, mask_op=True)
        st = _load(m, 7 + len(tag))
        x = torch.randn(2, cin, hw, hw, generator=g)
        hout = 2 * hw if up else hw
        nz = torch.randn(2, 1, hout, hout, generator=g)
        with torch.no_grad():
            y = m.to(DEV)(cu(x), cu(codes[:, :, 0]), cu(mask), noise=cu(nz))
        assert_close(y, O.styled_conv(x, codes[:, :, 0], mask, nz, st, "", up, True), 1e-5, f"{kind}/{tag}")
    for cin in (24, 48, 128, 136, 256, 512):      # thread-per-pixel kernel up to 256 channels, warp-per-pixel beyond
        m = ToRGB(cin, 512, upsample=True, mask_op=True)
        st = _load(m, 11)
        x = torch.randn(2, cin, 16, 16, generator=g)
        skip = torch.randn(2, 3, 8, 8, generator=g)
        with torch.no_grad():
            y = m.to(DEV)(cu(x), cu(codes[:, :, 1]), cu(mask), cu(skip))
        assert_close(y, O.to_rgb(x, codes[:, :, 1], mask, skip, st, "", True), 1e-5, f"{kind}/torgb{cin}")


# -------------------------------------------------------------------------------- Generator
def _generator(size, K):
    from e4s_b200.stylegan2.model import Generator
    G = Generator(size, 512, 8, split_layer_idx=5, remaining_layer_idx=K).eval()
    st = O.synthetic_state({k: tuple(v.shape) for k, v in G.state_dict().items()}, salt=size)
    G.load_state_dict(st)
    return G.to(DEV), st


@pytest.mark.parametrize("tag,size,K,B,nc,msz,kind", [
    ("g64_k5", 64, 5, 2, 5, 32, "blobs"),
    ("g32_k13_iid", 32, 13, 1, 12, 64, "iid"),
    ("g256_k13", 256, 13, 1, 12, 512, "blobs"),          # BASELINE.json configs[0]
])
def test_generator_golden(golden, tag, size, K, B, nc, msz, kind):
    """Same seeded parameters/latents/masks/noise as oracle/make_golden.py fed to the reference."""
    G, _ = _generator(size, K)
    codes, mask, _, noise = O.synthetic_inputs(B, nc, size, msz, seed=size + K, kind=kind)
    with torch.no_grad():
        img, lat, feats = G([cu(codes)], None, cu(mask), input_is_latent=True, noise=[cu(n) for n in noise])
    assert lat is None
    e = assert_close(img, golden[f"generator/{tag}/image"], REL_TOL, tag)
    assert_close(feats[:, ::16, ::2, ::2], golden[f"generator/{tag}/feats_sub"], REL_TOL, tag + " feats")
    print(f"{tag}: image max-rel err {e:.2e}")


@pytest.mark.parametrize("path", ["auto", "simt"])
@pytest.mark.parametrize("size,B,nc,kind", [(64, 2, 19, "blobs"), (64, 1, 19, "iid"), (32, 1, 32, "iid"), (32, 3, 1, "blobs")])
def test_generator_region_count_sweep_vs_oracle(monkeypatch, path, size, B, nc, kind):
    """SURVEY.md section 8: 12 regions is the default, 19 (the raw parser label count) the sweep point; 32 is the most
    the kernels' region bit masks hold and 1 the degenerate case.  Tensor-core and exact-fp32 paths against the CPU oracle."""
    monkeypatch.setenv("E4S_B200_CONV", path)
    G, st = _generator(size, 13)
    codes, mask, _, noise = O.synthetic_inputs(B, nc, size, 2 * size, seed=size + nc, kind=kind)
    with torch.no_grad():
        img, _, feats = G([cu(codes)], None, cu(mask), input_is_latent=True, noise=[cu(n) for n in noise])
        ref_img, ref_feats = O.generator_forward(st, codes, mask, noise, size, 13)
    assert_close(img, ref_img, REL_TOL, f"{nc} regions, image")
    assert_close(feats, ref_feats, REL_TOL, f"{nc} regions, feats")


def test_generator_api_surface():
    G, _ = _generator(32, 13)
    assert G.n_latent == 8 and G.num_layers == 7 and len(G.convs) == 6 and len(G.to_rgbs) == 3
    assert [n.shape[-1] for n in G.make_noise()] == [4, 8, 8, 16, 16, 32, 32]
    codes, mask, _, noise = O.synthetic_inputs(2, 12, 32, 32, seed=1)
    with torch.no_grad():
        img, lat, feats = G([cu(codes)], None, cu(mask), input_is_latent=True, return_latents=True)   # fresh noise
        img2, _, _ = G([cu(codes)], None, cu(mask), input_is_latent=True, randomize_noise=False)
    assert img.shape == (2, 3, 32, 32) and feats.shape == (2, 512, 16, 16) and lat.shape == codes.shape
    assert torch.isfinite(img).all() and torch.isfinite(img2).all()


def _net3():
    from e4s_b200.networks import Net3
    opts = types.SimpleNamespace(fsencoder_type="psp", remaining_layer_idx=13, num_seg_cls=12, out_size=64,
                                 train_G=False, start_from_latent_avg=True, learn_in_w=False)
    net = Net3(opts).eval()
    st = O.synthetic_state({k: tuple(v.shape) for k, v in net.state_dict().items()}, salt=5)
    net.load_state_dict(st)
    return net.to(DEV), st


def test_net3_gen_img_and_style_codes(golden):
    net, st = _net3()
    sv, lat, _, _ = O.net3_case()
    net.latent_avg = cu(lat)
    with torch.no_grad():
        codes = net.cal_style_codes(cu(sv))
    assert_close(codes[:, :, :, ::8], golden["net3/style_codes_sub"], 1e-4, "cal_style_codes")
    _, mask, _, noise = O.synthetic_inputs(2, 12, 64, 128, seed=9)
    gst = {k[2:]: v for k, v in st.items() if k.startswith("G.")}
    with torch.no_grad():
        img, minus1, feats = net.gen_img(None, codes, cu(mask), noise=[cu(n) for n in noise])
    assert minus1 == -1
    ref_img, _ = O.generator_forward(gst, O.cal_style_codes(st, sv, lat, 13), mask, noise, 64, 13)
    assert_close(img, ref_img, REL_TOL, "gen_img")


def test_get_style_vectors_golden(golden):
    net, _ = _net3()
    _, _, img, mask = O.net3_case()
    with torch.no_grad():
        vec, struct = net.get_style_vectors(cu(img), cu(mask))
    assert vec.shape == (1, 12, 1280) and float(struct.abs().max()) == 0.0
    assert_close(vec, golden["net3/style_vectors"], REL_TOL, "get_style_vectors")


def test_streaming_pipeline_matches_direct_calls():
    """e4s_b200.pipeline.SynthesisPipeline (H2D / generator / D2H on three streams, two slots) returns, per ticket, what a
    plain gen_img call on the same inputs returns (noise strengths zeroed: the generator draws fresh noise per call)."""
    from e4s_b200.pipeline import SynthesisPipeline
    from e4s_b200 import masks as M
    net, _ = _net3()
    with torch.no_grad():
        for name, prm in net.named_parameters():
            if name.endswith("noise.weight"):
                prm.zero_()
    sv, lat, _, _ = O.net3_case()
    net.latent_avg = cu(lat)
    pipe = SynthesisPipeline(net, ncls=12, depth=2)
    g = torch.Generator().manual_seed(77)
    batches, tickets = [], []
    for i in range(5):
        with torch.no_grad():
            codes = net.cal_style_codes(cu(sv) + 0.1 * i).cpu().pin_memory()
        labels = torch.randint(0, 12, (2, 1, 8, 8), generator=g, dtype=torch.uint8).repeat_interleave(16, 2).repeat_interleave(16, 3)
        labels = labels.contiguous().pin_memory()
        batches.append((codes, labels))
        tickets.append(pipe.submit(codes, labels))
        if i >= 1:                                      # consume with a lag of one batch, like a service would
            got = pipe.result(tickets[i - 1]).clone()
            c, l = batches[i - 1]
            with torch.no_grad():
                ref, _, _ = net.gen_img(None, cu(c), M.labelMap2OneHot(cu(l), 12))
            # not bit-identical: the three MMA-issuing warps of the conv kernel accumulate in no fixed order
            assert_close(got, ref.cpu(), 2e-5, f"pipeline batch {i - 1}")
    pipe.drain()
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError):
        pipe.result(tickets[0])                         # only `depth` results are held


# ---------------------------------------------------------------- small GEMMs (style modulation, LocalMLP)
@pytest.mark.parametrize("g,m,n,k,shared_x,shared_w", [
    (1, 192, 512, 512, True, True),        # one style modulation: [B * regions, 512] x [512, Cin]
    (1, 1, 32, 512, True, True),           # one face, unmasked layer
    (12, 16, 512, 1280, False, False),     # LocalMLP layer 1, grouped over the regions
    (12, 3, 6656, 512, False, False),      # LocalMLP layer 2, odd batch
    (5, 37, 68, 36, False, True),          # partial tiles in every dimension, shared weight
])
def test_linear_kernel(g, m, n, k, shared_x, shared_w):
    from e4s_b200 import kernels as K
    gen = torch.Generator().manual_seed(g + m + n + k)
    x = torch.randn((m, k) if (shared_x and shared_w) else (g, m, k), generator=gen)
    w = torch.randn((n, k) if shared_w else (g, n, k), generator=gen) / k ** 0.5
    bias = torch.randn((n,) if shared_w else (g, n), generator=gen)
    ref = torch.matmul(x.double(), w.double().transpose(-1, -2)) + (bias.double() if shared_w else bias.double()[:, None, :])
    out = K.linear(cu(x), cu(w), cu(bias), 0.01)
    assert_close(out, torch.nn.functional.leaky_relu(ref, 0.01).float(), 1e-5, "linear TN + bias + leaky")
    gy = torch.randn(ref.shape, generator=gen)
    gx = K.linear(cu(gy), cu(w), None, 1.0, w_is_kn=True)
    assert_close(gx, torch.matmul(gy.double(), w.double()).float(), 1e-5, "linear NN (input gradient)")


def test_local_mlps_match_oracle_and_autograd():
    """Net3.cal_style_codes (12 LocalMLPs, networks.py:135-158) on the own GEMM kernel: values and the gradient wrt the texture
    vectors (what the inversion loop optimises) against the oracle's autograd."""
    net, st = _net3()
    for prm in net.parameters():
        prm.requires_grad = False
    net.latent_avg = cu(0.5 * torch.randn(18, 512, generator=torch.Generator().manual_seed(77)))
    sv = torch.randn(3, 12, 1280, generator=torch.Generator().manual_seed(1))
    go = torch.randn(3, 12, 18, 512, generator=torch.Generator().manual_seed(2))
    a = cu(sv).requires_grad_(True)
    ours = net.cal_style_codes(a)
    ours.backward(cu(go))
    b = sv.clone().requires_grad_(True)
    ref = O.cal_style_codes(st, b, net.latent_avg.cpu(), 13)
    ref.backward(go)
    assert_close(ours, ref, 1e-5, "cal_style_codes")
    assert_close(a.grad, b.grad, 1e-5, "d cal_style_codes / d texture vectors")


# ---------------------------------------------------------------- tensor-core (tcgen05) kernel
def _tc_case(b, cin, cout, hw, up, ncls, kind, seed, act=True):
    from e4s_b200 import kernels as K
    from e4s_b200.stylegan2.modconv import PreparedConv
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(1, cout, cin, 3, 3, generator=g)
    blur = O.make_fir((1, 3, 3, 1), 4.0)
    prep = PreparedConv().get(cu(w), up, cu(blur) if up else None)
    x = cu(torch.randn(b, hw, hw, cin, generator=g))
    s = cu(1.0 + 0.3 * torch.randn(b, ncls, cin, generator=g))
    ho = 2 * hw if up else hw
    if kind == "iid":
        label = torch.randint(0, ncls, (b, ho, ho), generator=g, dtype=torch.uint8)
    else:
        coarse = torch.randint(0, ncls, (b, 1, max(2, ho // 16), max(2, ho // 16)), generator=g).float()
        label = torch.nn.functional.interpolate(coarse, size=(ho, ho), mode="nearest")[:, 0].to(torch.uint8)
    label = cu(label) if ncls > 1 else None
    noise = cu(torch.randn(b, 1, ho, ho, generator=g))
    nw = cu(torch.tensor([0.37]))
    bias = cu(0.1 * torch.randn(cout, generator=g))
    dm = K.demod(s, prep.wsq)
    args = (s, dm, label, noise, nw, bias, up, act)
    return K, prep, x, args


TC_CASES = [
    (1, 64, 64, 16, False, 1, "blobs"),       # smallest: one K chunk, single class
    (2, 128, 128, 32, False, 1, "blobs"),     # two chunks, N = 128
    (1, 64, 32, 24, False, 1, "blobs"),       # N = 32, partial tiles in both directions
    (2, 192, 256, 20, False, 5, "blobs"),     # N = 256 (persistent) / two N tiles (v1), masked
    (1, 128, 64, 16, False, 6, "iid"),        # every tile holds every class -> 6 passes per tile
    (2, 64, 128, 16, True, 4, "blobs"),       # up-sampling layer: 4 parity kernels
    (1, 512, 512, 16, True, 3, "iid"),        # full-width layer, up, mixed classes
]
TCP_EXTRA = [
    (2, 32, 32, 40, False, 1, "blobs"),       # 32-channel chunks (64-byte swizzle), resident weights, many tiles per CTA
    (1, 32, 64, 18, False, 4, "iid"),         # 32-channel chunks, masked
    (1, 64, 32, 36, True, 1, "blobs"),        # up, N = 4 x 32
    (1, 96, 32, 16, True, 3, "iid"),          # 32-channel chunks x3, up, masked
    (3, 512, 512, 64, False, 12, "blobs"),    # production shape c7@64: > 148 work items, two N tiles, 12 regions
    (1, 128, 64, 32, True, 2, "iid"),         # every tile holds exactly two regions (two-region mode of up-sampling layers)
    (2, 64, 64, 24, True, 2, "iid"),
    (1, 256, 256, 32, True, 3, "blobs"),
    (16, 512, 512, 4, False, 12, "iid"),      # the 4x4 / 8x8 layers of a 16-face batch (mostly-halo tiles)
    (16, 512, 512, 4, True, 3, "iid"),
    (4, 512, 512, 8, True, 12, "blobs"),
    (1, 64, 128, 40, False, 1, "blobs"),      # encoder shape: small K with N = 128
    (2, 32, 128, 24, False, 3, "iid"),        # small K, N = 128, masked
]
# production shapes of the 1024x1024 generator's top layers and of the encoder's first unit, B = 1: several work items
# per persistent CTA (ring wrap-around of every pipeline), checked against the fp32 SIMT kernel
PRODUCTION_CASES = [
    (1, 64, 64, 512, False, 1, "blobs"),      # c13 @512
    (1, 64, 32, 512, True, 1, "blobs"),       # c14 ^1024
    (1, 32, 32, 1024, False, 1, "blobs"),     # c15 @1024
    (1, 128, 64, 256, True, 1, "blobs"),      # c12 ^512
    (1, 64, 128, 256, False, 1, "blobs"),     # encoder unit 0 conv1
    (1, 128, 128, 256, False, 12, "blobs"),   # c11 @256, masked
    (1, 256, 128, 128, True, 12, "blobs"),    # c10 ^256, masked
    (1, 64, 64, 256, False, 12, "blobs"),     # small-K activation ring, mixed tiles
    (1, 64, 32, 256, True, 12, "blobs"),
    (2, 32, 32, 512, False, 5, "blobs"),
]


@pytest.mark.parametrize("b,cin,cout,hw,up,ncls,kind", TC_CASES + TCP_EXTRA + [
    (2, 64, 128, 30, True, 5, "blobs"),       # up-sampling with region borders: row-class pass + fix-up passes
    (1, 160, 256, 28, False, 12, "iid"),      # every row its own region: pure row-class mode, 5 K chunks
    (2, 256, 64, 16, True, 12, "iid"),        # up + iid: many fix-up passes
])
def test_tcr_kernel_matches_simt(b, cin, cout, hw, up, ncls, kind):
    """The fourth-generation tcgen05 kernel (one pass per tile on any mask) vs the fp32 SIMT kernel."""
    K, prep, x, args = _tc_case(b, cin, cout, hw, up, ncls, kind, seed=cin + cout + hw)
    ref = K.modconv3x3_fwd(x, prep.wt, *args)
    out = K.modconv3x3_tcr_fwd(x, prep.w_hilo, *args)
    torch.cuda.synchronize()
    e = assert_close(out, ref, 1e-4, f"tcr vs simt {b},{cin},{cout},{hw},{up},{ncls},{kind}")
    print(f"tcr-vs-simt rel err {e:.2e}")


@pytest.mark.parametrize("ntile", ["32", "64", "128", "256"])
@pytest.mark.parametrize("b,cin,cout,hw,up,ncls,kind", [
    (1, 512, 512, 8, False, 12, "iid"),       # low-resolution layers of ONE face: the occupancy rule narrows the N tile
    (1, 512, 512, 8, True, 3, "iid"),
    (2, 256, 256, 16, False, 4, "blobs"),
    (1, 128, 256, 32, True, 2, "iid"),
])
def test_tcr_kernel_every_n_tile_width(monkeypatch, ntile, b, cin, cout, hw, up, ncls, kind):
    """csrc/modconv_tcr.cu:pick_ntile chooses the N-tile width by occupancy; every width it can choose (forced here with
    E4S_B200_NTILE; widths a layer does not allow fall back to the automatic choice) gives the same result."""
    monkeypatch.setenv("E4S_B200_NTILE", ntile)
    K, prep, x, args = _tc_case(b, cin, cout, hw, up, ncls, kind, seed=cin + cout + hw)
    ref = K.modconv3x3_fwd(x, prep.wt, *args)
    out = K.modconv3x3_tcr_fwd(x, prep.w_hilo, *args)
    torch.cuda.synchronize()
    assert_close(out, ref, 1e-4, f"tcr vs simt, N tile {ntile}: {b},{cin},{cout},{hw},{up},{ncls},{kind}")


@pytest.mark.parametrize("up2", ["0", "1"])
@pytest.mark.parametrize("b,cin,cout,hw,up,ncls,kind", [
    (1, 512, 512, 16, True, 3, "iid"),        # N tile 256 (the auto choice for the 512-channel up-sampling layers)
    (4, 512, 512, 8, True, 12, "blobs"),
    (2, 512, 256, 24, True, 12, "blobs"),     # c8's channels; partial tiles; pure, two-region and mixed tiles
    (1, 256, 128, 40, True, 5, "blobs"),      # N tile 128
    (2, 128, 64, 20, True, 2, "iid"),         # N tile 64
    (1, 192, 32, 16, True, 12, "iid"),        # N tile 32, three K chunks
    (1, 128, 256, 16, True, 1, "blobs"),      # unmasked
])
def test_tcr_kernel_parity_work_items(monkeypatch, up2, b, cin, cout, hw, up, ncls, kind):
    """Up-sampling layers as parity work items (csrc/modconv_tcr.cu, UP2: one (tile, N tile, output parity) per item, N
    tiles up to 256 wide) and as four parities along N give the same result as the fp32 SIMT kernel."""
    monkeypatch.setenv("E4S_B200_UP2", up2)
    K, prep, x, args = _tc_case(b, cin, cout, hw, up, ncls, kind, seed=cin + cout + hw)
    ref = K.modconv3x3_fwd(x, prep.wt, *args)
    out = K.modconv3x3_tcr_fwd(x, prep.w_hilo, *args)
    torch.cuda.synchronize()
    e = assert_close(out, ref, 1e-4, f"tcr (UP2={up2}) vs simt {b},{cin},{cout},{hw},{up},{ncls},{kind}")
    print(f"tcr-vs-simt UP2={up2} rel err {e:.2e}")


@pytest.mark.parametrize("b,cin,cout,hw,ncls,kind", [
    (1, 64, 32, 16, 1, "blobs"),              # one K chunk of 64, one region, one N tile
    (2, 128, 64, 20, 1, "blobs"),             # two chunks, two N tiles, partial tiles in both directions
    (1, 96, 32, 18, 1, "blobs"),              # 32-channel chunks (64-byte swizzle) x 3
    (2, 64, 128, 16, 4, "blobs"),             # region borders: one- and two-region passes
    (1, 128, 64, 32, 2, "iid"),               # every tile holds exactly two regions: one pass, both accumulator buffers
    (1, 128, 32, 30, 3, "iid"),               # three regions: a two-region pass, then a one-region pass
    (1, 256, 64, 16, 12, "iid"),              # every tile holds all twelve regions: six passes
    (4, 512, 512, 8, 12, "blobs"),            # the low-resolution 512-channel layers (16 N tiles)
    (1, 256, 128, 128, 12, "blobs"),          # c10 ^256 of the 1024x1024 generator, masked, B = 1
    (1, 128, 64, 256, 1, "blobs"),            # c12 ^512: several work items per persistent CTA
    (1, 64, 32, 512, 1, "blobs"),             # c14 ^1024
])
def test_tch_kernel_matches_simt(b, cin, cout, hw, ncls, kind):
    """The H-form up-sampling kernel (csrc/modconv_tch.cu: vertical blur half folded into the weights, horizontal half and
    region selection in the epilogue; half the MACs of the polyphase form) against the fp32 SIMT kernel."""
    K, prep, x, args = _tc_case(b, cin, cout, hw, True, ncls, kind, seed=cin + cout + hw)
    assert prep.v_hilo is not None and tuple(prep.v_hilo.shape) == (2, 6, 3, cout, cin)
    s, dm, label, noise, nw, bias, up, act = args
    ref = K.modconv3x3_fwd(x, prep.wt, *args)
    out = K.modconv3x3_up_tch_fwd(x, prep.v_hilo, prep.fx, s, dm, label, noise, nw, bias, act)
    torch.cuda.synchronize()
    e = assert_close(out, ref, 1e-4, f"tch vs simt {b},{cin},{cout},{hw},{ncls},{kind}")
    print(f"tch-vs-simt rel err {e:.2e}")


def test_tch_kernel_asymmetric_fir_and_no_epilogue_inputs():
    """H-form with an asymmetric separable FIR (true convolution: the flipped taps matter), no noise, no bias, no activation,
    no demodulation - against conv_transpose2d + upfirdn2d of the oracle."""
    from e4s_b200 import kernels as K
    from e4s_b200.stylegan2.modconv import PreparedConv
    g = torch.Generator().manual_seed(11)
    cin, cout, hw = 64, 32, 12
    w = torch.randn(1, cout, cin, 3, 3, generator=g)
    fa, fb = torch.tensor([1., 2., 4., 3.]), torch.tensor([2., 1., 5., 1.])
    fir = torch.outer(fa, fb)
    fir = fir / fir.sum() * 4
    prep = PreparedConv().get(cu(w), True, cu(fir))
    assert prep.v_hilo is not None
    x = torch.randn(1, hw, hw, cin, generator=g)
    s = 1.0 + 0.3 * torch.randn(1, 1, cin, generator=g)
    out = K.modconv3x3_up_tch_fwd(cu(x), prep.v_hilo, prep.fx, cu(s), None, None, None, None, None, False)
    xs = (x * s[:, 0][:, None, None, :]).permute(0, 3, 1, 2).double()
    wt = (w[0] / (cin * 9) ** 0.5).double()
    u = torch.nn.functional.conv_transpose2d(xs, wt.transpose(0, 1), stride=2)
    ref = O.upfirdn2d(u.float(), fir, pad=(1, 1)).permute(0, 2, 3, 1)
    assert_close(out, ref, 1e-4, "tch, asymmetric FIR, bare conv")


@pytest.fixture
def deterministic():
    import e4s_b200
    e4s_b200.set_deterministic(True)
    assert e4s_b200.is_deterministic()
    yield
    e4s_b200.set_deterministic(False)


@pytest.mark.parametrize("b,cin,cout,hw,up,ncls,kind", [
    (2, 64, 64, 40, False, 1, "blobs"),       # small K, resident weights, several items per CTA
    (1, 128, 256, 28, False, 12, "iid"),      # row-class staging on every tile
    (2, 64, 64, 24, True, 2, "iid"),          # four parities along N, two-region tiles (both accumulator buffers)
    (2, 512, 256, 24, True, 12, "blobs"),     # parity work items
    (1, 256, 128, 40, True, 5, "blobs"),      # H-form kernel (auto choice for this shape): one- and two-region passes
])
def test_deterministic_mode_is_bit_reproducible(deterministic, b, cin, cout, hw, up, ncls, kind):
    """e4s_b200.set_deterministic(True): one warp issues the three split-precision products in a fixed order, so two runs give
    identical bits (the default, three concurrently issuing warps, is reproducible to fp32 rounding only); same values as
    the default mode and the fp32 SIMT kernel within the usual tolerance."""
    import e4s_b200
    from e4s_b200.stylegan2.modconv import up_form
    K, prep, x, args = _tc_case(b, cin, cout, hw, up, ncls, kind, seed=cin + cout + hw)
    s, dm, label, noise, nw, bias, up_, act = args

    def run():
        if up and up_form(prep) == "h":
            return K.modconv3x3_up_tch_fwd(x, prep.v_hilo, prep.fx, s, dm, label, noise, nw, bias, act)
        return K.modconv3x3_tcr_fwd(x, prep.w_hilo, *args)

    outs = [run() for _ in range(3)]
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), "deterministic mode is not bit-reproducible"
    assert_close(outs[0], K.modconv3x3_fwd(x, prep.wt, *args), 1e-4, "deterministic mode vs simt")
    e4s_b200.set_deterministic(False)
    assert_close(run(), outs[0], 2e-5, "default mode vs deterministic mode")


def test_deterministic_generator_is_bit_reproducible(deterministic):
    G, _ = _generator(64, 5)
    codes, mask, _, noise = O.synthetic_inputs(2, 5, 64, 32, seed=69)
    with torch.no_grad():
        a, _, _ = G([cu(codes)], None, cu(mask), input_is_latent=True, noise=[cu(n) for n in noise])
        b, _, _ = G([cu(codes)], None, cu(mask), input_is_latent=True, noise=[cu(n) for n in noise])
    assert torch.equal(a, b)


@pytest.mark.parametrize("stk", ["0", "1"])
@pytest.mark.parametrize("b,cin,cout,hw,up,ncls,kind", [
    (2, 32, 32, 40, False, 1, "blobs"),       # c15's channels: resident weights, several items per CTA
    (1, 64, 64, 36, False, 1, "blobs"),       # c13's channels: two K chunks
    (1, 32, 64, 18, False, 4, "iid"),         # masked: row-class path with the stacked product
    (2, 64, 32, 24, False, 3, "blobs"),
])
def test_tcr_kernel_stacked_hilo_weights(monkeypatch, stk, b, cin, cout, hw, up, ncls, kind):
    """Small-N plain layers with w_hi / w_lo stacked along N (csrc/modconv_tcr.cu STK: two MMAs per (tap, K step) instead of
    three, the two accumulator halves added in the epilogue) and without, against the fp32 SIMT kernel."""
    monkeypatch.setenv("E4S_B200_STK", stk)
    K, prep, x, args = _tc_case(b, cin, cout, hw, up, ncls, kind, seed=cin + cout + hw)
    ref = K.modconv3x3_fwd(x, prep.wt, *args)
    out = K.modconv3x3_tcr_fwd(x, prep.w_hilo, *args)
    torch.cuda.synchronize()
    assert_close(out, ref, 1e-4, f"tcr (STK={stk}) vs simt {b},{cin},{cout},{hw},{ncls},{kind}")


@pytest.mark.parametrize("b,cin,cout,hw,up,ncls,kind", PRODUCTION_CASES)
def test_tcr_kernel_production_shapes(b, cin, cout, hw, up, ncls, kind):
    K, prep, x, args = _tc_case(b, cin, cout, hw, up, ncls, kind, seed=cin + cout + hw)
    ref = K.modconv3x3_fwd(x, prep.wt, *args)
    out = K.modconv3x3_tcr_fwd(x, prep.w_hilo, *args)
    torch.cuda.synchronize()
    e = assert_close(out, ref, 1e-4, f"tcr vs simt (production shape) {b},{cin},{cout},{hw},{up},{ncls},{kind}")
    print(f"tcr-vs-simt rel err {e:.2e}")


def test_generator_golden_tensor_core_path(golden, monkeypatch):
    """Whole generator with every eligible layer forced onto the persistent tcgen05 kernel (also at 4x4..8x8, where
    the default policy would pick the SIMT kernel), against the reference vectors."""
    monkeypatch.setenv("E4S_B200_CONV", "tcr")
    for tag, size, K_, B, nc, msz, kind in [("g64_k5", 64, 5, 2, 5, 32, "blobs"), ("g256_k13", 256, 13, 1, 12, 512, "blobs")]:
        G, _ = _generator(size, K_)
        codes, mask, _, noise = O.synthetic_inputs(B, nc, size, msz, seed=size + K_, kind=kind)
        with torch.no_grad():
            img, _, feats = G([cu(codes)], None, cu(mask), input_is_latent=True, noise=[cu(n) for n in noise])
        e = assert_close(img, golden[f"generator/{tag}/image"], REL_TOL, tag + " (tc)")
        print(f"{tag} tensor-core path: image max-rel err {e:.2e}")


# ------------------------------------------------------------------------------ RGI encoder kernels
def test_encoder_building_blocks():
    """conv3x3 (stride 1/2, folded InstanceNorm, PReLU), instnorm statistics and the unit tail against torch CPU."""
    import torch.nn.functional as F
    from e4s_b200 import kernels as K
    g = torch.Generator().manual_seed(41)
    x = torch.randn(2, 64, 24, 20, generator=g) * 2.0 + 0.7
    w = torch.randn(96, 64, 3, 3, generator=g) / 24.0
    slope = 0.25 + 0.05 * torch.randn(96, generator=g)
    xpm = cu(x).permute(0, 2, 3, 1).contiguous()
    planes = K.split_bf16(cu(w).permute(2, 3, 0, 1).reshape(1, 9, 96, 64))
    sc, sh = K.instnorm_affine(xpm)
    mean, var = x.mean((2, 3)), x.var((2, 3), unbiased=False)
    assert_close(sc, torch.rsqrt(var + 1e-5), 1e-5, "instnorm scale")
    assert_close(sh, -mean * torch.rsqrt(var + 1e-5), 1e-4, "instnorm shift")
    for stride in (1, 2):
        y = K.conv3x3_tc(xpm, planes, sc, sh, cu(slope), out_stride=stride)
        ref = F.prelu(F.conv2d(F.instance_norm(x, eps=1e-5), w, stride=stride, padding=1), slope)
        assert_close(y.permute(0, 3, 1, 2), ref, 1e-4, f"IN->conv->PReLU stride {stride}")
    y = torch.randn(2, 12, 10, 96, generator=g)
    short = torch.randn(2, 24, 20, 96, generator=g)
    ys, yt = torch.rand(2, 96, generator=g) + 0.5, torch.randn(2, 96, generator=g)
    out = K.norm_residual(cu(y), cu(ys), cu(yt), 0.5, shortcut=cu(short), sc_stride=2)
    ref = 0.5 * (y * ys[:, None, None] + yt[:, None, None]) + short[:, ::2, ::2]
    assert_close(out, ref, 1e-6, "unit tail")


@pytest.mark.parametrize("b,cin,cout,h,w", [(2, 64, 64, 24, 20), (1, 128, 128, 34, 30), (2, 32, 96, 16, 16)])
def test_encoder_stride2_as_four_taps_on_space_to_depth(b, cin, cout, h, w):
    """helpers.py:138 (conv2 of the first unit of a stage, stride 2): conv1 stores its IN -> conv -> PReLU output space-to-depth
    (out_stride 4), conv2 runs as the taps (dy, dx) in {-1, 0}^2 over 4 C channels at the output resolution (tap mask 0x1B) -
    against torch's stride-2 convolution in fp64; and a 1x1 convolution as the centre tap alone (tap mask 0x10)."""
    import torch.nn.functional as F
    from e4s_b200 import kernels as K
    from e4s_b200.encoders.psp_encoders import _conv_planes, _conv_planes_s2d, TAPS_S2D, TAP_CENTRE
    g = torch.Generator().manual_seed(b + cin + h)
    x = torch.randn(b, cin, h, w, generator=g) * 1.5 + 0.3
    w1 = torch.randn(cin, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    w2 = torch.randn(cout, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    slope = 0.25 + 0.05 * torch.randn(cin, generator=g)
    xpm = cu(x).permute(0, 2, 3, 1).contiguous()
    sc, sh = K.instnorm_affine(xpm)
    mid = K.conv3x3_tc(xpm, _conv_planes(cu(w1)), sc, sh, cu(slope), out_stride=4)
    assert tuple(mid.shape) == (b, h // 2, w // 2, 4 * cin)
    ref_mid = F.prelu(F.conv2d(F.instance_norm(x.double(), eps=1e-5), w1.double(), padding=1), slope.double())
    s2d = ref_mid.permute(0, 2, 3, 1).reshape(b, h // 2, 2, w // 2, 2, cin).permute(0, 1, 3, 2, 4, 5).reshape(b, h // 2, w // 2, 4 * cin)
    assert_close(mid, s2d.float(), 1e-4, "conv1 with the space-to-depth store")
    y = K.conv3x3_tc(mid, _conv_planes_s2d(cu(w2)), tap_mask=TAPS_S2D)
    ref = F.conv2d(ref_mid, w2.double(), stride=2, padding=1)
    assert_close(y.permute(0, 3, 1, 2), ref.float(), 1e-4, "stride-2 conv as four taps")
    old = K.conv3x3_tc(K.conv3x3_tc(xpm, _conv_planes(cu(w1)), sc, sh, cu(slope)), _conv_planes(cu(w2)), out_stride=2)
    assert_close(y, old, 1e-4, "four-tap form vs every-pixel-keep-even form")
    wsc = torch.randn(cout, cin, 1, 1, generator=g) / cin ** 0.5
    xs = xpm[:, ::2, ::2, :].contiguous()
    ysc = K.conv3x3_tc(xs, _conv_planes(cu(wsc)), tap_mask=TAP_CENTRE)
    assert_close(ysc.permute(0, 3, 1, 2), F.conv2d(x.double()[:, :, ::2, ::2], wsc.double()).float(), 1e-4, "1x1 conv as the centre tap")


def test_generator_1024_tensor_core_path_matches_exact_fp32_path(monkeypatch):
    """BASELINE's full size (1024x1024, K=13, 12 regions, one face): every layer on the tensor-core kernel against every
    layer on the exact-fp32 SIMT kernel (which the 32/64/256 goldens pin to the reference).  Size-independent property:
    the two code paths share only the op sequence."""
    g, _ = _generator(1024, 13)
    codes, mask, _, noise = O.synthetic_inputs(1, 12, 1024, 256, seed=21)
    noise = [cu(n) for n in noise]
    outs = {}
    for mode in ("simt", "auto"):
        monkeypatch.setenv("E4S_B200_CONV", mode)
        with torch.no_grad():
            img, _, _ = g([cu(codes)], None, cu(mask), input_is_latent=True, noise=noise)
        outs[mode] = img.float().cpu()
    assert outs["auto"].shape == (1, 3, 1024, 1024)
    # split-bf16 x3 leaves <= 2e-5 per layer (tests above); 17 stacked layers measured 0.9e-4 ... 1.03e-4 run to run (the
    # accumulation order of the three MMA-issuing warps is not fixed), so the check sits at 3e-4 - a third of the path's bar
    e = assert_close(outs["auto"], outs["simt"], 3e-4, "1024x1024 generator, tensor-core vs exact path")
    print(f"1024 generator tc-vs-exact rel err {e:.2e}")


def test_generator_1024_matches_cpu_oracle_alone_and_inside_a_batch():
    """The benched configuration against the ORACLE (not against another kernel of this library): one 1024x1024 face, 12 regions
    of a blob mask, K = 13, default kernels, vs O.generator_forward on the host (~7 s); then the same face as sample 9 of a
    16-face batch with other codes and masks around it - batching must not change a face.  REL_TOL, both norms."""
    g, st = _generator(1024, 13)
    codes, mask, _, noise = O.synthetic_inputs(1, 12, 1024, 512, seed=21)
    with torch.no_grad():
        ref, _ = O.generator_forward(st, codes, mask, noise, 1024, 13)
        img, _, _ = g([cu(codes)], None, cu(mask), input_is_latent=True, noise=[cu(n) for n in noise])
    e = assert_close(img, ref, REL_TOL, "1024x1024 generator (default kernels) vs CPU oracle")
    print(f"1024 generator vs oracle: max-rel {e:.2e}")
    bc, bm, _, _ = O.synthetic_inputs(16, 12, 1024, 512, seed=33)
    bc[9], bm[9] = codes[0], mask[0]
    with torch.no_grad():
        batch, _, _ = g([cu(bc)], None, cu(bm), input_is_latent=True, noise=[cu(n) for n in noise])
    assert_close(batch[9:10], ref, REL_TOL, "face 9 of a 16-face batch vs CPU oracle")
    assert_close(batch[9:10], img, 5e-5, "face 9 of a 16-face batch vs the same face alone")


def test_dcodes_gradient_default_kernels_256():
    """d loss / d codes through the 256x256 generator on the DEFAULT (tensor-core) forward and backward kernels against the
    oracle's autograd.  Stated tolerance: rel-L2 <= 1e-2 and cosine >= 0.9999 over the whole gradient (observed 5.8e-3 /
    0.999983).  The gradient of a 15-layer leaky-ReLU network is not a smooth function of its rounding: the few pixels whose
    pre-activation sits within 1e-5 of zero take the other branch (slope 1 vs 0.2) under the split-bf16 forward, and each flip
    moves the gradient by O(1e-3) of its norm; on the exact-fp32 kernels the same quantity holds 1e-3 in the max norm
    (tests/test_backward_gpu.py)."""
    g, st = _generator(256, 13)
    codes, mask, _, noise = O.synthetic_inputs(1, 12, 256, 256, seed=5)
    w = torch.randn(1, 3, 256, 256, generator=torch.Generator().manual_seed(4))
    c_ref = codes.clone().requires_grad_(True)
    ref, _ = O.generator_forward(st, c_ref, mask, noise, 256, 13)
    (ref * w).sum().backward()
    c = cu(codes).requires_grad_(True)
    img, _, _ = g([c], None, cu(mask), input_is_latent=True, noise=[cu(n) for n in noise])
    (img * cu(w)).sum().backward()
    a, b = c.grad.double().cpu().flatten(), c_ref.grad.double().flatten()
    rel_l2 = float((a - b).norm() / b.norm())
    cos = float(torch.dot(a, b) / (a.norm() * b.norm()))
    print(f"dcodes @256, default kernels: rel-L2 {rel_l2:.2e}, cosine {cos:.7f}")
    assert rel_l2 < 1e-2 and cos > 0.9999, (rel_l2, cos)


def test_linear_multi_strided_rows_and_demod_form():
    """e4s_linear_multi_f32: problems of different shapes in one launch, x rows read in place from a strided latent slice, plain
    and demodulation forms, against fp64."""
    from e4s_b200 import kernels as K
    g = torch.Generator().manual_seed(5)
    latent = cu(torch.randn(3, 4, 6, 64, generator=g))                           # [B, ncls, n_latent, dim]
    shapes = [(1, True, 96), (4, True, 32), (2, False, 64), (5, False, 36)]      # (latent index, per-region rows?, N)
    probs, refs = [], []
    for idx, per_region, n in shapes:
        w = cu(torch.randn(n, 64, generator=g) / 8)
        b = cu(torch.randn(n, generator=g))
        rows = 12 if per_region else 3
        y = torch.empty(rows, n, device=DEV)
        x = latent[:, :, idx] if per_region else latent[:, 0, idx]
        probs.append((latent.data_ptr() + idx * 64 * 4, 6 * 64 if per_region else 4 * 6 * 64, w, b, y, rows, -1.0))
        refs.append((x.reshape(rows, 64).double() @ w.double().t() + b.double()).float())
    K.linear_multi(probs)
    dem = []
    for (_, _, _, _, y, rows, _), n in zip(probs, [s[2] for s in shapes]):
        wsq = cu(torch.rand(40, n, generator=g) / n)
        d = torch.empty(rows, 40, device=DEV)
        dem.append((y.data_ptr(), n, wsq, None, d, rows, 1e-8))
    K.linear_multi(dem)
    torch.cuda.synchronize()
    for (q, ref, dq) in zip(probs, refs, dem):
        assert_close(q[4], ref, 1e-5, "linear_multi plain")
        assert_close(dq[4], torch.rsqrt(ref.double().pow(2) @ dq[2].double().t() + 1e-8).float(), 1e-5, "linear_multi demod form")
    many = [(latent.data_ptr(), 64, probs[0][2], None, torch.empty(72, 96, device=DEV), 72, -1.0) for _ in range(101)]   # > 48: several launches
    K.linear_multi(many)
    ref = (latent.reshape(72, 64).double() @ probs[0][2].double().t()).float()
    for q in (many[0], many[47], many[48], many[100]):
        assert_close(q[4], ref, 1e-5, "linear_multi > 48 problems")


def test_generator_batched_modulations_equal_per_layer_modulations(monkeypatch):
    """Generator.forward without gradients computes all style modulations in one launch and all demodulations in a second
    (model.py:_layer_styles); E4S_B200_STYLE_BATCH=0 keeps one EqualLinear + one demod launch per layer.  Same image."""
    G, _ = _generator(64, 13)
    codes, mask, _, noise = O.synthetic_inputs(3, 12, 64, 128, seed=8, kind="blobs")
    args = ([cu(codes)], None, cu(mask))
    kw = dict(input_is_latent=True, noise=[cu(n) for n in noise])
    from e4s_b200 import kernels as K
    with torch.no_grad():
        K.LaunchStats.reset()
        a, _, fa = G(*args, **kw)
        batched = K.LaunchStats.launches
        monkeypatch.setenv("E4S_B200_STYLE_BATCH", "0")
        K.LaunchStats.reset()
        b, _, fb = G(*args, **kw)
        per_layer = K.LaunchStats.launches
    assert batched < per_layer - 20, (batched, per_layer)
    assert_close(a, b, 1e-5, "batched vs per-layer modulations: image")
    assert_close(fa, fb, 1e-5, "batched vs per-layer modulations: feats")
    monkeypatch.delenv("E4S_B200_STYLE_BATCH")
    c = cu(codes).requires_grad_(True)                  # gradients wanted: the differentiable per-layer path
    img, _, _ = G([c], None, cu(mask), **kw)
    img.square().mean().backward()
    assert c.grad is not None and torch.isfinite(c.grad).all() and float(c.grad.abs().max()) > 0


def test_graphed_synthesis_equals_eager_and_draws_fresh_noise():
    """e4s_b200.pipeline.GraphedSynthesis: the forward of one batch shape as a CUDA graph.  With fixed noise buffers a replay
    equals the eager forward, for the inputs of the CALL (not of the capture); with randomize_noise every replay
    draws new noise maps."""
    from types import SimpleNamespace
    from e4s_b200.networks import Net3
    from e4s_b200.pipeline import GraphedSynthesis, SynthesisPipeline
    from e4s_b200.stylegan2.modconv import LabelPyramid
    from e4s_b200.synthetic import load_synthetic
    opts = SimpleNamespace(num_seg_cls=6, remaining_layer_idx=13, out_size=64, train_G=False, start_from_latent_avg=False,
                           learn_in_w=False, fsencoder_type="psp")
    net = Net3(opts).eval()
    load_synthetic(net.G, salt=3)
    net = net.to(DEV)
    g = torch.Generator().manual_seed(12)
    synth = GraphedSynthesis(net, 6, (2, 6, 18, 512), (2, 1, 128, 128), randomize_noise=False)
    for trial in range(2):
        codes = cu(torch.randn(2, 6, 18, 512, generator=g))
        labels = cu(torch.randint(0, 6, (2, 1, 128, 128), generator=g).to(torch.uint8))
        with torch.no_grad():
            ref = net.gen_img(None, codes, LabelPyramid(labels[:, 0], 6), randomize_noise=False)[0]
        out = synth(codes, labels)
        assert_close(out, ref, 1e-5, f"replay {trial} vs the eager forward")     # (MMA warps race: equal to fp32 rounding)
    fresh = GraphedSynthesis(net, 6, (2, 6, 18, 512), (2, 1, 128, 128))
    a = fresh(codes, labels).clone()
    b = fresh(codes, labels).clone()
    assert not torch.equal(a, b), "randomize_noise: two replays must not share their noise maps"
    assert torch.isfinite(a).all() and torch.isfinite(b).all()
    with pytest.raises(RuntimeError):
        fresh(codes[:1], labels[:1])
    pipe = SynthesisPipeline(net, 6, depth=2, cuda_graph=True)
    t = pipe.submit(codes.cpu().pin_memory(), labels.cpu().pin_memory())
    img = pipe.result(t)
    assert tuple(img.shape) == (2, 3, 64, 64) and torch.isfinite(img).all()


def test_demod_gemm_form_equals_reference_formula():
    """e4s_demod_gemm_f32 (tiled small-GEMM kernel, x squared on load, rsqrt epilogue) == rsqrt(s^2 @ wsq^T + 1e-8) in fp64
    (model.py:279-281 in the shared-weight form) == the warp-per-output kernel e4s_demod_f32."""
    from e4s_b200 import kernels as K, _lib
    g = torch.Generator().manual_seed(31)
    for rows, cin, cout in ((192, 512, 512), (1, 32, 32), (37, 64, 36)):
        s = 1.0 + 0.3 * torch.randn(rows, cin, generator=g)
        wsq = torch.rand(cout, cin, generator=g) / cin
        ref = torch.rsqrt(s.double().pow(2) @ wsq.double().t() + 1e-8).float()
        sd, wd = cu(s), cu(wsq)
        out = K.demod(sd, wd)
        assert_close(out, ref, 1e-5, f"demod gemm form {rows}x{cin}x{cout}")
        old = torch.empty(rows, cout, device=DEV)
        _lib.check(_lib.load().e4s_demod_f32(_lib.ptr(sd), _lib.ptr(wd), _lib.ptr(old), rows, cin, cout, 1e-8, _lib.stream_ptr()), "e4s_demod_f32")
        assert_close(old, ref, 1e-5, "demod warp form")


@pytest.mark.parametrize("size,batch", [(32, 4), (64, 8), (128, 2)])
def test_discriminator_matches_reference_vectors(size, batch):
    """SURVEY section 8 f4: the StyleGAN2 discriminator (reference model.py:740-799) on this package's blur / fused-activation
    ops, against the reference's logits; and its input gradient (R1 regularisation differentiates through it) against the
    oracle's autograd."""
    import os
    from conftest import ROOT
    from oracle import disc_oracle as DO
    from e4s_b200.stylegan2.model import Discriminator
    gold = np.load(os.path.join(ROOT, "tests", "golden", "disc_vectors.npz"))
    D = Discriminator(size).eval()
    D.load_state_dict(O.synthetic_state({k: tuple(v.shape) for k, v in D.named_parameters()}, salt=size + 1), strict=False)
    st = {k: v.detach().clone() for k, v in D.state_dict().items()}
    D = D.to(DEV)
    x = DO.synthetic_inputs(batch, size, seed=size)
    xg = cu(x).requires_grad_(True)
    from e4s_b200.criteria.inversion_loss import conv_precision
    with conv_precision(True):                               # full-fp32 library convolutions for the comparison
        out = D(xg)
        out.sum().backward()
    assert_close(out, gold[f"d{size}/logits"], REL_TOL, f"discriminator {size}")
    xc = x.clone().requires_grad_(True)
    DO.discriminator_forward(st, xc, size).sum().backward()
    # the gradient of a leaky-ReLU stack is discontinuous where a pre-activation crosses zero; the few units that sit within
    # fp32 rounding of it take the other branch on the GPU (observed max-norm deviations 2e-3 ... 1.4e-2 with exact logits), so
    # the gradient is compared in the L2 sense: rel-L2 <= 2e-2, cosine >= 0.9998
    a, b = xg.grad.double().cpu().flatten(), xc.grad.double().flatten()
    rel_l2, cos = float((a - b).norm() / b.norm()), float(torch.dot(a, b) / (a.norm() * b.norm()))
    print(f"discriminator {size} input gradient: rel-L2 {rel_l2:.2e}, cosine {cos:.6f}")
    assert rel_l2 <= 2e-2 and cos >= 0.9998, (rel_l2, cos)


def test_bench_dump_outputs_do_not_depend_on_the_warmup(tmp_path):
    """`bench.py --dump-outputs` writes the images of the last timed step; the noise of the timed steps is seeded after the
    warm-up, so runs with different warm-up counts dump the same images up to the default kernels' accumulation order
    (different noise would differ by O(1)), and they are the images an eager recomputation of those steps returns."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    dumps = []
    for warmup in (1, 2):
        d = tmp_path / f"warmup{warmup}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", "256", "--batch", "2", "--steps", "2",
                              "--warmup", str(warmup), "--no-cpu-baseline", "--no-gpu-baseline", "--no-e2e", "--faceswap-pairs", "0",
                              "--gpen-batch", "0", "--inversion-batch", "0", "--inversion-steps", "0", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        dumps.append(np.load(d / "image.npy"))
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (2, 3, 256, 256) and np.isfinite(dumps[0]).all()
    assert_close(torch.from_numpy(dumps[1]), torch.from_numpy(dumps[0]), REL_TOL, "image dumped after 1 vs 2 warm-up steps")
    # the two timed steps again, eagerly, from bench.py's rank-0 seeds: weights (build_net), codes 100, label maps 200, noise 700
    import bench
    from e4s_b200.masks import labelMap2OneHot
    net = bench.build_net(256, 12, torch.device(DEV))
    codes = cu(torch.randn(2, 12, 18, 512, generator=torch.Generator().manual_seed(100)))
    onehot = labelMap2OneHot(cu(bench.face_label_maps(2, 12, "faces", seed=200)), 12)
    with torch.random.fork_rng(devices=[0]), torch.no_grad():
        torch.cuda.manual_seed(700)
        for _ in range(2):
            img = net.gen_img(None, codes, onehot)[0]
    assert_close(torch.from_numpy(dumps[0]), img, REL_TOL, "dumped image vs the eager recomputation of the last timed step")
