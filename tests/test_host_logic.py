"""Host-side logic that needs no GPU: weight folding, state-dict contract, batched LocalMLPs."""
import math
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import e4s_oracle as O
from conftest import assert_close


def test_fold_upsample_kernels_matches_convT_plus_blur():
    """4 parity kernels == conv_transpose2d(stride 2) followed by the [1,3,3,1] blur (model.py:287-300)."""
    from e4s_b200.stylegan2.modconv import fold_upsample_kernels
    g = torch.Generator().manual_seed(0)
    cin, cout, h = 5, 7, 6
    w = torch.randn(cout, cin, 3, 3, generator=g)
    x = torch.randn(2, cin, h, h + 1, generator=g)
    for blur in (O.make_fir((1, 3, 3, 1), 4.0), torch.rand(4, 4, generator=g)):   # symmetric and arbitrary FIR
        ref = O.upfirdn2d(F.conv_transpose2d(x, w.transpose(0, 1), stride=2), blur, pad=(1, 1))
        folded = fold_upsample_kernels(w, blur)
        out = torch.zeros_like(ref)
        for py in range(2):
            for px in range(2):
                out[:, :, py::2, px::2] = F.conv2d(x, folded[py * 2 + px], padding=1)
        assert_close(out, ref, 1e-5)


def test_region_selection_equals_mask_sum():
    """Selecting each pixel's own-region conv == the reference's sum_c mask_c * conv_c for one-hot masks."""
    st = O.synthetic_state({"conv.weight": (1, 8, 6, 3, 3), "conv.modulation.weight": (6, 512),
                            "conv.modulation.bias": (6,), "noise.weight": (1,), "activate.bias": (8,)})
    codes, mask, label, _ = O.synthetic_inputs(2, 4, 16, 16, seed=4)
    x = torch.randn(2, 6, 8, 8)
    nz = torch.randn(2, 1, 16, 16)
    ref = O.styled_conv(x, codes[:, :, 0], mask, nz, st, "", True, True)
    seg = O.nearest_resize(mask, 16).argmax(1)
    per_cls = torch.stack([O.styled_conv(x, codes[:, c, 0], None, nz, st, "", True, False) for c in range(4)], 1)
    sel = torch.gather(per_cls, 1, seg[:, None, None].expand(-1, 1, 8, -1, -1))[:, 0]
    assert torch.equal(sel, ref) or float((sel - ref).abs().max()) < 1e-6


def test_state_dict_contract():
    from e4s_b200.networks import Net3
    opts = types.SimpleNamespace(fsencoder_type="psp", remaining_layer_idx=13, num_seg_cls=12, out_size=64,
                                 train_G=False, start_from_latent_avg=True, learn_in_w=False)
    net = Net3(opts)
    sd = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    want = {}
    want.update(O.generator_param_shapes(64, prefix="G."))
    want.update(O.mlp_param_shapes(12))
    want.update(O.encoder_param_shapes())
    for k, shape in want.items():
        assert sd.get(k) == tuple(shape), (k, sd.get(k), shape)
    extra = [k for k in sd if k not in want and not k.startswith("G.style.")]
    assert not extra, extra
    assert all(not p.requires_grad for p in net.G.parameters())


def test_local_mlps_need_the_gpu_kernel():
    """cal_style_codes runs on the library's own small-GEMM kernel: no CPU / PyTorch fallback (a CPU tensor raises the
    reference's pybind message); the numerical checks are tests/test_parity_gpu.py::test_local_mlps_*."""
    from e4s_b200.networks import Net3
    opts = types.SimpleNamespace(fsencoder_type="psp", remaining_layer_idx=13, num_seg_cls=12, out_size=32,
                                 train_G=False, start_from_latent_avg=True, learn_in_w=False)
    net = Net3(opts).eval()
    net.latent_avg = torch.zeros(18, 512)
    for p in net.MLPs.parameters():
        p.requires_grad = False
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        net.cal_style_codes(torch.randn(1, 12, 1280))


def test_bench_reference_arm_emits_contract_line(tmp_path):
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints one JSON line with the contract's keys;
    run here at 64x64 so that it takes seconds."""
    import json
    import os
    import subprocess
    import sys
    from conftest import ROOT
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "64", "--steps", "1",
                          "--warmup", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "faces/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "faces/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["steps"] == 1 and line["n_gpus"] == 1 and line["gpu_launches"] == 0
    img = np.load(tmp_path / "image.npy")
    assert img.dtype == np.float32 and img.shape == (1, 3, 64, 64) and np.isfinite(img).all()


def test_dropin_overlay_resolves_reference_import_paths():
    """e4s_b200.dropin.install() points the reference's module names at this package (run in a subprocess: it edits
    sys.modules).  Works without the reference checkout on sys.path - the GPU box has none."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import e4s_b200.dropin as d; d.install()\n"
        "from src.models.networks import Net3\n"
        "from src.models.stylegan2.model import Generator, StyledConv\n"
        "from src.models.stylegan2.op import upfirdn2d, fused_leaky_relu, FusedLeakyReLU, conv2d_gradfix\n"
        "from src.models.encoders.psp_encoders import FSEncoder_PSP\n"
        "from src.pretrained.gpen.face_model.gpen_model import FullGenerator\n"
        "from src.utils.swap_face_mask import swap_head_mask_revisit_considerGlass\n"
        "import e4s_b200.networks, e4s_b200.gpen.gpen_model, e4s_b200.masks\n"
        "assert Net3 is e4s_b200.networks.Net3 and FullGenerator is e4s_b200.gpen.gpen_model.FullGenerator\n"
        "assert swap_head_mask_revisit_considerGlass is e4s_b200.masks.swap_head_mask_revisit_considerGlass\n"
        "print('ok')\n") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=os.path.dirname(ROOT))
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]


def test_package_synthetic_state_equals_the_oracles():
    """bench.py builds its random-init models with e4s_b200.synthetic (the product package may not import the oracle); the
    golden vectors were generated with the oracle's copy of the recipe.  The two are bit-identical, and loading parameters
    only leaves GPEN's registered FIR buffers equal to what the oracle's GPEN state holds."""
    from e4s_b200.synthetic import synthetic_state, load_synthetic
    from oracle import gpen_oracle as GO
    from e4s_b200.gpen.gpen_model import FullGenerator
    shapes = dict(O.generator_param_shapes(64))
    shapes.update(O.mlp_param_shapes(12))
    shapes.update(O.encoder_param_shapes())
    a, b = synthetic_state(shapes, salt=64), O.synthetic_state(shapes, salt=64)
    assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
    m = FullGenerator(64, 512, 8)
    load_synthetic(m, salt=64, parameters_only=True)
    ref = GO.synthetic_state(64, salt=64)
    got = m.state_dict()
    assert got.keys() == ref.keys()
    for k in ref:
        assert torch.allclose(got[k], ref[k], rtol=0, atol=1e-7), k


def test_up2_polyphase_index_math():
    """The index arithmetic of csrc/upfirdn2d.cu:upfirdn2d_up2_kernel (parity of the taps that meet a sample, the 2x4 input
    window of four consecutive outputs, arithmetic shifts on negative positions) restated in Python against the oracle's
    zero-stuff / pad / convolve definition, for asymmetric FIRs and pads."""
    import numpy as np

    def emulate(x, fir, pad0, pad1):
        planes, h, w = x.shape
        oh, ow = h * 2 + pad0 + pad1 - 3, w * 2 + pad0 + pad1 - 3
        kf = fir[::-1, ::-1]
        y = np.zeros((planes, oh, ow), np.float32)
        for oy in range(oh):
            my0 = oy - pad0
            py = my0 & 1
            iy0 = (my0 + py) >> 1
            for q in range(ow // 4):
                base = 4 * q - pad0
                c0 = (base + (base & 1)) >> 1
                v = np.zeros((planes, 2, 4), np.float32)
                for a in range(2):
                    for c in range(4):
                        if 0 <= iy0 + a < h and 0 <= c0 + c < w:
                            v[:, a, c] = x[:, iy0 + a, c0 + c]
                for j in range(4):
                    mx0 = base + j
                    px = mx0 & 1
                    cj = ((mx0 + px) >> 1) - c0
                    assert 0 <= cj <= 2
                    y[:, oy, 4 * q + j] = sum(v[:, a, cj] * kf[2 * a + py][px] + v[:, a, cj + 1] * kf[2 * a + py][px + 2] for a in range(2))
        return y

    rng = np.random.default_rng(0)
    for h, w, p0, p1 in [(8, 8, 2, 1), (6, 10, 1, 2), (7, 8, 2, 1), (5, 6, 3, 4), (4, 4, 0, 3)]:
        assert (w * 2 + p0 + p1 - 3) % 4 == 0
        x = rng.standard_normal((3, h, w)).astype(np.float32)
        fir = rng.standard_normal((4, 4)).astype(np.float32)
        ref = O.upfirdn2d(torch.from_numpy(x)[None], torch.from_numpy(fir), up=2, down=1, pad=(p0, p1))[0].numpy()
        assert np.abs(emulate(x, fir, p0, p1) - ref).max() < 1e-5, (h, w, p0, p1)


def test_proposed_upsampling_dataflow_spec():
    """tools/ubench/upconv_dataflow.py - the executable specification of the round-2 kernel design (DESIGN.md section 10): one
    tap-free GEMM per 8x16 pixel patch, then horizontal and vertical combination of the per-tap products - equals
    conv_transpose2d + blur; each output parity combines exactly six (neighbour, tap) products per axis."""
    import importlib.util
    import os
    import numpy as np
    from conftest import ROOT
    spec = importlib.util.spec_from_file_location("upconv_dataflow", os.path.join(ROOT, "tools", "ubench", "upconv_dataflow.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.self_check(seed=3) < 1e-12
    c = mod.axis_coefficients(np.array([1.0, 3.0, 3.0, 1.0]) / 4.0)
    assert [(c[p] != 0).sum() for p in range(2)] == [6, 6]


def test_fold_upsample_vertical_equals_convT_blur():
    """H-form weight folding (vertical half of the blur into the weights, horizontal half as six epilogue terms per output
    parity; specification tools/ubench/hform_dataflow.py) == conv_transpose2d(stride 2) + upfirdn2d blur of the oracle."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "ubench"))
    import hform_dataflow as H
    from e4s_b200.stylegan2.modconv import fold_upsample_vertical
    g = torch.Generator().manual_seed(3)
    for taps in ([1., 3., 3., 1.], [1., 2., 4., 3.]):
        f = torch.tensor(taps)
        fir = torch.outer(f, f)
        fir = fir / fir.sum() * 4
        w = torch.randn(5, 4, 3, 3, generator=g)
        x = torch.randn(1, 4, 6, 7, generator=g)
        v, fx = fold_upsample_vertical(w, fir)
        out = H.combine_horizontal(H.gemm_rows(x[0], v.double()), torch.tensor(fx, dtype=torch.float64))
        u = torch.nn.functional.conv_transpose2d(x, w.transpose(0, 1), stride=2)
        ref = O.upfirdn2d(u, fir, pad=(1, 1))[0]
        assert float((out - ref.double()).abs().max() / ref.abs().max()) < 1e-5
    assert fold_upsample_vertical(w, torch.randn(4, 4, generator=g)) is None      # not separable -> polyphase form


@pytest.mark.parametrize("size,K", [(64, 5), (256, 13), (1024, 13), (256, 17)])
def test_generator_style_schedule_follows_the_reference_latent_indexing(size, K):
    """Generator._schedule (what the batched modulation launch is built from) = the latent index and the per-region / global
    choice the reference's forward makes layer by layer (model.py:639-657): conv1 <- 0, to_rgb1 <- 1, then per resolution
    (up conv, conv, to_rgb) <- (i, i + 1, i + 2) with i = 1, 3, 5, ...; per-region styles while i < K on masked layers."""
    from e4s_b200.stylegan2.model import Generator
    G = Generator(size, 512, 8, split_layer_idx=5, remaining_layer_idx=K)
    sched = G._schedule()
    assert len(sched) == 2 + 3 * len(G.to_rgbs) and [s[1] for s in sched[:2]] == [0, 1] and all(s[2] for s in sched[:2])
    assert sched[0][0] is G.conv1 and sched[1][0] is G.to_rgb1
    i = 1
    for r, to_rgb in enumerate(G.to_rgbs):
        up, conv, rgb = sched[2 + 3 * r: 5 + 3 * r]
        assert (up[0], conv[0], rgb[0]) == (G.convs[2 * r], G.convs[2 * r + 1], to_rgb)
        assert (up[1], conv[1], rgb[1]) == (i, i + 1, i + 2)
        if i < K:
            assert up[2] == G.convs[2 * r].mask_op and conv[2] == G.convs[2 * r + 1].mask_op
            assert rgb[2] == (to_rgb.mask_op if (K == 17 or i + 2 != K) else False)
        else:
            assert not (up[2] or conv[2] or rgb[2])
        # a layer that receives per-region styles must be a masked layer (its kernel indexes the styles by label)
        for mod, _, per_region in (up, conv, rgb):
            assert mod.mask_op or not per_region
        i += 2
    assert i + 1 == G.n_latent


def test_encoder_stride2_weights_on_space_to_depth_equal_the_strided_convolution():
    """encoders/psp_encoders.py:_conv_planes_s2d: a stride-2 3x3 convolution = a stride-1 convolution of the space-to-depth
    tensor with the re-indexed weights, of which exactly the taps 0, 1, 3, 4 are non-zero (host arithmetic only)."""
    import torch.nn.functional as F
    from e4s_b200.encoders.psp_encoders import _conv_planes_s2d, TAPS_S2D
    g = torch.Generator().manual_seed(0)
    w = torch.randn(8, 4, 3, 3, generator=g)
    x = torch.randn(2, 4, 10, 12, generator=g)
    planes = _conv_planes_s2d(w)
    w4 = (planes[0].float() + planes[1].float())[0]                     # [9, Cout, 4 C]: bf16 hi + lo ~ fp32 to 2^-16
    assert [bool(w4[t].abs().max() > 0) for t in range(9)] == [bool((TAPS_S2D >> t) & 1) for t in range(9)]
    b, c, h, wd = x.shape
    x4 = x.permute(0, 2, 3, 1).reshape(b, h // 2, 2, wd // 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(b, h // 2, wd // 2, 4 * c)
    out = F.conv2d(x4.permute(0, 3, 1, 2), w4.reshape(3, 3, 8, 4 * c).permute(2, 3, 0, 1), padding=1)
    ref = F.conv2d(x, w, stride=2, padding=1)
    assert float((out - ref).abs().max()) < 1e-4 * float(ref.abs().max())
