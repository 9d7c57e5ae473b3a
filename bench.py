#!/usr/bin/env python
"""Benchmark of the E4S synthesis hot path (BASELINE.json configs[1]: 1024x1024 synthesis, batch 16 per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one mask-guided synthesis pass (`Net3.gen_img`, the call scripts/face_swap.py:273 and
scripts/optimization.py:216 make) over a batch of `--batch` synthetic faces per GPU: random-init weights of the
real architecture, random W+ codes, 12-region masks derived from the reference's example parsing masks
(tests/golden fixture), fresh Gaussian noise per layer like the reference (model.py:333).

Prints ONE JSON line (rank 0).  `value` = faces/s with inputs resident in HBM; `e2e` = the same call fed from
pinned HOST buffers (codes + uint8 label maps copied H2D, final images copied D2H inside the timed region);
`roofline` = the modulated-convolution kernels' achieved TFLOP/s (algorithmic FLOPs / CUDA-event time inside
the timed region) against the measured bf16 tensor peak; `cpu_baseline` = one full 1024x1024 face through the
reference-structured CPU oracle on the host cores.  `--impl reference` times that CPU path alone.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (the images; with N ranks, rank 0's, which
are all N ranks' images when `--gather` is set) to DIR/image.npy.  Weights,
codes, masks and the noise of the timed steps are seeded, so runs with the same arguments get the same inputs and the dumps
of two builds can be compared element for element.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = "{size}x{size} faces/sec (mask-guided StyleGAN2 synthesis, {ncls} regions, K=13)"
ALGO_GFLOP_PER_FACE = {1024: 148.1, 512: 118.8, 256: 89.5}   # 3x3 modulated convs, SURVEY.md section 8d
# Numbers only a profiler can give (dram__bytes per conv launch, tensor-pipe activity) come from a COMMITTED ncu --set full
# capture of the 17 conv launches of one step of the default workload: profiles/ncu_conv_static.json, written by
# tools/ncu_summary.py together with the SHA-256 of the kernel sources it was taken from.  bench.py reports them as
# "static" and flags them "stale" when the sources have changed since (they are never silently reused).
NCU_STATIC = os.path.join(ROOT, "profiles", "ncu_conv_static.json")
KERNEL_SOURCES = ("e4s_b200/csrc/modconv_tcr.cu", "e4s_b200/csrc/modconv_tch.cu", "e4s_b200/csrc/tc_ptx.cuh")


def kernel_source_hash() -> str:
    import hashlib
    h = hashlib.sha256()
    for rel in KERNEL_SOURCES:
        with open(os.path.join(ROOT, rel), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def ncu_static():
    if not os.path.exists(NCU_STATIC):
        return None
    d = json.load(open(NCU_STATIC))
    d["stale"] = d.get("kernel_source_sha16") != kernel_source_hash()
    return d


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=16, help="faces per GPU per step")
    ap.add_argument("--ncls", type=int, default=12)
    ap.add_argument("--mask", default="faces", choices=["faces", "iid"], help="region-mask distribution")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the reference's own GPU formulation (cuDNN grouped convolutions)")
    ap.add_argument("--no-loss-nets", action="store_true", help="inversion: skip the full-loss (ID + l2 + LPIPS + parsing) measurement")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--eager", action="store_true",
                    help="time `value` / `e2e` on eager launches (Net3.gen_img per step) instead of one CUDA-graph replay per step "
                         "(e4s_b200.pipeline.GraphedSynthesis); the eager figure is reported either way (`eager`)")
    ap.add_argument("--gather", action="store_true",
                    help="N>1: also all-gather every rank's images inside the timed step (the path itself has no exchange step)")
    ap.add_argument("--faceswap-pairs", type=int, default=None,
                    help="also time steps 3-5 of scripts/face_swap.py (encoder, shape/texture swap, generator, blending masks) on "
                         "this many (driven, target) pairs per GPU; default: BASELINE configs[3]'s 64 pairs split over the ranks "
                         "(strong scaling: 8 per GPU at 8 GPUs, capped at 16 per GPU); 0 disables")
    ap.add_argument("--gpen-batch", type=int, default=16,
                    help="also time GPEN-BFR-512's FullGenerator (stage 2 of scripts/face_swap.py:208; e4s_b200.gpen) on this many "
                         "512x512 faces per GPU; 0 disables")
    ap.add_argument("--inversion-batch", type=int, default=8,
                    help="also run one complete 100-step inversion of this many faces AT ONCE per GPU (independent faces, one "
                         "optimiser over [B, ncls, 1280]); 0 disables")
    ap.add_argument("--inversion-steps", type=int, default=20,
                    help="also time this many steps of the texture-vector optimisation (scripts/optimization.py:209-232, "
                         "l2 loss) on one face per GPU; 0 disables")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the images of the last one as DIR/image.npy (float32; a fixed, seeded "
                         "sample of them when they exceed %d elements; with N ranks, rank 0's images)" % DUMP_MAX_ELEMENTS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------ inputs
def face_label_maps(batch: int, ncls: int, kind: str, seed: int) -> torch.Tensor:
    """uint8 [batch, 1, 512, 512] region labels.  'faces': the two example parsing masks of the reference
    (example/input/faceswap/*_mask.png, converted 19->12 classes; stored in tests/golden), cycled with
    mirror images; 'iid': independent uniform labels per pixel (worst case: every tile sees every class)."""
    g = torch.Generator().manual_seed(seed)
    if kind == "iid":
        return torch.randint(0, ncls, (batch, 1, 512, 512), generator=g, dtype=torch.uint8)
    gold = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"))
    base = [torch.from_numpy(gold["mask/source_cls12"]), torch.from_numpy(gold["mask/target_cls12"])]
    base += [b.flip(1) for b in base]
    maps = [base[i % 4].clamp(max=ncls - 1) for i in range(batch)]
    return torch.stack(maps).unsqueeze(1).contiguous()


def build_net(size: int, ncls: int, device):
    from e4s_b200.networks import Net3
    from e4s_b200.synthetic import synthetic_state      # seeded stand-in for the checkpoint that cannot be downloaded
    opts = types.SimpleNamespace(fsencoder_type="psp", remaining_layer_idx=13, num_seg_cls=ncls, out_size=size,
                                 train_G=False, start_from_latent_avg=True, learn_in_w=False)
    net = Net3(opts).eval()
    state = synthetic_state({k: tuple(v.shape) for k, v in net.state_dict().items()}, salt=size)
    net.load_state_dict(state)
    net = net.to(device)
    net.latent_avg = torch.zeros(18, 512, device=device)
    return net


# -------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


class NvmlClockSampler:
    """Same samples through NVML from a thread (about one per 5 ms, so a 250-ms timed region gets dozens instead of the
    one or two `nvidia-smi -lms 100` yields).  The device is found by UUID: NVML does not see CUDA_VISIBLE_DEVICES."""

    def __init__(self, index: int):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(index).uuid)
        self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        self.samples, self.bits, self.power = [], 0, 0.0
        self.stop_flag = threading.Event()

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                self.power = max(self.power, nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        self.stop_flag.set()
        self.thread.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap,
                 "hw_power_brake_slowdown": nv.nvmlClocksEventReasonHwPowerBrakeSlowdown}
        reasons = sorted(k for k, bit in names.items() if self.bits & bit)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_min_mhz": float(min(self.samples)), "sm_max_mhz": self.max_sm,
                "reasons": reasons, "samples": len(self.samples), "power_w_max": round(self.power, 1), "source": "nvml"}


def make_clock_sampler(index: int):
    try:
        return NvmlClockSampler(index)
    except Exception:
        return ClockSampler(index)


# --------------------------------------------------------------------------------------- CPU baseline
def cpu_reference_face(size: int, ncls: int, state=None, seed: int = 1, want_inputs: bool = False):
    """One full synthesis forward of ONE face through the reference-structured CPU oracle (all host threads)."""
    from oracle import e4s_oracle as O
    if state is None:
        state = O.synthetic_state(O.generator_param_shapes(size), salt=size)
    codes, mask, _, noise = O.synthetic_inputs(1, ncls, size, 512, seed=seed)
    t0 = time.perf_counter()
    with torch.no_grad():
        img, _ = O.generator_forward(state, codes, mask, noise, size, 13)
    dt = time.perf_counter() - t0
    return (dt, state, img, (codes, mask, noise)) if want_inputs else (dt, state, img)


def gpu_baseline_leg(net, size: int, ncls: int, batch: int, dev):
    """The reference's own GPU formulation on this GPU (oracle/gpu_baseline.py: per-region loop, per-sample weights, cuDNN
    grouped convolution with groups = batch, model.py:287-318 / 395-398) - the stronger baseline of BASELINE.md section 4.
    TF32 off (fp32 parity setting) and on (torch's default for cuDNN convolutions = what the reference runs with)."""
    from oracle import e4s_oracle as O, gpu_baseline as GB
    gst = {k[2:]: v.detach() for k, v in net.state_dict().items() if k.startswith("G.")}
    out = {"what": "reference-structured forward (12 grouped cuDNN convolutions + mask-sum per masked layer) on the same GPU, "
                   "weights and inputs resident, torch " + torch.__version__, "runs": []}
    for b in sorted({1, batch}):
        codes, mask, _, noise = O.synthetic_inputs(1, ncls, size, 512, seed=21)
        codes, mask = codes.to(dev).expand(b, -1, -1, -1).contiguous(), mask.to(dev).expand(b, -1, -1, -1).contiguous()
        noise = [n.to(dev) for n in noise]
        for tf32 in (False, True):
            try:
                from e4s_b200.criteria.inversion_loss import conv_precision      # sets the legacy AND the new cuDNN precision switch
                bench_before = torch.backends.cudnn.benchmark
                torch.backends.cudnn.benchmark = True                                  # let cuDNN pick its fastest algorithms
                with torch.no_grad(), conv_precision(not tf32):
                    GB.generator_forward(gst, codes, mask, noise, size, 13)            # warm-up (cuDNN algorithm search)
                    torch.cuda.synchronize()
                    reps = 3 if b == 1 else 2
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(reps):
                        GB.generator_forward(gst, codes, mask, noise, size, 13)
                    e1.record()
                    torch.cuda.synchronize()
                torch.backends.cudnn.benchmark = bench_before
                ms = e0.elapsed_time(e1) / reps
                out["runs"].append({"batch": b, "tf32": tf32, "ms_per_step": ms, "faces_per_sec": b / (ms * 1e-3)})
            except Exception as exc:                                   # e.g. out of memory at the full batch: reported
                out["runs"].append({"batch": b, "tf32": tf32, "error": repr(exc)[:200]})
                torch.cuda.empty_cache()
        del codes, mask, noise
        torch.cuda.empty_cache()
    ok = [r for r in out["runs"] if "faces_per_sec" in r]
    if ok:
        out["best_fp32_faces_per_sec"] = max((r["faces_per_sec"] for r in ok if not r["tf32"]), default=None)
        out["best_tf32_faces_per_sec"] = max((r["faces_per_sec"] for r in ok if r["tf32"]), default=None)
    return out


_PROBE_BEST_S = {}


def pick_cpu_threads(ncls: int, probe: int = 256) -> int:
    """torch's default (one thread per logical core) oversubscribes this path's convolutions on many-core hosts; give the CPU
    arm its best setting: one 256x256 forward (convolutions of the size class that dominates the timed 1024x1024 face: a
    64x64 probe, as in round 1, favoured too few threads) per candidate thread count, after a 64x64 warm-up of the thread
    pool, and keep the fastest.  Candidates 16 / 32 / 64 (8 and all-cores lost every probe of this round's runs and all-cores
    alone could take a minute): the probe has to leave the default bench run within minutes."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (16, 32, 64) if c <= ncpu}) or [ncpu]
    best, best_t, state = cands[-1], float("inf"), None
    for c in cands:
        torch.set_num_threads(c)
        cpu_reference_face(64, ncls)
        dt, state, _ = cpu_reference_face(probe, ncls, state, seed=3)
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    _PROBE_BEST_S[probe] = best_t
    return best


def run_reference(args):
    """The reference's own CPU implementation of the path (oracle port: the python reference cannot travel to
    the GPU box), timed on the host cores.  Each step = one full face."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pick_cpu_threads(args.ncls)
    state = None
    for _ in range(max(args.warmup, 1)):
        _, state, _ = cpu_reference_face(args.size, args.ncls, state)
    times = []
    for i in range(args.steps):
        dt, state, img = cpu_reference_face(args.size, args.ncls, state, seed=2 + i)
        times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"image": img})
    sec = float(np.mean(times))
    val = 1.0 / sec
    cores = torch.get_num_threads()
    sample = f"{args.steps} steps x one full {args.size}x{args.size} face (B=1, {args.ncls} regions, K=13), fp32, torch CPU"
    line = {"impl": "reference", "metric": METRIC.format(size=args.size, ncls=args.ncls), "value": val, "unit": "faces/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": max(args.warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.size}x{args.size} synthesis, CPU reference path, 1 face per step", "ncls": args.ncls,
                       "faces_per_step": 1,
                       "note": "the CPU arm times ONE face per step (a 16-face step would take minutes); the unit is faces/s, so the "
                               "ratio to the GPU arm's 16-face steps stands"},
            "cpu_baseline": {"value": val, "unit": "faces/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "faces/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(json.dumps(line))


# ------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    t_run0 = time.perf_counter()
    import torch.distributed as dist
    from e4s_b200 import kernels as K
    from e4s_b200.dist import gather_images
    from e4s_b200.masks import labelMap2OneHot

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (the product path has no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    B, size, ncls = args.batch, args.size, args.ncls
    if args.faceswap_pairs is None:
        args.faceswap_pairs = min(16, max(1, 64 // world))
    net = build_net(size, ncls, dev)
    g = torch.Generator().manual_seed(100 + rank)
    codes_host = torch.randn(B, ncls, 18, 512, generator=g).pin_memory()
    labels_host = face_label_maps(B, ncls, args.mask, seed=200 + rank).pin_memory()
    images_host = torch.empty(B, 3, size, size).pin_memory()
    codes_dev = codes_host.to(dev)
    onehot_dev = labelMap2OneHot(labels_host.to(dev), ncls)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_eager():
        with torch.no_grad():
            img, _, _ = net.gen_img(None, codes_dev, onehot_dev)
            return gather_images(img) if (world > 1 and args.gather) else img

    # the same forward for this batch shape captured once and replayed as one CUDA graph per step (fresh noise per replay);
    # inputs resident in HBM are copied device-to-device into the graph's static buffers inside the timed region
    from e4s_b200.pipeline import SynthesisPipeline, GraphedSynthesis
    labels_dev = labels_host.to(dev)
    synth, graph_error = None, None
    if not args.eager:
        try:
            synth = GraphedSynthesis(net, ncls, codes_dev.shape, labels_dev.shape, dev)
        except Exception as exc:                          # reported in the line (config.execution), never hidden: time eager launches
            graph_error = repr(exc)[:300]
            print(f"bench.py: CUDA-graph capture of the forward failed, timing eager launches instead: {graph_error}", file=sys.stderr)
            args.eager = True
            torch.cuda.synchronize()

    def step_graph():
        img = synth(codes_dev, labels_dev)
        return gather_images(img) if (world > 1 and args.gather) else img

    step_device = step_eager if args.eager else step_graph

    # end to end through the package's streaming API: pinned host codes + uint8 label maps in, pinned host images out,
    # every step; H2D / generator / D2H on three streams (e4s_b200/pipeline.py), all copies inside the timed region
    pipe = SynthesisPipeline(net, ncls, depth=2, device=dev, cuda_graph=not args.eager)

    def step_e2e():
        pipe.submit(codes_host, labels_host)

    def timed(fn, steps, warmup, sample_clocks=False, kernel_timing=False, finish=None):
        for _ in range(warmup):
            fn()
        barrier()
        sampler = make_clock_sampler(local) if sample_clocks else None
        if sampler:
            sampler.start()
        profile_range = sample_clocks and os.environ.get("E4S_BENCH_PROFILE_RANGE") == "1"
        if profile_range:                             # ncu --profile-from-start off: the launch list is the timed region
            torch.cuda.profiler.start()
        K.LaunchStats.reset(timing=kernel_timing)
        torch.cuda.manual_seed(700 + rank)            # the timed steps' noise maps do not depend on what ran before them
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        if finish is not None:
            finish()                                  # the timing stream waits for the copy streams
        e1.record()
        barrier()
        if profile_range:
            torch.cuda.profiler.stop()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if sampler else None
        launches, summary = K.LaunchStats.launches, (K.LaunchStats.summary() if kernel_timing else {})
        K.LaunchStats.reset(False)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, clocks, launches, summary, out

    ms, clocks, launches, _, last = timed(step_device, args.steps, args.warmup, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"image": last})        # before the next pass overwrites the graph's static image
    del last
    faces = B * world * args.steps
    value = faces / (ms * 1e-3)
    # the same K steps on eager launches: once clean, once with CUDA events around EVERY launch (per-kernel times for the
    # roofline / `kernels` breakdown; the events cost time themselves, so this pass is not the reported value)
    ms_eager, _, launches_eager, _, _ = timed(step_eager, args.steps, args.warmup)
    ms_inst, _, _, summary, _ = timed(step_eager, args.steps, args.warmup, kernel_timing=True)
    eager = {"value": faces / (ms_eager * 1e-3), "ms_per_step": ms_eager / args.steps, "gpu_launches": launches_eager,
             "ms_per_step_with_per_launch_events": ms_inst / args.steps}

    leg_s, _t_leg = {}, [t_run0]

    def leg_done(name):                                   # wall-clock seconds per section of this run (host side; for the record)
        torch.cuda.synchronize()
        now = time.perf_counter()
        leg_s[name] = round(now - _t_leg[0], 1)
        _t_leg[0] = now

    leg_done("setup+value+eager passes")
    e2e = None
    if not args.no_e2e:
        ms2, _, _, _, _ = timed(step_e2e, args.steps, max(args.warmup, 3), finish=pipe.drain)
        e2e = {"value": faces / (ms2 * 1e-3), "unit": "faces/s", "ms_per_step": ms2 / args.steps,
               "h2d_bytes_per_step": int(codes_host.numel() * 4 + labels_host.numel()),
               "d2h_bytes_per_step": int(images_host.numel() * 4),
               "api": "e4s_b200.pipeline.SynthesisPipeline.submit (3 streams, depth 2" + (")" if args.eager else ", forward as one CUDA graph)")}

    # ---- the path's only collective (SURVEY 8e): all-gather of the final images, alone and overlapped with the next step
    leg_done("e2e")
    gather = None
    if world > 1:
        with torch.no_grad():
            def one_step():                      # a private copy: the graph's static image is overwritten by the next replay
                return net.gen_img(None, codes_dev, onehot_dev)[0] if synth is None else synth(codes_dev, labels_dev).clone()
            img = one_step()
            for _ in range(2):
                gather_images(img)
            barrier()
            reps = 5
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(reps):
                gathered = gather_images(img)
            g1.record()
            barrier()
            alone = g0.elapsed_time(g1) / reps
            # overlapped: the gather of step i runs on a side stream while step i + 1 computes
            side = torch.cuda.Stream()
            o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            o0.record()
            prev = img
            for _ in range(reps):
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    gathered = gather_images(prev)
                prev = one_step()
                torch.cuda.current_stream().wait_stream(side)
            o1.record()
            barrier()
            overlapped = o0.elapsed_time(o1) / reps
        t = torch.tensor([alone, overlapped], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        alone, overlapped = float(t[0]), float(t[1])
        recv = float(img.numel() * 4 * (world - 1))
        gather = {"collective": "ncclAllGather (all_gather_into_tensor) of the final images", "bytes_per_rank_in": img.numel() * 4,
                  "bytes_per_rank_received": recv, "ms_alone": alone, "recv_GBps_per_rank": recv / (alone * 1e-3) / 1e9,
                  "ms_step_plus_overlapped_gather": overlapped, "ms_step": ms / args.steps,
                  "overlap_cost_ms": overlapped - ms / args.steps,
                  "nvlink_note": "NVLink 5 gives 900 GB/s per direction and GPU; a 16-face step's images are 201 MB per rank"}
        del gathered, img

    # ---- roofline of the dominant kernel family: the modulated 3x3 convolutions
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        pk = json.load(open(peaks_path))
        peak_tf, peak_src = float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"])), "measured (MEASURED_PEAKS.json, sustained bf16)"
        hbm_gbs = float(pk["hbm_gbs"])
    else:
        peak_tf, peak_src, hbm_gbs = 1590.0, "fallback (B200_PROFILING.md)", 6650.0
    roofline, kernels = None, {}
    static = ncu_static()
    default_workload = (size, B, ncls, args.mask) == (1024, 16, 12, "faces")
    for name, (n, kms, work) in summary.items():
        kernels[name] = {"launches": n, "ms": round(kms, 3), "share": round(kms / ms_inst, 4)}
    conv_names = [n for n in summary if n.startswith("e4s_modconv3x3")]
    if conv_names:
        n = sum(summary[k][0] for k in conv_names)
        kms = sum(summary[k][1] for k in conv_names)
        flops = sum(summary[k][2] for k in conv_names)
        top = max(conv_names, key=lambda k: summary[k][1])
        ach = flops / (kms * 1e-3) / 1e12
        roofline = {"kernel": f"modulated 3x3 convolutions (all 17 StyledConv layers; dominant entry point {top})",
                    "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                    "traffic": (static or {}).get("dram_bytes_per_launch") if default_workload else None,
                    "tensor_pipe_active_pct_ncu": (static or {}).get("tensor_pipe_active_pct") if default_workload else None,
                    "static": None if (static is None or not default_workload) else
                              {"what": "traffic and tensor_pipe_active_pct_ncu are NOT measured in this run: they come from the committed ncu "
                                       "--set full capture of the 17 conv launches of one step", "source": static.get("source"),
                               "kernel_source_sha16": static.get("kernel_source_sha16"), "stale": static["stale"]},
                    "peak_source": peak_src, "algorithmic_gflop_per_face": flops / 1e9 / (B * args.steps), "launches": n,
                    "avg_launch_ms": kms / n, "share_of_step": kms / ms_inst,
                    "timed_in": f"an eager pass of the same {args.steps} steps with CUDA events around every launch "
                                f"({ms_inst / args.steps:.2f} ms/step; the reported value's pass carries no per-launch events)",
                    "note": "achieved = ALGORITHMIC fp32 FLOPs / event time; the kernel issues 3 bf16 MMAs per algorithmic MAC "
                            "(split-bf16 for fp32 parity) and 4x MACs on up-sampling layers, so tensor-pipe activity is ~3-12x "
                            "this fraction (ncu sm__pipe_tensor_cycles_active in profiles/)"}

    # ---- BASELINE configs[2]: regional latent optimisation of one face per GPU (forward + backward + Adam per step)
    leg_done("gather+roofline")
    inversion = None
    if args.inversion_steps > 0:
        from e4s_b200.optimization import invert
        for prm in net.parameters():
            prm.requires_grad = False
        g2 = torch.Generator().manual_seed(300 + rank)
        sv = 0.5 * torch.randn(1, ncls, 1280, generator=g2).to(dev)
        onehot1 = onehot_dev[:1].contiguous()
        with torch.no_grad():
            target, _, _ = net.gen_img(None, net.cal_style_codes(0.5 * torch.randn(1, ncls, 1280, generator=g2).to(dev)), onehot1)
        invert(net, target, onehot1, style_vectors=sv, steps=3)                      # warm-up (allocator, weight prep)
        barrier()
        K.LaunchStats.reset(False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _, _, hist = invert(net, target, onehot1, style_vectors=sv, steps=args.inversion_steps)
        e1.record()
        barrier()
        ims = e0.elapsed_time(e1) / args.inversion_steps
        inv_launches = K.LaunchStats.launches
        if world > 1:
            tt = torch.tensor([ims], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ims = float(tt.item())
        # where the step goes: per-entry CUDA-event times of 5 further steps (event overhead makes these steps slower)
        K.LaunchStats.reset(timing=True)
        invert(net, target, onehot1, style_vectors=sv, steps=5)
        torch.cuda.synchronize()
        inv_kernels = {k: {"launches_per_step": v[0] / 5, "ms_per_step": round(v[1] / 5, 3)} for k, v in K.LaunchStats.summary().items()}
        K.LaunchStats.reset(False)
        graphed = None
        try:
            invert(net, target, onehot1, style_vectors=sv, steps=6, cuda_graph=True)          # capture warm-up
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            gstats = {}
            _, _, ghist = invert(net, target, onehot1, style_vectors=sv, steps=100, cuda_graph=True, stats=gstats)
            g1.record()
            barrier()
            # one complete 100-step inversion of one face: 3 eager steps + graph capture + 96 replays, all inside the timed call
            gtot = g0.elapsed_time(g1)
            if world > 1:
                tg = torch.tensor([gtot], device=dev)
                dist.all_reduce(tg, op=dist.ReduceOp.MAX)
                gtot = float(tg.item())
            graphed = {"ms_total_100_steps": gtot, "ms_per_replayed_step": gstats.get("replay_ms_per_step"), "loss_first": float(ghist[0]),
                       "loss_last": float(ghist[-1]), "faces_per_sec_100_steps": world / (gtot * 1e-3)}
        except Exception as exc:                                  # reported, never hidden
            graphed = {"error": repr(exc)[:300]}
        batched = None
        if args.inversion_batch > 1:
            # independent faces optimised side by side: the low-resolution layers of one face cannot fill the GPU
            try:
                nb = args.inversion_batch
                onehot_b = onehot_dev[:nb].contiguous() if onehot_dev.shape[0] >= nb else onehot_dev[:1].expand(nb, -1, -1, -1).contiguous()
                svb = 0.5 * torch.randn(nb, ncls, 1280, generator=g2).to(dev)
                with torch.no_grad():
                    target_b, _, _ = net.gen_img(None, net.cal_style_codes(0.5 * torch.randn(nb, ncls, 1280, generator=g2).to(dev)), onehot_b)
                invert(net, target_b, onehot_b, style_vectors=svb, steps=6, cuda_graph=True)                   # capture warm-up
                barrier()
                b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                b0.record()
                bstats = {}
                _, _, bhist = invert(net, target_b, onehot_b, style_vectors=svb, steps=100, cuda_graph=True, stats=bstats)
                b1.record()
                barrier()
                btot = b0.elapsed_time(b1)
                if world > 1:
                    tb = torch.tensor([btot], device=dev)
                    dist.all_reduce(tb, op=dist.ReduceOp.MAX)
                    btot = float(tb.item())
                batched = {"faces_per_gpu": nb, "ms_total_100_steps": btot, "ms_per_replayed_step": bstats.get("replay_ms_per_step"),
                           "loss_first": float(bhist[0]), "loss_last": float(bhist[-1]),
                           "faces_per_sec_100_steps": nb * world / (btot * 1e-3)}
                del target_b, svb, onehot_b
            except Exception as exc:                              # reported, never hidden
                batched = {"error": repr(exc)[:300]}
        full_loss = None
        if not args.no_loss_nets:
            # the reference's default loss (scripts/optimization.py:88-122: 0.1 ID + 1.0 l2 + 0.8 LPIPS x3 scales + 0.1 parsing) on
            # seeded stand-in loss networks (their checkpoints cannot be downloaded), target features cached, whole step graphed
            try:
                from e4s_b200.criteria import InversionLoss
                from e4s_b200.synthetic import load_synthetic_losses
                crit = InversionLoss()
                load_synthetic_losses(crit, 11)
                crit = crit.to(dev)
                invert(net, target, onehot1, style_vectors=sv, steps=3, criterion=crit)           # warm-up (cuDNN algorithm choice)
                barrier()
                l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                l0.record()
                _, _, lhist = invert(net, target, onehot1, style_vectors=sv, steps=args.inversion_steps, criterion=crit)
                l1.record()
                barrier()
                lms = l0.elapsed_time(l1) / args.inversion_steps
                invert(net, target, onehot1, style_vectors=sv, steps=6, criterion=crit, cuda_graph=True)      # capture warm-up
                barrier()
                q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                q0.record()
                qstats = {}
                _, _, qhist = invert(net, target, onehot1, style_vectors=sv, steps=100, criterion=crit, cuda_graph=True, stats=qstats)
                q1.record()
                barrier()
                qtot = q0.elapsed_time(q1)
                # what the reference's loop pays in addition: the target image through all three networks every step
                with torch.no_grad():
                    for _ in range(2):
                        crit.set_target(target)
                    barrier()
                    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    r0.record()
                    for _ in range(5):
                        crit.set_target(target)
                    r1.record()
                    barrier()
                # the loss networks with cuDNN's TF32 convolutions: what torch (and so the reference's script) runs by default
                tf32_ms = None
                try:
                    crit.exact = False
                    invert(net, target, onehot1, style_vectors=sv, steps=6, criterion=crit, cuda_graph=True)
                    barrier()
                    tstats = {}
                    invert(net, target, onehot1, style_vectors=sv, steps=40, criterion=crit, cuda_graph=True, stats=tstats)
                    barrier()
                    tf32_ms = tstats.get("replay_ms_per_step")
                finally:
                    crit.exact = True
                full_loss = {"lambdas": {"id": 0.1, "l2": 1.0, "lpips": 0.8, "face_parsing": 0.1}, "ms_per_step_eager": lms,
                             "ms_per_replayed_step_tf32_loss_networks": tf32_ms,
                             "ms_per_replayed_step": qstats.get("replay_ms_per_step"), "ms_total_100_steps": qtot,
                             "faces_per_sec_100_steps": world / (qtot * 1e-3), "loss_first": float(qhist[0]), "loss_last": float(qhist[-1]),
                             "target_feature_pass_ms": r0.elapsed_time(r1) / 5,
                             "note": "loss networks = library convolutions (cuDNN; exact fp32 = InversionLoss's default, TF32 = torch's); target-image features cached once per face - the "
                                     "reference recomputes them every step (target_feature_pass_ms each); seeded stand-in weights"}
                del crit
            except Exception as exc:                                  # reported, never hidden
                full_loss = {"error": repr(exc)[:300]}
        inversion = {"steps_timed": args.inversion_steps, "full_loss": full_loss, "ms_per_step": ims, "batched": batched, "launches_per_step": inv_launches / args.inversion_steps,
                     "cuda_graph": graphed, "kernels": inv_kernels,
                     "faces_per_sec_100_steps": world / (ims * 100 * 1e-3), "loss_first": float(hist[0]), "loss_last": float(hist[-1]),
                     "config": f"one {size}x{size} face per GPU, {ncls} regions, Adam lr 1e-2, l2 loss, fresh noise per step"}

    # ---- BASELINE configs[3]: face swapping, steps 3-5 of scripts/face_swap.py on (driven, target) pairs, sharded like faces
    leg_done("inversion")
    faceswap = None
    if args.faceswap_pairs > 0:
        try:
            from e4s_b200.face_swap import swap_faces
            P = args.faceswap_pairs
            g3 = torch.Generator().manual_seed(400 + rank)
            driven, target = torch.randn(P, 3, size, size, generator=g3).to(dev), torch.randn(P, 3, size, size, generator=g3).to(dev)
            labs = face_label_maps(2 * P, ncls, args.mask, seed=500 + rank)[:, 0].to(dev)
            d_lab, t_lab = labs[0::2].contiguous(), labs[1::2].contiguous()        # source / target example masks, alternating
            fs_steps = max(3, args.steps // 2)
            for _ in range(2):
                swap_faces(net, driven, target, d_lab, t_lab)
            barrier()
            K.LaunchStats.reset(False)
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(fs_steps):
                res = swap_faces(net, driven, target, d_lab, t_lab)
            f1.record()
            barrier()
            fms = f0.elapsed_time(f1) / fs_steps
            fs_launches = K.LaunchStats.launches / fs_steps
            if world > 1:
                tf = torch.tensor([fms], device=dev)
                dist.all_reduce(tf, op=dist.ReduceOp.MAX)
                fms = float(tf.item())
            faceswap = {"pairs_per_gpu": P, "steps_timed": fs_steps, "ms_per_step": fms, "pairs_per_sec": P * world / (fms * 1e-3),
                        "launches_per_step": fs_launches,
                        "config": f"{size}x{size} driven + target faces and their {ncls}-class parsing maps resident in HBM -> RGI encoder on "
                                  f"both, shape swap, texture swap, MLPs, generator, blending masks (e4s_b200.face_swap.swap_faces)"}
            del driven, target, res
        except Exception as exc:                                      # reported, never hidden; the headline metric stands on its own
            faceswap = {"error": repr(exc)[:300]}

    # ---- SURVEY section 8f.2: GPEN's generator on the same kernels (512x512 restoration, stage 2 of every swap)
    leg_done("faceswap")
    gpen = None
    if args.gpen_batch > 0:
        try:
            from e4s_b200.gpen.gpen_model import FullGenerator
            from e4s_b200.synthetic import load_synthetic
            gm = FullGenerator(512, 512, 8, channel_multiplier=2, narrow=1).eval()
            load_synthetic(gm, salt=512, parameters_only=True)         # the blur / up-sampling FIR buffers keep their registered values
            gm = gm.to(dev)
            gx = torch.randn(args.gpen_batch, 3, 512, 512, generator=torch.Generator().manual_seed(600 + rank)).to(dev)
            g_steps = max(3, args.steps // 2)
            with torch.no_grad():
                for _ in range(3):
                    gm(gx)
                barrier()
                K.LaunchStats.reset(False)
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                for _ in range(g_steps):
                    gm(gx)
                p1.record()
                barrier()
            gms = p0.elapsed_time(p1) / g_steps
            g_launches = K.LaunchStats.launches / g_steps
            if world > 1:
                tg2 = torch.tensor([gms], device=dev)
                dist.all_reduce(tg2, op=dist.ReduceOp.MAX)
                gms = float(tg2.item())
            gpen = {"faces_per_gpu": args.gpen_batch, "steps_timed": g_steps, "ms_per_step": gms,
                    "faces_per_sec": args.gpen_batch * world / (gms * 1e-3), "launches_per_step": g_launches,
                    "config": "GPEN-BFR-512 FullGenerator (size 512, 8 mapping layers, channel multiplier 2, concatenated encoder maps), "
                              "512x512 inputs resident in HBM, random-init weights"}
            del gm, gx
        except Exception as exc:                                      # reported, never hidden
            gpen = {"error": repr(exc)[:300]}

    leg_done("gpen")
    gpu_base = None
    if rank == 0 and world == 1 and not args.no_gpu_baseline:
        try:
            gpu_base = gpu_baseline_leg(net, size, ncls, B, dev)
            if gpu_base.get("best_fp32_faces_per_sec"):
                gpu_base["speedup_vs_fp32"] = value / gpu_base["best_fp32_faces_per_sec"]
            if gpu_base.get("best_tf32_faces_per_sec"):
                gpu_base["speedup_vs_tf32"] = value / gpu_base["best_tf32_faces_per_sec"]
        except Exception as exc:                                      # reported, never hidden
            gpu_base = {"error": repr(exc)[:300]}

    leg_done("gpu_baseline")
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        pick_cpu_threads(ncls)                                        # also warms the thread pool / allocator
        # the timed CPU face runs with THIS net's generator weights, so that its image is also the parity reference
        gst = {k[2:]: v.detach().cpu() for k, v in net.state_dict().items() if k.startswith("G.")}
        dt, _, cpu_img, (pc, pm, pn) = cpu_reference_face(size, ncls, gst, want_inputs=True)
        with torch.no_grad():
            gpu_img, _, _ = net.G([pc.to(dev)], None, pm.to(dev), input_is_latent=True, noise=[n.to(dev) for n in pn])
            # the same face as sample 5 of a full batch: batching must not change a face
            pcb = torch.randn(B, *pc.shape[1:], generator=torch.Generator().manual_seed(77))
            pmb = labelMap2OneHot(labels_host.to(dev), ncls).clone()
            slot = min(5, B - 1)
            pcb[slot] = pc[0]
            pmb[slot] = pm[0].to(dev)
            batch_img, _, _ = net.G([pcb.to(dev)], None, pmb, input_is_latent=True, noise=[n.to(dev) for n in pn])
        d = (gpu_img.cpu().double() - cpu_img.double())
        db = (batch_img[slot:slot + 1].cpu().double() - cpu_img.double())
        ref_max, ref_rms = float(cpu_img.abs().max()), float(cpu_img.double().pow(2).mean().sqrt())
        parity = {"what": f"one {size}x{size} face, {ncls} regions, K=13, fixed noise: e4s_b200 (default kernels) vs the CPU oracle",
                  "max_rel": float(d.abs().max()) / ref_max, "rel_rms": float(d.pow(2).mean().sqrt()) / ref_rms,
                  "in_batch_max_rel": float(db.abs().max()) / ref_max, "in_batch_rel_rms": float(db.pow(2).mean().sqrt()) / ref_rms,
                  "tolerance": 1e-3}
        del gpu_img, batch_img
        dt256 = _PROBE_BEST_S.get(256) or cpu_reference_face(256, ncls)[0]      # BASELINE configs[0]'s size: the probe's best run
        cpu = {"value": 1.0 / dt, "unit": "faces/s", "cores": torch.get_num_threads(), "kind": "port",
               "value_256x256": 1.0 / dt256,
               "host_logical_cpus": os.cpu_count(),
               "sample": f"one full {size}x{size} face (B=1, {ncls} regions, K=13) through the reference-structured CPU "
                         f"oracle (fp32, torch CPU; thread count = fastest of 16/32/64 on a 256x256 probe)"}

    leg_done("cpu_baseline+parity")
    if rank == 0:
        line = {"metric": METRIC.format(size=args.size, ncls=args.ncls), "value": value, "unit": "faces/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"{size}x{size} synthesis, batch {B} per GPU, {ncls} regions, K=13 (BASELINE configs[1])",
                           "global_batch": B * world, "mask": args.mask, "noise": "fresh N(0,1) per layer per step",
                           "execution": ("eager launches (Net3.gen_img)" + (f"; graph capture failed: {graph_error}" if graph_error else "")) if args.eager else
                                        "one CUDA-graph replay per step (e4s_b200.pipeline.GraphedSynthesis; codes + label maps copied into its static buffers every step)",
                           "l2": "activations per layer (>= 0.5 GB at the top resolutions) exceed the 126 MB L2; no flush needed",
                           "parallelism": (f"dp{world}: faces sharded across ranks, weights replicated, no data-path collective"
                                           + (" + NCCL all-gather of the final images" if args.gather else "")) if world > 1 else "single GPU"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "eager": eager, "roofline": roofline, "cpu_baseline": cpu,
                f"parity_{size}": parity, "gpu_baseline": gpu_base, "gather": gather,
                "kernels": kernels, "leg_seconds": leg_s, "hbm_peak_gbs": hbm_gbs, "inversion": inversion, "faceswap": faceswap, "gpen": gpen}
        emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_ELEMENTS = 1 << 23                          # 32 MiB of float32: a dump stays below 64 MB


def dump_outputs(outdir: str, arrays) -> None:
    """Each tensor as <outdir>/<name>.npy in float32.  One with more than DUMP_MAX_ELEMENTS elements is replaced by its
    elements at a fixed, seeded set of flat indices (sorted, 1-D): the same set for the same shape in every run."""
    os.makedirs(outdir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMENTS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(outdir, name + ".npy"), t.cpu().numpy())


_OUT_FD = None


def emit(text: str) -> None:
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout when
    NCCL_DEBUG is set, as it is on the GPU boxes), so main() points file descriptor 1 at stderr for the whole run and the
    result line goes to the process's original stdout."""
    if _OUT_FD is None:
        print(text, flush=True)
    else:
        data = (text + "\n").encode()
        while data:
            data = data[os.write(_OUT_FD, data):]


def main():
    global _OUT_FD
    args = parse_args()
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
