#!/usr/bin/env python
"""bench.py -- ZigMa denoiser hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one denoiser evaluation (ZigMa.forward at the per-GPU batch of the workload, bf16, synthetic weights /
latents) followed by the Euler update of the flow-matching sampler (transport/integrators.py:105-123).  The default
workload is BASELINE.json configs[1] (zigzag8_b1, bs=64 per GPU); --config selects one of the other BASELINE
configs, and the default run also measures them (a few evaluations each) into the `configs` block of its line.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how every field is obtained.

--impl reference: the reference's own implementation of the path on the HOST cores (no GPU, no import of the
product package): the pinned CPU restatement in oracle/ (the reference is Python and cannot travel to the GPU box),
same workload and batch, unscaled.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NUM_GRID = 50           # linspace(0, 1, 50): the sampler's time grid (49 evaluations per sample)

# BASELINE.json `configs` (configs[0] is the CPU correctness case: tests/).  Per-GPU batches: configs 3 / 4 are quoted as
# bs 256 / 128 "sharded across 8xB200" = 32 / 16 per GPU; model hyper-parameters from /root/reference/config/model/*.yaml.
WORKLOADS = {
    "zigzag8_b1": dict(
        cfg=dict(in_channels=4, embed_dim=640, depth=18, img_dim=32, patch_size=1, scan_type="zigzagN8", use_pe=2),
        bs=64, latent=(4, 32, 32), tokens=1024,
        desc="zigzag8_b1: ZigMa D=640 depth=18 img 32 patch 1 zigzagN8 (BASELINE configs[1])",
        scan_shapes=[("spatial", 1, 1024)]),
    "sweep2_b1": dict(
        cfg=dict(in_channels=4, embed_dim=640, depth=18, img_dim=32, patch_size=1, scan_type="v2", use_pe=2),
        bs=64, latent=(4, 32, 32), tokens=1024,
        desc="sweep2_b1: same dims, scan_type v2 = forward + backward sweep per layer, no permutation (BASELINE configs[2])",
        scan_shapes=[("sweep", 1, 1024)]),
    "faceshq1024": dict(
        cfg=dict(in_channels=4, embed_dim=768, depth=24, img_dim=128, patch_size=2, scan_type="zigzagN8"),
        bs=32, latent=(4, 128, 128), tokens=4096,
        desc="FacesHQ-1024 (s1024_zigzag8_b2_old.yaml): D=768 depth=24 128x128 latent patch 2 -> L=4096, bs 256 / 8 GPUs (BASELINE configs[3])",
        scan_shapes=[("spatial", 1, 4096)]),
    "ucf101_sst": dict(
        cfg=dict(in_channels=4, embed_dim=768, depth=24, img_dim=32, patch_size=2, scan_type="zzvideo_sst", use_pe=2, video_frames=16,
                 num_classes=101),
        bs=16, latent=(16, 4, 32, 32), tokens=4096,
        desc="UCF101 3d_zigzag8sst_b2: 16 frames x 16x16 tokens, factorised s/s/t scans, D=768 depth=24, bs 128 / 8 GPUs (BASELINE configs[4])",
        scan_shapes=[("spatial", 16, 256), ("temporal", 256, 16)]),    # (kind, sequences per sample, L)
}
DEFAULT = "zigzag8_b1"


def scan_algorithmic_bytes(Bt, E, L, N, s):
    """SURVEY.md section 8d: 4 s B E L (u, delta, z read; out written) + 2 s B N L (B, C) + 4 (E N + 2E)."""
    return 4 * s * Bt * E * L + 2 * s * Bt * N * L + 4 * (E * N + 2 * E)


def scan_mufu_floor_ms(Bt, E, L, N, sm_mhz=1965.0, n_sm=148):
    """Compute ceiling of the scan that sits ABOVE its HBM time: N exp2 per (b, e, l) for the state decays plus 4 for
    softplus (ex2 + lg2) and SiLU (ex2 + rcp) on the 16-lane/SM MUFU pipe (DESIGN.md 4.1)."""
    return (N + 4) * Bt * E * L / (n_sm * 16 * sm_mhz * 1e6) * 1e3


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None, "reasons": reasons,
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy kernel, burst)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's algorithm on the host cores.  NOTHING here imports zigma_b200.
# ------------------------------------------------------------------------------------------------
def cpu_reference_setup(name):
    import torch
    from oracle import zigma_oracle as zo, synth as osynth, c_oracle
    from oracle.shapes import zigma_state_shapes
    wl = WORKLOADS[name]
    zo.USE_C_SCAN = True                       # the plain-C OpenMP port of the recurrence (fp32)
    # all host cores for the C loops whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1 in every rank)
    c_oracle.set_threads(os.cpu_count() or 1)
    sd = osynth.synth_state_dict(zigma_state_shapes(wl["cfg"]), seed=0)
    cfg = dict(wl["cfg"], norm_epsilon=1e-5)
    return zo, osynth, sd, cfg, torch


def cpu_reference_eval(name, bs, state=None, nthreads=None):
    """One denoiser evaluation of workload `name` at batch `bs` through the CPU restatement of the reference path (torch
    GEMMs + the plain-C OpenMP scan, fp32).  Returns (seconds, state)."""
    state = state or cpu_reference_setup(name)
    zo, osynth, sd, cfg, torch = state
    if nthreads:
        torch.set_num_threads(nthreads)
    wl = WORKLOADS[name]
    x = osynth.synth_latents((bs,) + tuple(wl["latent"]), seed=0)
    t = torch.full((bs,), 0.5)
    y = torch.zeros(bs, dtype=torch.long) if wl["cfg"].get("num_classes", -1) > 0 else None
    with torch.no_grad():
        t0 = time.perf_counter()
        out = zo.zigma_forward(sd, cfg, x, t, y)
        dt = time.perf_counter() - t0
    assert torch.isfinite(out).all()
    return dt, state


def run_reference(args, rank):
    """--impl reference: the reference's own (CPU) implementation of the path, timed on the host cores -- the pinned CPU
    restatement in oracle/ (kind 'port': the Python reference cannot travel to the GPU box).  SAME workload and batch as
    the `ours` arm, unscaled; the number of timed evaluations is capped so that the run ends within a few minutes."""
    if rank != 0:
        return          # one host: rank 0 alone runs the CPU arm
    name = args.config
    wl = WORKLOADS[name]
    bs = args.bs or wl["bs"]
    cores = os.cpu_count() or 1
    threads = int(os.environ.get("ZIGMA_REF_THREADS", "0")) or min(cores, 32)      # torch intra-op threads; measured on the 128-core box: 55 s / evaluation with 32, 112 s with 128 (the C scan uses OpenMP's default: all cores)
    state = cpu_reference_setup(name)
    cpu_reference_eval(name, 1, state, threads)                  # page in / build the C oracle (not timed)
    budget_s = float(os.environ.get("ZIGMA_REF_BUDGET_S", "150"))
    t_first, _ = cpu_reference_eval(name, bs, state, threads)    # first full-batch evaluation = the warm-up
    n = max(1, min(args.steps, int(budget_s / max(t_first, 1e-3))))
    dts = [cpu_reference_eval(name, bs, state, threads)[0] for _ in range(n)]
    dt = sum(dts) / len(dts)
    val = bs * wl["tokens"] / dt
    import torch
    line = {
        "impl": "reference", "metric": f"denoiser tokens/s (bs*L*evals/s), {name}, Euler sampling loop",
        "value": val, "unit": "tokens/s", "n_gpus": args.gpus, "steps": n, "warmup": 1,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl['desc']}, bs={bs} (one host: rank 0 runs the whole CPU arm; the other ranks exit)",
                   "global_batch": bs, "seq_len": wl["tokens"],
                   "steps_note": f"requested steps={args.steps} warmup={args.warmup}; CPU evaluations cost {t_first:.1f} s each, so 1 warm-up and {n} timed evaluations are run (budget {budget_s:.0f} s)",
                   "denoiser_steps_per_s": 1.0 / dt},
        "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": cores, "kind": "port",
                         "sample": f"{n} denoiser evaluation(s) at the full bs={bs} (fp32 CPU restatement: torch GEMMs on {torch.get_num_threads()} threads + OpenMP C scan)"},
        "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# ours
# ------------------------------------------------------------------------------------------------
def reference_cuda_numbers(name, bs, n_iter=3):
    """The reference's vendored CUDA kernels (oracle/_ref, built from the unmodified sources for sm_100a) on this GPU:
    (a) selective_scan_cuda.fwd and causal_conv1d_fwd at the layer shape of the workload in the reference's own layout,
    (b) one denoiser evaluation through the reference's (restated) PyTorch glue around those kernels.  Returns None when
    oracle/_ref is absent.  (Runs in the `ours` arm only: it needs the GPU.)"""
    import torch
    from oracle import ref_cuda, zigma_oracle as zo
    if not (ref_cuda.available() and torch.cuda.is_available()):
        return None
    from zigma_b200 import synth, rms_norm_fn
    from oracle.shapes import zigma_state_shapes
    wl = WORKLOADS[name]
    cfg0 = wl["cfg"]
    dev = torch.device("cuda", torch.cuda.current_device())
    dtype = torch.bfloat16
    E, N = 2 * cfg0["embed_dim"], 16
    kind, nseq, L = wl["scan_shapes"][0]
    sb = bs * nseq

    def timeit(fn, n=n_iter, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n
    gen = torch.Generator(device=dev).manual_seed(0)
    xz = torch.randn(sb, 2 * E, L, device=dev, generator=gen).to(dtype)
    u, z = xz[:, :E], xz[:, E:]
    delta = (0.5 * torch.rand(E, sb * L, device=dev, generator=gen)).to(dtype).reshape(E, sb, L).transpose(0, 1)   # view like :323
    Bm = torch.randn(sb, 1, N, L, device=dev, generator=gen).to(dtype)
    Cm = torch.randn(sb, 1, N, L, device=dev, generator=gen).to(dtype)
    A = -0.5 * torch.rand(E, N, device=dev, generator=gen)
    Dp, bias = torch.randn(E, device=dev, generator=gen), 0.5 * torch.rand(E, device=dev, generator=gen)
    cw, cb = torch.randn(E, 4, device=dev, generator=gen).to(dtype), torch.randn(E, device=dev, generator=gen).to(dtype)
    out = {"scan_fwd_ms": timeit(lambda: ref_cuda.scan_fwd(u, delta, A, Bm, Cm, Dp, z, bias, True), 5),
           "conv_fwd_ms": timeit(lambda: ref_cuda.conv_fwd(u, cw, cb, True), 5),
           "layer_shape": f"{kind}: ({sb}, {E}, {L})"}
    from zigma_b200 import selective_scan_fn, causal_conv1d_fn
    out["ours_same_layout_scan_fwd_ms"] = timeit(lambda: selective_scan_fn(u, delta, A, Bm, Cm, Dp, z=z, delta_bias=bias, delta_softplus=True), 5)
    out["ours_same_layout_conv_fwd_ms"] = timeit(lambda: causal_conv1d_fn(u, cw, cb, "silu"), 5)
    del xz, u, z, delta, Bm, Cm
    # whole denoiser evaluation: restated reference glue + reference kernels
    sd = {k: v.to(dev) for k, v in synth.synth_state_dict(zigma_state_shapes(cfg0), seed=0, dtype=dtype).items()}
    norm = lambda x, w, b, residual=None, prenorm=False, residual_in_fp32=False, eps=1e-6: rms_norm_fn(
        x, w, b, residual=residual, prenorm=prenorm, residual_in_fp32=residual_in_fp32, eps=eps)
    zo.BACKEND = ref_cuda.backend(norm)
    x = torch.randn((bs,) + tuple(wl["latent"]), device=dev, generator=gen).to(dtype)
    t = torch.full((bs,), 0.5, device=dev, dtype=dtype)
    y = torch.zeros(bs, dtype=torch.long, device=dev) if cfg0.get("num_classes", -1) > 0 else None
    cfg = dict(cfg0, norm_epsilon=1e-5)
    try:
        with torch.no_grad():
            ms = timeit(lambda: zo.zigma_forward(sd, cfg, x, t, y), n_iter)
    finally:
        zo.BACKEND = {}
    out.update({"denoiser_eval_ms": ms, "tokens_per_s": bs * wl["tokens"] / (ms * 1e-3), "bs": bs, "dtype": "bf16",
                "what": "reference dis_mamba/dis_causal_conv1d CUDA kernels (sm_100a build of the unmodified sources) + the reference's PyTorch glue (restated), eager"})
    return out


def scan_roofline(name, bs, dev, step_ms=None, depth=None):
    """The dominant kernel (selective scan forward) timed alone at the layer shape(s) of the workload, token-major, z gathered
    through the zigzag table where the workload has one.  Returns the `roofline` object (first / dominant shape) with the
    other shapes of the workload under `shapes`."""
    import torch
    from zigma_b200 import zigzag_path
    from zigma_b200.selective_scan_interface import _scan_fwd
    wl = WORKLOADS[name]
    E, N = 2 * wl["cfg"]["embed_dim"], 16
    R = (wl["cfg"]["embed_dim"] + 15) // 16
    dtype = torch.bfloat16
    peak, how = measured_peaks()
    res = []
    for kind, nseq, L in wl["scan_shapes"]:
        sb = bs * nseq
        gen = torch.Generator(device=dev).manual_seed(0)
        xz = torch.randn(sb, L, 2 * E, device=dev, generator=gen).to(dtype)
        xc = torch.randn(sb, L, E, device=dev, generator=gen).to(dtype)
        dl = (0.5 * torch.rand(sb, L, E, device=dev, generator=gen)).to(dtype)
        xdbl = torch.randn(sb, L, R + 2 * N, device=dev, generator=gen).to(dtype)
        A = -0.5 * torch.rand(E, N, device=dev, generator=gen)
        Dp, bias = torch.randn(E, device=dev, generator=gen), 0.5 * torch.rand(E, device=dev, generator=gen)
        side = int(round(L ** 0.5))
        if kind == "sweep":
            perm = None
        elif side * side == L:
            perm = torch.from_numpy(zigzag_path(side)[1]).to(dev).to(torch.int32)
        else:
            perm = torch.arange(L - 1, -1, -1, device=dev, dtype=torch.int32)
        Bv = xdbl[:, :, R:R + N].permute(0, 2, 1).unsqueeze(1)
        Cv = xdbl[:, :, R + N:].permute(0, 2, 1).unsqueeze(1)
        outb = torch.empty(sb, L, E, device=dev, dtype=dtype).transpose(1, 2)
        call = lambda: _scan_fwd(xc.transpose(1, 2), dl.transpose(1, 2), A, Bv, Cv, Dp, xz[:, :, E:].transpose(1, 2), bias, True,
                                 z_rowmap=perm, want_last_state=False, out=outb)
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        n_it = 20
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(n_it):
            call()      # working set 4 x (sb L E 2 B) >> 126 MB L2 at every benchmark shape: each launch streams from HBM
        s1.record()
        torch.cuda.synchronize()
        kms = s0.elapsed_time(s1) / n_it
        abytes = scan_algorithmic_bytes(sb, E, L, N, 2)
        ach = abytes / (kms * 1e-3) / 1e9
        floor = scan_mufu_floor_ms(sb, E, L, N)
        from zigma_b200 import _lib as _zl
        res.append({"shape": f"{kind}: batch {sb} x dim {E} x seqlen {L}", "kernel": _zl.last_scan_kernel(), "ms_per_launch": kms, "algorithmic_bytes": abytes, "achieved": ach,
                    "frac": ach / peak, "hbm_floor_ms": abytes / (peak * 1e9) * 1e3, "compute_floor_ms": floor, "frac_of_compute_floor": floor / kms})
        del xz, xc, dl, xdbl, outb
    r0 = res[0]
    kname = res[0]["kernel"]
    traffic, tsrc = None, None
    if name == DEFAULT:     # DRAM bytes of one launch from this round's ncu capture of the kernel that actually ran
        for fn in ("r02b_scan_fwd_traffic.json", "r02_scan_fwd_traffic.json"):
            tp = os.path.join(ROOT, "profiles", fn)
            if os.path.exists(tp):
                tj = json.load(open(tp))
                if tj.get("kernel", "zg::scan_fwd_tma_kernel") in kname:
                    traffic, tsrc = tj.get("dram_bytes_per_launch"), tj.get("source")
                    break
    roof = {"bound": "hbm", "kernel": kname + " <bf16>: dstate 16, token-major, z gathered through the zigzag table",
            "achieved": r0["achieved"], "peak": peak, "unit": "GB/s", "frac": r0["frac"], "traffic": traffic, "traffic_source": tsrc,
            "peak_source": how, "ms_per_launch": r0["ms_per_launch"], "algorithmic_bytes": r0["algorithmic_bytes"],
            "hbm_floor_ms": r0["hbm_floor_ms"],
            "compute_floor_ms": r0["compute_floor_ms"], "frac_of_compute_floor": r0["frac_of_compute_floor"],
            "compute_floor_what": "MUFU pipe: (16 + 4) ex2/lg2/rcp per (b, e, l) at 16 lanes/SM/clk, 148 SMs, 1965 MHz -- the scan is compute-bound ABOVE its HBM time, so frac (of the HBM roofline) cannot exceed hbm_floor_ms / compute_floor_ms",
            "shapes": res}
    if step_ms and depth:
        per_layer = sum(r["ms_per_launch"] for r in res) if name != "ucf101_sst" else None
        launches = depth * (2 if name == "sweep2_b1" else 1)
        roof["launches_per_step"] = launches
        if per_layer is not None:
            roof["share_of_step"] = launches * r0["ms_per_launch"] / step_ms
        else:   # s, s, t rounds: 2/3 of the layers run the spatial shape, 1/3 the temporal one
            roof["share_of_step"] = (depth * 2 / 3 * res[0]["ms_per_launch"] + depth / 3 * res[1]["ms_per_launch"]) / step_ms
    return roof


def other_kernel_rooflines(name, bs, dev):
    """The other kernels of a layer of the workload, each timed alone (20 launches, CUDA events, working sets > L2) against the roofline
    that bounds it: conv and block tail -> HBM (algorithmic bytes), the four projections -> tensor pipe (in / out) or HBM (x_proj reads,
    dt_proj writes one (tokens, d_inner) tensor; their flops are negligible).  GEMMs also carry the library's (cuBLAS) time as the bar."""
    import torch
    import torch.nn.functional as F
    from zigma_b200 import zigzag_path, reverse_permut_np
    from zigma_b200.causal_conv1d_interface import _conv_fwd
    from zigma_b200.engine import block_tail
    from zigma_b200.gemm import linear_bf16
    wl = WORKLOADS[name]
    D = wl["cfg"]["embed_dim"]
    E, N, R = 2 * D, 16, (D + 15) // 16
    kind, nseq, L = wl["scan_shapes"][0]
    Bt = bs * nseq
    M = Bt * L
    dtype = torch.bfloat16
    hbm, _ = measured_peaks()
    pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    tf_peak = float(pk.get("bf16_tflops", 1666.9))          # burst figure: each kernel is timed alone

    def timeit(fn, n=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    out = []
    side = int(round(L ** 0.5))
    perm = torch.from_numpy(zigzag_path(side)[1]).to(dev).to(torch.int32) if (kind != "sweep" and side * side == L) else None
    rev = torch.from_numpy(reverse_permut_np(zigzag_path(side)[1])).to(dev).to(torch.int32) if perm is not None else None
    # conv: reads the x half of xz through the zigzag table, writes xc
    xz = torch.randn(Bt, L, 2 * E, device=dev).to(dtype)
    cw, cb = torch.randn(E, 4, device=dev).to(dtype), torch.randn(E, device=dev).to(dtype)
    xc = torch.empty(Bt, L, E, device=dev, dtype=dtype).transpose(1, 2)
    ms = timeit(lambda: _conv_fwd(xz[:, :, :E].transpose(1, 2), cw, cb, True, x_rowmap=perm, out=xc))
    by = 2 * 2 * M * E
    out.append({"kernel": "zg::conv_fwd_tok4_kernel<bf16> (causal conv1d + SiLU, rows gathered through the zigzag table)", "bound": "hbm", "ms_per_launch": ms,
                "algorithmic_bytes": by, "achieved": by / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": by / ms / 1e6 / hbm})
    del xz, xc
    # block tail: x, mix (bf16) + residual (fp32) in; residual (fp32), normed, modded (bf16) out
    x, mix = torch.randn(Bt, L, D, device=dev).to(dtype), torch.randn(Bt, L, D, device=dev).to(dtype)
    mods, res, nw = torch.randn(Bt, 3 * D, device=dev).to(dtype), torch.randn(Bt, L, D, device=dev), torch.ones(D, device=dev, dtype=dtype)
    ms = timeit(lambda: block_tail(x, mix, mods[:, :D], mods[:, D:2 * D], mods[:, 2 * D:], nw, res, rev, 1e-5))
    by = M * D * (2 + 2 + 4 + 4 + 2 + 2)
    out.append({"kernel": "zg::block_tail_row4_kernel<bf16> (gated residual + add + RMSNorm + modulate, un-permuting)", "bound": "hbm", "ms_per_launch": ms,
                "algorithmic_bytes": by, "achieved": by / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": by / ms / 1e6 / hbm})
    del x, mix, res
    # the four projections of a layer
    for pname, Nn, Kk, bound in (("in_proj", 2 * E, D, "tensor"), ("out_proj", D, E, "tensor"), ("x_proj", R + 2 * N, E, "hbm"), ("dt_proj", E, R, "hbm")):
        Kp = (Kk + 7) // 8 * 8
        a = torch.randn(M, Kp, device=dev).to(dtype)[:, :Kk]
        w = (torch.randn(Nn, Kp, device=dev) / Kk ** 0.5).to(dtype)[:, :Kk]
        c = torch.empty(M, Nn, device=dev, dtype=dtype)
        ms = timeit(lambda: linear_bf16(a, w, out=c))
        ms_lib = timeit(lambda: F.linear(a, w))
        ent = {"kernel": f"zg::gemm_bf16_tn_kernel {pname} ({M} x {Nn} x {Kk})", "bound": bound, "ms_per_launch": ms, "library_ms_per_launch": ms_lib}
        if bound == "tensor":
            fl = 2.0 * M * Nn * Kk
            ent.update({"algorithmic_flops": fl, "achieved": fl / ms / 1e9, "peak": tf_peak, "unit": "TFLOP/s", "frac": fl / ms / 1e9 / tf_peak})
        else:
            by = 2 * (M * Kk + Nn * Kk + M * Nn)
            ent.update({"algorithmic_bytes": by, "achieved": by / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": by / ms / 1e6 / hbm})
        out.append(ent)
        del a, w, c
    torch.cuda.empty_cache()
    return out


def run_workload(name, bs, K, W, dev, world, rank, use_graph=True, with_e2e=True, keep_outputs=False):
    """Builds the model of workload `name`, times K Euler steps (one CUDA graph for the whole K-step loop), the end-to-end
    leg with host buffers, and returns the measurements (with keep_outputs, also the final latents of the timed loop under
    "outputs").  Every rank calls this; collectives only when world > 1."""
    import torch
    import torch.distributed as dist
    from zigma_b200 import ZigMa, _lib, synth
    from zigma_b200.sharding import gather_latents
    from zigma_b200.engine import ZigMaEngine
    wl = WORKLOADS[name]
    dtype = torch.bfloat16
    model = ZigMa(device=dev, dtype=dtype, **wl["cfg"]).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth.synth_state_dict(shapes, seed=0, dtype=dtype))
    lat = tuple(wl["latent"])
    # initial noise indexed by the global sample id (weak scaling: bs per GPU fixed)
    z0 = torch.stack([synth.synth_latents(lat, seed=1000 + rank * bs + i) for i in range(bs)]).to(dev).to(dtype)
    y = torch.zeros(bs, dtype=torch.long, device=dev) if wl["cfg"].get("num_classes", -1) > 0 else None
    grid = torch.linspace(0, 1, NUM_GRID)
    ts_all, dts_all = grid.tolist(), (grid[1:] - grid[:-1]).tolist()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        # launches of OUR kernels per evaluation, counted on one eager (non-graph) pass
        os.environ["ZIGMA_CUDA_GRAPH"] = "0"
        eager = ZigMaEngine(model)
        tvec = torch.full((bs,), 0.5, device=dev, dtype=dtype)
        c0 = _lib.launch_count()
        eager._forward_impl(z0, tvec, y)
        per_eval = _lib.launch_count() - c0
        os.environ["ZIGMA_CUDA_GRAPH"] = "1" if use_graph else "0"
        model._engine = None
        model._engine = eng = ZigMaEngine(model)

        # K consecutive grid steps (wrapping around the 49-step grid if K > 49), the whole loop as one graph replay
        idx = [i % (NUM_GRID - 1) for i in range(K)]
        ts = [ts_all[i] for i in idx] + [0.0]
        dts = [dts_all[i] for i in idx]
        sample = lambda x: eng.sample_euler(x, ts, y, False, dts=dts)
        x = z0
        n_warm = max(1, -(-W // K))                # >= W warm-up steps (each replay = K steps)
        for _ in range(n_warm):
            x = sample(x)
        barrier()
        clocks = ClockSampler(dev.index or 0)
        if rank == 0:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda.profiler.start()     # no-op unless run under `ncu --profile-from-start off`
        e0.record()
        x = sample(z0)                  # exactly K steps
        full = gather_latents(x, bs * world, world)      # the single collective of the sampling job
        e1.record()
        barrier()
        torch.cuda.profiler.stop()
        outputs = {"latents": full.float().cpu().numpy()} if keep_outputs else None
        ms = e0.elapsed_time(e1)
        clk = clocks.stop() if rank == 0 else None
        if world > 1:
            tm = torch.tensor([ms], device=dev)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms = tm.item()
        assert torch.isfinite(full.float()).all()
        res = {"ms": ms, "ms_per_step": ms / K, "per_eval": per_eval, "clocks": clk, "bs": bs, "warm_steps": n_warm * K,
               "tokens_per_s": bs * world * wl["tokens"] * K / (ms * 1e-3), "outputs": outputs}

        if with_e2e:
            # ---- e2e: public API with HOST buffers: pinned latents/t H2D, forward, result D2H, every step
            hx = z0.cpu().pin_memory()
            ht = torch.empty(bs, dtype=dtype).pin_memory()
            hout = torch.empty_like(hx).pin_memory()
            dx = torch.empty_like(z0)
            tv = torch.empty(bs, device=dev, dtype=dtype)

            def e2e_step(i):
                ht.fill_(ts_all[i % (NUM_GRID - 1)])
                dx.copy_(hx, non_blocking=True)
                tv.copy_(ht, non_blocking=True)
                out = model(dx, tv, y) if y is not None else model(dx, tv)
                hout.copy_(out, non_blocking=True)
                torch.cuda.current_stream().synchronize()     # the caller reads the result on the host
            for i in range(3):
                e2e_step(i)
            barrier()
            t0 = time.perf_counter()
            for i in range(K):
                e2e_step(i)
            barrier()
            e2e_ms = (time.perf_counter() - t0) * 1e3
            if world > 1:
                tm = torch.tensor([e2e_ms], device=dev)
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                e2e_ms = tm.item()
            res["e2e"] = {"value": bs * world * wl["tokens"] * K / (e2e_ms * 1e-3), "unit": "tokens/s",
                          "h2d_bytes_per_step": z0.numel() * z0.element_size() + bs * 2, "d2h_bytes_per_step": z0.numel() * z0.element_size(),
                          "ms_per_step": e2e_ms / K, "api": "ZigMa.forward(x, t) with pinned host latents in, host velocity out"}
    del model, eng, eager
    torch.cuda.empty_cache()
    return res


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each array as <out_dir>/<name>.npy in float32, so that two builds run with the same arguments can be compared
    output for output.  An array larger than DUMP_LIMIT_BYTES is replaced by a fixed, seeded sample of its leading-dimension
    rows (sorted; the same rows for the same shape in every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > DUMP_LIMIT_BYTES:
            rows = np.random.default_rng(0).choice(a.shape[0], DUMP_LIMIT_BYTES // (a.nbytes // a.shape[0]), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=DEFAULT, choices=list(WORKLOADS))
    ap.add_argument("--bs", type=int, default=0, help="batch per GPU (default: the workload's BASELINE batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly (for ncu launch lists)")
    ap.add_argument("--no-train", action="store_true", help="skip the forward+backward (training step) side measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the side measurements of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the final latents of the timed sampling loop to DIR/latents.npy "
                    "(float32; inputs and weights are seeded, so runs with the same arguments can be compared)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    name = args.config
    wl = WORKLOADS[name]
    bs = args.bs or wl["bs"]

    main_res = run_workload(name, bs, K, W, dev, world, rank, use_graph=not args.no_graph, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main_res.pop("outputs"))
    roof = scan_roofline(name, bs, dev, main_res["ms_per_step"], wl["cfg"]["depth"]) if rank == 0 else None
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if name == DEFAULT and not args.no_configs:
        try:        # the rest of a layer, each kernel against its own roofline (side information next to `roofline`; rank 0 alone, after the job)
            roof["other_kernels"] = other_kernel_rooflines(name, bs, dev)
        except Exception as ex:
            roof["other_kernels"] = {"error": repr(ex)[:300]}

    ms, per_eval = main_res["ms"], main_res["per_eval"]
    line = {
        "metric": f"denoiser tokens/s (bs*L*evals/s), {name}, Euler sampling loop",
        "value": main_res["tokens_per_s"], "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": main_res["warm_steps"], "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{wl['desc']}, bs={bs}/GPU, fixed-grid Euler (linspace(0,1,50))",
                   "global_batch": bs * world, "seq_len": wl["tokens"], "parallelism": f"dp{world}",
                   "l2_policy": "no flush: per-step working set (xz alone >= 335 MB per layer) >> 126 MB L2",
                   "denoiser_steps_per_s": K / (ms * 1e-3), "cuda_graph": "one graph replay = the whole K-step Euler loop" if not args.no_graph else False,
                   "gemm": "hand-written tcgen05 (zg_gemm_bf16_tn)" if os.environ.get("ZIGMA_TCGEN05", "1") == "1" else "library (cuBLAS)",
                   "collective": "one all_gather of final latents, inside the timed region"},
        "clocks": main_res["clocks"],
        "e2e": main_res.get("e2e"),
        "gpu_launches": per_eval * K,
        "gpu_launches_per_eval": per_eval,
        "roofline": roof,
    }
    if not args.no_ref_cuda:
        try:
            rc = reference_cuda_numbers(name, bs)
        except Exception as ex:
            rc = {"error": repr(ex)[:300]}
        line["reference_cuda"] = rc
        if rc and "denoiser_eval_ms" in rc:
            line["speedup_vs_reference_cuda"] = rc["denoiser_eval_ms"] / (ms / K)
    if not args.no_configs and name == DEFAULT:
        # the other BASELINE configs, per GPU (rank 0 alone, after the timed job): a few evaluations each
        cfgs = {}
        for other in WORKLOADS:
            if other == name:
                continue
            try:
                obs = WORKLOADS[other]["bs"]
                r = run_workload(other, obs, 5, 3, dev, 1, 0, use_graph=not args.no_graph, with_e2e=False)
                ro = scan_roofline(other, obs, dev, r["ms_per_step"], WORKLOADS[other]["cfg"]["depth"])
                ent = {"workload": WORKLOADS[other]["desc"], "bs_per_gpu": obs, "seq_len": WORKLOADS[other]["tokens"], "steps": 5,
                       "ms_per_eval": r["ms_per_step"], "tokens_per_s_per_gpu": r["tokens_per_s"], "gpu_launches_per_eval": r["per_eval"],
                       "scan": [{k: s[k] for k in ("shape", "ms_per_launch", "frac", "frac_of_compute_floor")} for s in ro["shapes"]],
                       "scan_share_of_step": ro.get("share_of_step")}
                if not args.no_ref_cuda:
                    try:
                        rc = reference_cuda_numbers(other, obs, n_iter=2)
                        if rc:
                            ent["reference_cuda"] = {k: rc[k] for k in ("denoiser_eval_ms", "scan_fwd_ms", "conv_fwd_ms", "layer_shape") if k in rc}
                            ent["speedup_vs_reference_cuda"] = rc["denoiser_eval_ms"] / r["ms_per_step"]
                    except Exception as ex:
                        ent["reference_cuda"] = {"error": repr(ex)[:200]}
                    torch.cuda.empty_cache()
                cfgs[other] = ent
            except Exception as ex:
                cfgs[other] = {"error": repr(ex)[:300]}
                torch.cuda.empty_cache()
        line["configs"] = cfgs
    if not args.no_train and world == 1 and name == DEFAULT:
        # side measurement (not the headline): one flow-matching training step, forward + backward, of the same
        # denoiser at bs 16 -- ours vs the reference's forward/backward CUDA kernels in the reference's glue
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "train_bench.py")], capture_output=True, text=True, timeout=600,
                               env=dict(os.environ, BS="16", DTYPE="bf16", CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local))))
            js = [l for l in r.stdout.splitlines() if l.startswith("{")]
            line["train_step"] = json.loads(js[-1]) if js else {"error": (r.stderr or r.stdout)[-300:]}
        except Exception as ex:
            line["train_step"] = {"error": repr(ex)[:300]}
    if not args.no_cpu_baseline:
        # bounded sample of the same workload on the host cores: ONE evaluation at a reduced batch (the full batch is what
        # `--impl reference` times); reported per token
        cores = os.cpu_count() or 1
        threads = int(os.environ.get("ZIGMA_REF_THREADS", "0")) or min(cores, 32)
        sbs = max(1, min(bs, 8))
        st = cpu_reference_setup(name)
        cpu_reference_eval(name, 1, st, threads)
        dt, _ = cpu_reference_eval(name, sbs, st, threads)
        line["cpu_baseline"] = {"value": sbs * wl["tokens"] / dt, "unit": "tokens/s", "cores": cores, "kind": "port",
                                "sample": f"1 denoiser evaluation at bs={sbs} of the same workload (fp32 CPU restatement of the reference path: torch GEMMs on {threads} threads + OpenMP C scan on all cores); the full bs={bs} evaluation is what --impl reference times"}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
