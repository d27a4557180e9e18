"""bench.py -- BASELINE.json's metric: Mpix/s of GRL-Base x4 SR on 256x256 tiles (released hyper-parameters:
window 32, stripes 64x64, df 2, CAB on, pixelshuffle head), batch-sharded over the GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's own CPU PyTorch path
    python bench.py --workload cfg2|cfg3|cfg5 ...                  # the other BASELINE configs (lines kept in profiles/)
    python bench.py --scaling strong ...                           # cfg4's global batch of 128 fixed as N grows
    python bench.py --dump-outputs DIR ...                         # also write the last timed step's output as .npy

One "step" = one forward of the hot path over one batch of synthetic tiles (cfg5: one 1280x720 frame through the
tiled-inference loop, tiles sharded over the ranks).  Prints ONE JSON line (rank 0).
Weights and inputs are seeded, so the same arguments give the same inputs on every run and build; --dump-outputs lets
two builds be compared output for output.
`value` is device-resident throughput; `e2e` goes through the public nn.Module call with pinned HOST buffers
(H2D of inputs + ground truth, forward, reference PSNR on the device, D2H of the per-image PSNR) and ends with the
only collective this path has -- the all-gather of (index, psnr) pairs (NCCL).
The kernel-level roofline is timed in a SEPARATE pass after the headline loop (CUDA events around every attention
launch on the launching stream), so no event records sit inside `value` or `e2e`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree bench.py runs from may be read-only: leave no bytecode caches in it
# keep stdout to the single JSON line: libraries below us (NCCL's version banner, for one) write to file descriptor 1.
# Everything that is not the result line goes to stderr; the result line goes to the saved real stdout.
sys.stdout.flush()
RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(result):
    RESULT_OUT.write(json.dumps(result) + "\n")
    RESULT_OUT.flush()


WORKLOADS = {
    # name: (variant, task, scale, tile, tiles per GPU (weak), global batch (strong), noise sigma)
    "cfg4": ("base", "sr", 4, 256, 16, 128, 0.0),  # the configuration the metric is quoted on
    "cfg2": ("small", "sr", 4, 256, 16, 16, 0.0),
    "cfg3": ("base", "dn", 1, 256, 8, 8, 50.0),
    "cfg1": ("tiny", "sr", 2, 64, 1, 1, 0.0),
    "cfg5": ("base", "deblur", 1, 480, 0, 0, 0.0),  # one 1280x720 frame, tile 480 / overlap 48 -> 6 tiles
}
CFG5_FRAME, CFG5_TILE, CFG5_OVERLAP = (720, 1280), 480, 48
CPU_SAMPLE_TILE = 64  # cpu legs run ONE 64x64 tile of the same network per step (same per-pixel attention structure)
MICRO_BATCH = 16
DUMP_MAX_BYTES = 64 * 10**6  # --dump-outputs: all .npy files of one run together


def dump_outputs(dirname, arrays, max_bytes=DUMP_MAX_BYTES):
    """Writes each tensor of `arrays` as <dirname>/<name>.npy in float32.  A tensor larger than its share of max_bytes
    is replaced by a fixed sample of its elements: flat indices drawn from a generator seeded with 0 and sorted, so the
    sample is the same on every run and build and two builds can be compared element for element."""
    import numpy as np

    os.makedirs(dirname, exist_ok=True)
    cap = (max_bytes // len(arrays) - 4096) // 4  # elements per array, leaving room for the .npy header
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > cap:
            idx = torch.randint(t.numel(), (cap,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(tflops=d.get("bf16_tflops_sustained", 1447.6), hbm=d.get("hbm_gbs", 6574.8), src="measured")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.rows.append(l) for l in self.proc.stdout], daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.rows:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])), mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------------------------
# reference legs (test infrastructure: the only places bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------------------
def _oracle_modules():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import grl_oracle as orc
    from _pkgload import load_package

    return orc, load_package()


def _reference_forward(cfg, sd, device):
    """Returns (callable x -> y, kind).  kind "reference": the UNMODIFIED reference modules staged under oracle/_ref
    (oracle/make_ref.py) or found at /root/reference; "port": the restatement oracle/grl_oracle.py."""
    orc, _ = _oracle_modules()
    try:
        from _ref_import import import_reference, reference_available

        if reference_available():
            grl_mod = import_reference()[0]
            torch.manual_seed(0)
            m = grl_mod.GRL(**cfg).eval()
            missing, unexpected = m.load_state_dict(sd, strict=False)
            assert not unexpected
            m = m.to(device)

            def run(x):
                with torch.no_grad():
                    return m(x)

            return run, "reference"
    except Exception as e:  # noqa: BLE001 -- fall back to the port, and say so
        print(f"bench.py: reference import failed ({e!r}); using the oracle port", file=sys.stderr)

    sd_dev = {k: v.to(device) for k, v in sd.items()}

    def run_port(x):
        with torch.no_grad():
            return orc.grl_forward(sd_dev, cfg, x)

    return run_port, "port"


def cpu_leg(workload, steps, warmup):
    """The reference's own CPU implementation of the path (fp32, all useful host threads), one 64x64 tile of the
    workload's network per step -- a bounded sample: a 256x256 Base tile is ~2-3 minutes per forward on the CPU."""
    orc, pkg = _oracle_modules()
    variant, task, scale, tile, _, _, sigma = WORKLOADS[workload]
    size = {"sr": CPU_SAMPLE_TILE, "dn": 128, "deblur": 96}[task]  # one stripe of the task's released geometry
    cfg = pkg.configs.grl_config(variant, task, scale, size)
    sd = orc.synth_state_dict(cfg, seed=0, style="init")  # weights distributed like the reference constructor's
    x = orc.synth_input((1, 3, size, size), seed=1234, noise_sigma=sigma)
    # "all the host threads it can use": ATen's intra-op pool stops scaling (and then collapses) long before 128
    # threads on these small per-window ops, so pick the fastest of a few pool sizes on a 1-stage probe.
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    probe_cfg = dict(cfg, depths=cfg["depths"][:1], num_heads_window=cfg["num_heads_window"][:1],
                     num_heads_stripe=cfg["num_heads_stripe"][:1])
    probe_sd = orc.synth_state_dict(probe_cfg, seed=0, style="init")
    probe, _ = _reference_forward(probe_cfg, probe_sd, "cpu")
    best, cores = None, avail
    for n in sorted({min(avail, c) for c in (8, 16, 32, 64, avail)}):
        torch.set_num_threads(n)
        probe(x)
        t0 = time.perf_counter()
        probe(x)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, n
    torch.set_num_threads(cores)
    run, kind = _reference_forward(cfg, sd, "cpu")
    ts, y = [], None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        y = run(x)
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    sec = sum(ts) / len(ts)
    return dict(value=size * size / 1e6 / sec, sec_per_step=sec, cores=cores, kind=kind, size=size, y=y,
                sample=f"bounded sample: ONE {size}x{size} px tile of the {workload} network (GRL-{variant} {task} x{scale}, "
                       f"released hyper-parameters) per step, {steps} timed + {warmup} warm-up, fp32, {cores} threads")


def gpu_eager_leg(workload, dev):
    """SURVEY.md 2.2's bar: the reference run as eager PyTorch on this B200 (cuBLAS / cuDNN / ATen kernels), fp32,
    B = 1, one full-size tile of the workload."""
    orc, pkg = _oracle_modules()
    variant, task, scale, tile, _, _, sigma = WORKLOADS[workload]
    cfg = pkg.configs.grl_config(variant, task, scale, tile)
    sd = orc.synth_state_dict(cfg, seed=0, style="init")
    run, kind = _reference_forward(cfg, sd, dev)
    x = orc.synth_input((1, 3, tile, tile), seed=1234, noise_sigma=sigma).to(dev)
    run(x)
    torch.cuda.synchronize()
    ts = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(x)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = sorted(ts)[1]
    return dict(value=tile * tile / 1e6 / (ms / 1e3), unit="Mpix/s", ms_per_tile=ms, kind=kind, dtype="f32",
                sample=f"1 tile of {tile}x{tile} px, B=1, eager PyTorch on the GPU (median of 3)")


def native_parity(model, workload, dev):
    """Parity of the benchmarked build against the UNMODIFIED reference at the workload's native shape: the golden
    written by oracle/make_golden_native.py (reference fp32 CPU forward, same seeded weights / input)."""
    import numpy as np

    orc, _ = _oracle_modules()
    path = os.path.join(ROOT, "tests", "golden", f"native_{workload}_init.npz")
    if not os.path.exists(path):
        return None
    gold = np.load(path)
    variant, task, scale, tile, _, _, sigma = WORKLOADS[workload]
    x = orc.synth_input((1, 3, tile, tile), seed=1234, noise_sigma=sigma)
    y = model(x.to(dev)).float().cpu()
    s = int(gold["stride"])
    ref_sub = torch.from_numpy(gold["sub"])
    sub = y[..., ::s, ::s]
    gt = torch.rand(y.shape, generator=torch.Generator().manual_seed(9))
    b = scale if scale > 1 else 0
    return {"max_abs_vs_reference": (sub - ref_sub).abs().max().item(),
            "psnr_cand_vs_reference_db": (-10 * torch.log10(((sub - ref_sub) ** 2).mean())).item(),
            "delta_psnr_vs_gt_db": abs(orc.psnr(y, gt, b).mean().item() - float(gold["psnr_ref_gt"][0])),
            "sample": f"one {tile}x{tile} tile of {workload} (native shape), reference = unmodified models.networks.grl.GRL "
                      f"fp32 on the CPU (tests/golden/native_{workload}_init.npz; max-abs / PSNR(cand, ref) on its "
                      f"stride-{s} sub-sample, delta-PSNR over the full output)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--tiles-per-gpu", type=int, default=None)
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "fp16", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the bf16 pass, the eager-GPU baseline and the parity block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output of the last one as DIR/output.npy (float32; a fixed "
                         f"seeded sample of its elements when larger than {DUMP_MAX_BYTES // 10**6} MB; under torchrun "
                         "one DIR/output_rank<r>.npy per rank)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    variant, task, scale, tile, per_gpu, global_strong, sigma = WORKLOADS[a.workload]
    frame = a.workload == "cfg5"
    if a.tiles_per_gpu:
        per_gpu = a.tiles_per_gpu
    if frame:
        n_global, scaling = 1, "strong"
    elif a.scaling == "strong":
        n_global, scaling = max(global_strong, world), "strong"
    else:
        n_global, scaling = per_gpu * world, "weak"
    W = max(a.warmup, 3)
    metric = "Mpix/s (input pixels) GRL-Base x4 SR 256x256 tiles" if a.workload == "cfg4" else f"Mpix/s {a.workload}"
    if frame:
        wl = (f"cfg5: GRL-{variant} {task}, one {CFG5_FRAME[1]}x{CFG5_FRAME[0]} synthetic frame per step, tiled inference "
              f"tile {CFG5_TILE} / overlap {CFG5_OVERLAP} (6 tiles of 480x480), tiles round-robin over the ranks, released "
              f"hyper-parameters")
    else:
        wl = f"{a.workload}: GRL-{variant} {task} x{scale}, {tile}x{tile} synthetic tiles, released hyper-parameters"
    cfg_desc = dict(workload=wl, global_batch=n_global, tile=tile,
                    parallelism=f"{'tile' if frame else 'batch'}-sharded dp{world}, weights replicated",
                    l2="per-step working set (GBs of activations) >> 126 MB L2; no explicit flush needed")
    if not frame:
        cfg_desc["tiles_per_gpu"] = n_global // world if scaling == "strong" else per_gpu

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if a.impl == "reference":
        if rank != 0:
            return
        r = cpu_leg(a.workload, a.steps, max(a.warmup, 0))
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, {"output": r["y"]})
        cfg_ref = dict(cfg_desc)
        cfg_ref["workload"] = wl + f" -- CPU arm measured on a {r['sample']}"
        emit({
            "impl": "reference", "metric": metric, "value": r["value"], "unit": "Mpix/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": max(a.warmup, 0), "ms_per_step": r["sec_per_step"] * 1e3, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg_ref,
            "cpu_baseline": {"value": r["value"], "unit": "Mpix/s", "cores": r["cores"], "kind": r["kind"],
                             "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        })
        return

    # ------------------------------------------------------------------ our arm
    import torch.distributed as dist
    from _pkgload import load_package

    pkg = load_package()
    from grl_image_restoration_b200 import capi, flops, functional as K, metrics, sharding, tiling

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import grl_oracle as orc  # synthetic weights/inputs shared with the checker; not on the timed path

    cfg = pkg.configs.grl_config(variant, task, scale, tile)
    model = pkg.GRL(**cfg)
    model.load_state_dict(orc.synth_state_dict(cfg, seed=0, style="init"), strict=False)
    model = model.to(dev).eval()
    precision = model.set_precision(a.precision)
    g = torch.Generator().manual_seed(1234 + (0 if frame else rank))
    if frame:
        lo, hi = 0, 1
        x_host = torch.rand(1, 3, *CFG5_FRAME, generator=g).pin_memory()
        gt_host = torch.rand(1, 3, *CFG5_FRAME, generator=g).pin_memory()
        mpix_step = CFG5_FRAME[0] * CFG5_FRAME[1] / 1e6
    else:
        lo, hi = sharding.shard_range(n_global, rank, world)
        x_host = torch.rand(hi - lo, 3, tile, tile, generator=g)
        if sigma > 0:
            x_host = x_host + (sigma / 255.0) * torch.randn(x_host.shape, generator=g)
        x_host = x_host.pin_memory()
        gt_host = torch.rand(hi - lo, 3, tile * scale, tile * scale, generator=g).pin_memory()
        mpix_step = n_global * tile * tile / 1e6
    x_dev = x_host.to(dev)
    idx = torch.arange(lo, hi, device=dev)

    def forward(xd):
        if frame:
            return tiling.forward_tile_sharded(model, xd, CFG5_TILE, CFG5_OVERLAP, max_batch=MICRO_BATCH)
        if xd.shape[0] <= MICRO_BATCH:
            return model(xd)
        return torch.cat([model(xd[i:i + MICRO_BATCH]) for i in range(0, xd.shape[0], MICRO_BATCH)])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), out

    # ---- device-resident throughput (headline): no event records, no host work inside the timed loop
    for _ in range(W):
        y = forward(x_dev)
    barrier()
    launches0 = capi.lib().grl_launch_count()
    vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    smi_index = vis.split(",")[local_rank] if vis and all(v.strip().isdigit() for v in vis.split(",")) else local_rank
    sampler = ClockSampler(smi_index)
    sampler.start()
    ms_total, y = timed(lambda: forward(x_dev), a.steps)
    clocks = sampler.stop()
    launches = capi.lib().grl_launch_count() - launches0
    ms_step = ms_total / a.steps
    value = mpix_step / (ms_step / 1e3)
    if a.dump_outputs:  # this rank's share of the batch (cfg5: the whole frame, identical on every rank)
        dump_outputs(a.dump_outputs, {"output" if world == 1 else f"output_rank{rank}": y},
                     DUMP_MAX_BYTES // world)

    # ---- end to end through the public API with host buffers (+ the final metric all-gather)
    def e2e_step():
        xd = x_host.to(dev, non_blocking=True)
        gd = gt_host.to(dev, non_blocking=True)
        out = forward(xd)
        p, _ = metrics.psnr_fused(out, gd, border=scale if scale > 1 else 0)  # one fused kernel (csrc/metric.cu)
        if frame:
            return p.cpu(), idx.cpu()
        gv, gi = sharding.gather_metric(p, idx)
        return gv.cpu(), gi.cpu()

    e2e_step()
    ms_e2e, (pv, pi) = timed(e2e_step, a.steps)
    e2e_value = mpix_step / (ms_e2e / a.steps / 1e3)
    mean_psnr = sharding.average_metric(pv, pi)

    # ---- roofline pass (separate from the headline): CUDA events around every attention launch
    K.timer = K.KernelTimer()
    roof_steps = max(1, min(a.steps, 3))
    ms_roof, _ = timed(lambda: forward(x_dev), roof_steps)
    attn_ms = K.timer.totals_ms()
    K.timer = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    feat = tuple((s + model.pad_size - 1) // model.pad_size * model.pad_size for s in ((CFG5_TILE, CFG5_TILE) if frame else (tile, tile)))
    counts = flops.attention_counts(cfg, feat)
    attn_total_ms = sum(v[0] for v in attn_ms.values())
    attn_launches = sum(v[1] for v in attn_ms.values())
    imgs_this_rank = len(tiling.shard_tiles(6, rank, world)) if frame else (hi - lo)
    flops_timed = counts["f_attn"] * imgs_this_rank * roof_steps
    achieved = flops_timed / (attn_total_ms / 1e3) / 1e12 if attn_total_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if precision != "fp32" and a.workload == "cfg4" and os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj["attention_dram_bytes_per_image_per_block"] * (hi - lo) / tj["launches_per_block"]
    mufu_peak_tf = None
    if clocks.get("sm_mhz"):
        # exp2 co-bound: 16 MUFU ops / clk / SM x 148 SMs at the clock seen during the run; one exp2 per score element
        mufu_peak_tf = 16 * 148 * clocks["sm_mhz"] * 1e6 * (counts["f_attn"] / counts["score_elems"]) / 1e12
    roof = {"bound": "tensor", "kernel": "fused window + anchored-stripe attention (QK^T + PV), all launches",
            "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"],
            "peak_source": f"bf16 sustained, {pk['src']}", "traffic": traffic,
            "traffic_note": "average DRAM bytes per attention launch from profiles/traffic.json (one ncu --set full capture)",
            "co_bound": "softmax exp2: one MUFU op per score element (4 x head_dim MMA FLOP); 16 MUFU/clk/SM",
            "mufu_bound_tflops": mufu_peak_tf, "frac_of_mufu_bound": (achieved / mufu_peak_tf) if mufu_peak_tf else None,
            "share_of_step": attn_total_ms / ms_roof, "launches_timed": attn_launches,
            "avg_launch_ms": attn_total_ms / max(attn_launches, 1),
            "timed_in": f"separate pass of {roof_steps} step(s) after the headline loop",
            "algorithmic_gflop_per_image": counts["f_attn"] / 1e9, "qk_frac": achieved / 2 / pk["tflops"]}

    out = {"metric": metric, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": a.steps, "warmup": W,
           "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
           "dtype": {"fp32": "f32", "fp16": "f16", "bf16": "bf16"}[precision],
           "dtype_note": "MMA operand format (tcgen05 kind::f16, fp32 accumulate); residual stream, LayerNorm, softmax "
                         "statistics in fp32. f16 (11-bit mantissa) >= bf16 precision; the bf16-operand pass is under extra",
           "data": "synthetic", "config": cfg_desc,
           "output_mpix_per_s": value * scale * scale, "clocks": clocks, "gpu_launches": int(launches),
           "e2e": {"value": e2e_value, "unit": "Mpix/s", "h2d_bytes_per_step": int(x_host.numel() * 4 + gt_host.numel() * 4),
                   "d2h_bytes_per_step": int(pv.numel() * 4 + pi.numel() * 8),
                   "includes": "H2D inputs+GT from pinned memory, forward, fused PSNR kernel (RGB + luma) on device, all-gather, D2H"},
           "mean_psnr_vs_random_gt_db": mean_psnr, "roofline": roof}

    if world == 1 and not a.no_extras:
        extra = {}
        # second operand format on the same build (BASELINE's configs say bf16; fp16 is what meets its PSNR gate)
        other = "bf16" if precision == "fp16" else "fp16"
        try:
            model.set_precision(other)
            for _ in range(2):
                forward(x_dev)
            ms_o, _ = timed(lambda: forward(x_dev), max(1, min(a.steps, 3)))
            extra[f"{other}_operands"] = {"value": mpix_step / (ms_o / max(1, min(a.steps, 3)) / 1e3), "unit": "Mpix/s",
                                          "parity": native_parity(model, a.workload, dev) if not frame else None}
        except RuntimeError as e:
            extra[f"{other}_operands"] = {"error": str(e)}
        model.set_precision(precision)
        if not frame:
            out["parity"] = native_parity(model, a.workload, dev)
            try:
                extra["gpu_eager_baseline"] = gpu_eager_leg(a.workload, dev)
            except Exception as e:  # noqa: BLE001
                extra["gpu_eager_baseline"] = {"error": repr(e)}
        out["extra"] = extra
    # ---- CPU baseline (rank 0, N=1 only)
    if world == 1 and not a.no_cpu_baseline:
        r = cpu_leg(a.workload, 2, 1)
        out["cpu_baseline"] = {"value": r["value"], "unit": "Mpix/s", "cores": r["cores"], "kind": r["kind"],
                               "sample": r["sample"]}
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
