"""Dev tool: time the transformer MLP of one GRL block on cuda:0 (CUDA events).

  (a) the two-launch route through grl_tc_gemm: fc1 + GELU -> 16-bit hidden in HBM, then fc2 + LayerNorm2 + residual;
  (b) the fused launch through grl_tc_mlp (tc.mlp): the hidden activation stays on the SM.

Shapes are one block of the benchmark configurations (B tiles of 256^2 tokens).  Achieved bandwidth is quoted against
the algorithmic bytes of the fused operation, M * (2 cpad + 4 C + 4 C + 2 cpad): 16-bit input, fp32 residual, fp32 and
16-bit outputs.  Every working set is larger than the 126 MB L2."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from _pkgload import load_package  # noqa: E402

SHAPES = {  # name: (tiles, C, mlp_ratio)
    "cfg4": (16, 180, 2),
    "cfg2": (16, 128, 2),
    "cfg3": (8, 180, 2),
}
PEAK_BW = 6.57e12  # bytes/s, the copy bandwidth measured on this card type (DESIGN.md)

ap = argparse.ArgumentParser()
ap.add_argument("--shapes", default="cfg4,cfg2,cfg3")
ap.add_argument("--parts", default="a,b", help="a = fc1 + fc2 through grl_tc_gemm, b = the fused grl_tc_mlp launch")
ap.add_argument("--iters", type=int, default=50)
ap.add_argument("--warmup", type=int, default=5)
ap.add_argument("--fmt", type=int, default=0, help="0 = fp16 operands, 1 = bf16")
a = ap.parse_args()
load_package()
from grl_image_restoration_b200 import tc as T  # noqa: E402

try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except (OSError, IndexError, subprocess.SubprocessError):
    smi = "nvidia-smi unavailable"
print(f"device: {torch.cuda.get_device_name(0)} | {smi}")


def timed(fn):
    for _ in range(a.warmup):
        fn()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(a.iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / a.iters


dev = "cuda"
for name in a.shapes.split(","):
    tiles, C, ratio = SHAPES[name]
    M = tiles * 256 * 256
    hid = ratio * C
    cpad, hpad = T.round_up(C, 64), T.round_up(hid, 64)
    n_ln = 64 if C <= 64 else 128 if C <= 128 else 192
    g = torch.Generator(device=dev).manual_seed(0)
    dt = T.DTYPE[a.fmt]
    y16 = torch.zeros(M, cpad, device=dev, dtype=dt)
    y16[:, :C] = torch.randn(M, C, device=dev, generator=g).to(dt)
    x32 = torch.randn(M, C, device=dev, generator=g)
    w1 = T._pad_matrix(torch.randn(hid, C, device=dev, generator=g) * C ** -0.5, hpad, cpad, fmt=a.fmt)
    b1 = T._pad_vector(torch.randn(hid, device=dev, generator=g), hpad)
    w2 = T._pad_matrix(torch.randn(C, hid, device=dev, generator=g) * hid ** -0.5, n_ln, hpad, fmt=a.fmt)
    b2 = T._pad_vector(torch.randn(C, device=dev, generator=g), n_ln)
    gamma, beta = torch.randn(C, device=dev, generator=g) + 1.0, torch.randn(C, device=dev, generator=g)
    z32 = torch.empty(M, C, device=dev)
    z16 = torch.empty(M, cpad, device=dev, dtype=dt)
    nbytes = M * (2 * cpad + 4 * C + 4 * C + 2 * cpad)

    def report(label, ms):
        print(f"{name} M={M} C={C} hidden={hid} {label}: {ms:.3f} ms/launch, {nbytes / ms / 1e6:.0f} GB/s "
              f"({nbytes / ms / 1e-3 / PEAK_BW * 100:.1f}% of {PEAK_BW / 1e12:.2f} TB/s)")

    if "a" in a.parts:
        h16 = torch.empty(M, hpad, device=dev, dtype=dt)

        def fc1():
            T.gemm(y16, w1, b1, M=M, kpad=cpad, npad=hpad, epi=T.EPI_BIAS_ACT, n_store=hpad, act=T.K.ACT_GELU, out_bf16=h16)

        def fc2():
            T.gemm(h16, w2, b2, M=M, kpad=hpad, npad=n_ln, epi=T.EPI_LN, n_store=n_ln, n_real=C, out_bf16=z16,
                   out_f32=z32, res_f32=x32, C=C, gamma=gamma, beta=beta, eps=1e-5, res_scale=1.0, L=65536)

        t1, t2 = timed(fc1), timed(fc2)
        t12 = timed(lambda: (fc1(), fc2()))
        print(f"{name} (a) fc1+GELU {t1:.3f} ms, fc2+LN2 {t2:.3f} ms")
        report("(a) fc1 + fc2", t12)
        ref32, ref16 = z32.clone(), z16.clone()
        del h16
    if "b" in a.parts:
        def fused():
            T.mlp(y16, w1, b1, w2, b2, M=M, C=C, out_f32=z32, out_bf16=z16, res_f32=x32, gamma=gamma, beta=beta, eps=1e-5,
                  res_scale=1.0)

        report("(b) fused", timed(fused))
        if "a" in a.parts:
            print(f"{name} max |(b) - (a)|: z32 {(z32 - ref32).abs().max().item():.3e}, "
                  f"z16 {(z16.float() - ref16.float()).abs().max().item():.3e}")
    del y16, x32, z32, z16
    torch.cuda.empty_cache()
