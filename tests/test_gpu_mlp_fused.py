"""Fused transformer MLP (grl_tc_mlp: fc1 -> GELU -> fc2 -> LayerNorm2 + residual in one launch) against an fp32 reference
on 16-bit-rounded operands, and against the two-launch route it replaces (grl_tc_gemm fc1 with the GELU epilogue, then
fc2 with the LayerNorm epilogue), which computes the same arithmetic and must agree bit for bit."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def r16(t, fmt):
    return t.to(torch.bfloat16 if fmt else torch.float16).float()


@pytest.fixture(scope="module")
def T(pkg, device):
    from grl_image_restoration_b200 import capi, tc

    if capi.lib().grl_device_ok() != 1:
        pytest.skip("tcgen05 path needs sm_100")
    return tc


def _problem(T, device, M, C, hid, fmt, seed=0):
    cpad, hpad = T.round_up(C, 64), T.round_up(hid, 64)
    n_ln = 64 if C <= 64 else 128 if C <= 128 else 192
    x = rnd((M, C), seed + 1)
    w1, b1 = rnd((hid, C), seed + 2, C ** -0.5), rnd((hid,), seed + 3)
    w2, b2 = rnd((C, hid), seed + 4, hid ** -0.5), rnd((C,), seed + 5)
    res, g, be = rnd((M, C), seed + 6), rnd((C,), seed + 7) + 1.0, rnd((C,), seed + 8)
    dev = dict(x16=T.pack_rows(x.to(device), cpad, fmt), w1=T._pad_matrix(w1.to(device), hpad, cpad, fmt=fmt),
               b1=T._pad_vector(b1.to(device), hpad), w2=T._pad_matrix(w2.to(device), n_ln, hpad, fmt=fmt),
               b2=T._pad_vector(b2.to(device), n_ln), res=res.to(device), g=g.to(device), be=be.to(device))
    host = dict(x=x, w1=w1, b1=b1, w2=w2, b2=b2, res=res, g=g, be=be)
    return dev, host, cpad, hpad, n_ln


def _fused(T, d, M, C, cpad, fmt, res_scale):
    z32 = torch.empty(M, C, device=d["res"].device)
    z16 = torch.full((M, cpad), 7.0, device=d["res"].device, dtype=T.DTYPE[fmt])  # the pad must be overwritten with zeros
    T.mlp(d["x16"], d["w1"], d["b1"], d["w2"], d["b2"], M=M, C=C, out_f32=z32, out_bf16=z16, res_f32=d["res"], gamma=d["g"],
          beta=d["be"], eps=1e-5, res_scale=res_scale)
    return z32, z16


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("M", [515, 100])
@pytest.mark.parametrize("ratio", [2, 4])
@pytest.mark.parametrize("C", [36, 64, 128, 180])
def test_mlp_fused_vs_reference(T, device, C, ratio, M, fmt):
    d, h, cpad, hpad, n_ln = _problem(T, device, M, C, ratio * C, fmt)
    hidden = r16(F.gelu(F.linear(r16(h["x"], fmt), r16(h["w1"], fmt), h["b1"])), fmt)
    ref = h["res"] + 0.5 * F.layer_norm(F.linear(hidden, r16(h["w2"], fmt), h["b2"]), (C,), h["g"], h["be"], 1e-5)
    z32, z16 = _fused(T, d, M, C, cpad, fmt, 0.5)
    # the hidden is rounded to 16 bits on both sides from GELUs that differ by ~1e-6: a value may round one step apart
    tol = 5e-3 if fmt == 0 else 2e-2
    assert (z32.cpu() - ref).abs().max().item() <= tol
    assert (z16.cpu().float()[:, :C] - ref).abs().max().item() <= 10 * tol
    if cpad > C:
        assert z16.cpu().float()[:, C:].abs().max().item() == 0


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("M", [2 * 256 * 256, 2 * 256 * 256 - 37])
def test_mlp_fused_equals_two_launches(T, device, M, fmt):
    """cfg4 block shape (GRL-Base, C = 180, mlp_ratio 2, two 256^2 tiles) and a ragged row count: same gelu_as, same
    16-bit rounding of the hidden, same K order of every fp32 accumulation, same LayerNorm epilogue -> identical bits."""
    C, hid = 180, 360
    d, _, cpad, hpad, n_ln = _problem(T, device, M, C, hid, fmt, seed=40)
    rs = 0.75
    hid16 = torch.empty(M, hpad, device=device, dtype=T.DTYPE[fmt])
    T.gemm(d["x16"], d["w1"], d["b1"], M=M, kpad=cpad, npad=hpad, epi=T.EPI_BIAS_ACT, n_store=hpad, act=T.K.ACT_GELU,
           out_bf16=hid16)
    a32 = torch.empty(M, C, device=device)
    a16 = torch.empty(M, cpad, device=device, dtype=T.DTYPE[fmt])
    T.gemm(hid16, d["w2"], d["b2"], M=M, kpad=hpad, npad=n_ln, epi=T.EPI_LN, n_store=n_ln, n_real=C, out_bf16=a16,
           out_f32=a32, res_f32=d["res"], C=C, gamma=d["g"], beta=d["be"], eps=1e-5, res_scale=rs, L=M)
    z32, z16 = _fused(T, d, M, C, cpad, fmt, rs)
    assert torch.equal(z32, a32), (z32 - a32).abs().max().item()
    assert torch.equal(z16, a16)


def test_mlp_rejects_unsupported_shapes(T, device):
    d, _, cpad, hpad, n_ln = _problem(T, device, 64, 36, 72, 0)
    z32 = torch.empty(64, 36, device=device)
    z16 = torch.empty(64, cpad, device=device, dtype=torch.float16)
    with pytest.raises(RuntimeError, match="tc_mlp"):  # C % 4 != 0
        T.mlp(d["x16"], d["w1"], d["b1"], d["w2"], d["b2"], M=64, C=34, out_f32=z32, out_bf16=z16, res_f32=d["res"],
              gamma=d["g"], beta=d["be"])
    with pytest.raises(RuntimeError, match="tc_mlp"):  # hidden pad not a multiple of 64
        T.mlp(d["x16"], d["w1"][:96], d["b1"], d["w2"][:, :96].contiguous(), d["b2"], M=64, C=36, out_f32=z32, out_bf16=z16,
              res_f32=d["res"], gamma=d["g"], beta=d["be"])
