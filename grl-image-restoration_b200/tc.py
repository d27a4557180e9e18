"""bf16 tensor-core execution of a GRL block / stage / network (the throughput path).

Host-side orchestration only: one-time weight packing (pad head_dim to 32-wide slots, pad channel pitches to
multiples of 64, permute the QKV rows into [window q|k|v][stripe q|k|v] x head order, im2col-order the 3x3 kernels)
and the launch sequence of the tcgen05 kernels behind the C ABI (grl_tc_gemm / grl_tc_mlp / grl_tc_attn, include/grl_b200.h).
Numerics contract (DESIGN.md): bf16 only for MMA operands; residual stream, LayerNorm, L2-normalisation, softmax
statistics and every accumulator are fp32.
Reference semantics: mixed_attn_block_efficient.py:351-381,:539-556; mixed_attn_block.py:948-983; grl.py:164-170,:506-551.
"""
import ctypes

import torch

from . import capi
from . import functional as K
from . import geometry as G

LOG2E = 1.4426950408889634
EPI_BIAS_ACT, EPI_QKV, EPI_LN = 0, 1, 2
SLOT = 32
FMT = {"fp16": 0, "bf16": 1}
DTYPE = {0: torch.float16, 1: torch.bfloat16}


def fmt_of(t):
    return 1 if t.dtype == torch.bfloat16 else 0


def round_up(a, b):
    return (a + b - 1) // b * b


LN_MAX_C = 188  # the LayerNorm epilogue keeps a whole 128 x C fp32 row tile in the GEMM's staging area (gemm_tc.cu)


def supported(C, heads_w, heads_s):
    """Architectures the tensor-core path covers: head_dim <= 32 (one 32-wide slot per head), <= 8 heads per
    attention, C % 4 == 0 and C <= LN_MAX_C (launch_gemm_tc's LayerNorm-epilogue limit).  Anything else runs on the
    fp32 kernels ("auto") or is rejected up front (explicit "fp16" / "bf16")."""
    c = C // 2
    return (C % 4 == 0 and C <= LN_MAX_C and c % heads_w == 0 and c % heads_s == 0 and c // heads_w <= SLOT
            and c // heads_s <= SLOT and heads_w <= 8 and heads_s <= 8)


def _h16(*shape, device, fmt, zero=False):
    return (torch.zeros if zero else torch.empty)(*shape, device=device, dtype=DTYPE[fmt])


def head_pack(x, hp, wp, mean, img_range, cpad=64, fmt=0, want_f32=False):
    """Network input (B, Cin, H, W) fp32 -> 16-bit channels-last (B, hp, wp, cpad) [+ fp32 (B, hp, wp, Cin)]: reflect pad,
    (x - mean) * img_range, layout change and operand pack in one kernel (grl_tc_head_pack)."""
    B, Cin, H, W = x.shape
    y16 = _h16(B, hp, wp, cpad, device=x.device, fmt=fmt)
    y32 = torch.empty(B, hp, wp, Cin, device=x.device, dtype=torch.float32) if want_f32 else None
    m = [float(v) for v in (mean if isinstance(mean, (list, tuple)) else mean.flatten().tolist())]
    m = (m * 4)[:4] if len(m) == 1 else (m + [0.0] * 4)[:4]
    arr = (ctypes.c_float * 4)(*m)
    capi.check(capi.lib().grl_tc_head_pack(capi.ptr(x), B, Cin, H, W, hp, wp, arr, float(img_range), capi.ptr(y16), cpad,
                                           capi.ptr(y32), fmt, capi.stream()))
    return y16, y32


def pack_rows(x, cpad, fmt=0):
    """fp32 (..., C) contiguous -> 16-bit (..., cpad), zero padded."""
    C = x.shape[-1]
    M = x.numel() // C
    y = _h16(*x.shape[:-1], cpad, device=x.device, fmt=fmt)
    capi.check(capi.lib().grl_tc_pack16(capi.ptr(x), C, capi.ptr(y), M, C, cpad, fmt, capi.stream()))
    return y


def unpack_rows(x16, C, off=0):
    """16-bit (..., ld) -> fp32 (..., C) taking columns [off, off + C)."""
    ld = x16.shape[-1]
    M = x16.numel() // ld
    y = torch.empty(*x16.shape[:-1], C, device=x16.device, dtype=torch.float32)
    capi.check(capi.lib().grl_tc_unpack16(capi.ptr(x16), ld, off, capi.ptr(y), C, M, C, fmt_of(x16), capi.stream()))
    return y


def _pad_matrix(w, npad, kpad, row_map=None, col_map=None, fmt=0):
    """Scatter fp32 (N, K) into 16-bit (npad, kpad): dest row row_map[i] <- src row i, dest col col_map[j] <- src col j."""
    N, Kd = w.shape
    out = torch.zeros(npad, kpad, device=w.device, dtype=torch.float32)
    r = torch.arange(N, device=w.device) if row_map is None else torch.as_tensor(row_map, device=w.device)
    c = torch.arange(Kd, device=w.device) if col_map is None else torch.as_tensor(col_map, device=w.device)
    out[r[:, None], c[None, :]] = w.detach().float()
    return out.to(DTYPE[fmt]).contiguous()


def _pad_vector(b, npad, row_map=None):
    out = torch.zeros(npad, device=b.device, dtype=torch.float32)
    if b is not None:
        r = torch.arange(b.numel(), device=b.device) if row_map is None else torch.as_tensor(row_map, device=b.device)
        out[r] = b.detach().float()
    return out


def pack_conv(conv, cin_pad, npad, fmt=0, ps_r=0):
    """nn.Conv2d(3x3) weight (Cout, Cin, 3, 3) -> 16-bit (npad, 9*cin_pad), k = (ky*3+kx)*cin_pad + c; bias fp32 (npad).
    ps_r > 0: the conv feeds nn.PixelShuffle(ps_r): output channel c*r^2 + q (torch order) is stored at row q*(Cout/r^2) + c,
    so the channels of one shuffled pixel are consecutive output columns (grl_tc_gemm's ps_r store)."""
    w = conv.weight.detach().float()
    co, ci = w.shape[:2]
    rows = torch.arange(co, device=w.device)
    if ps_r > 0:
        cq = co // (ps_r * ps_r)
        rows = (rows % (ps_r * ps_r)) * cq + rows // (ps_r * ps_r)
    out = torch.zeros(npad, 9, cin_pad, device=w.device, dtype=torch.float32)
    out[rows, :, :ci] = w.permute(0, 2, 3, 1).reshape(co, 9, ci)
    bias = torch.zeros(npad, device=w.device, dtype=torch.float32)
    if conv.bias is not None:
        bias[rows] = conv.bias.detach().float()
    return out.reshape(npad, 9 * cin_pad).to(DTYPE[fmt]).contiguous(), bias


def gemm(x16, w16, bias, *, M=0, image=None, kpad, npad, taps=1, epi=EPI_BIAS_ACT, n_store=0, n_real=0, out_bf16=None,
         out_f32=None, res_f32=None, act=K.ACT_NONE, slope=0.0, slot_scale=None, C=0, gamma=None, beta=None, eps=1e-5,
         res_scale=1.0, cab_y=None, cab_gate=None, L=1, ps_r=0, out_nchw=None, nchw_r=1, post_scale=1.0, post_shift=None):
    p = capi.GrlTcGemm()
    if x16.dtype != w16.dtype:
        raise RuntimeError("grl_b200: activation / weight operand formats differ")
    p.fmt = fmt_of(x16)
    p.x, p.w, p.bias = x16.data_ptr(), w16.data_ptr(), bias.data_ptr()
    p.M = M
    if image is not None:
        p.B, p.H, p.W = image
    p.kpad, p.npad, p.taps, p.epi = kpad, npad, taps, epi
    p.n_store, p.n_real = n_store, n_real
    if out_bf16 is not None:
        p.out_bf16, p.ldo_bf16 = out_bf16.data_ptr(), out_bf16.shape[-1]
    if out_f32 is not None:
        p.out_f32, p.ldo_f32 = out_f32.data_ptr(), out_f32.shape[-1]
    if res_f32 is not None:
        p.res_f32, p.ldr = res_f32.data_ptr(), res_f32.shape[-1]
    p.act, p.slope = act, slope
    if slot_scale is not None:
        p.slot_scale = slot_scale.data_ptr()
    p.C = C
    if gamma is not None:
        p.gamma, p.beta = gamma.data_ptr(), beta.data_ptr()
    p.eps, p.res_scale = eps, res_scale
    if cab_y is not None:
        p.cab_y, p.ld_caby, p.cab_gate = cab_y.data_ptr(), cab_y.shape[-1], cab_gate.data_ptr()
    p.L = L
    p.ps_r = ps_r
    if out_nchw is not None:  # (B, C_out, Hc, Wc) fp32 planes: denormalise + crop + bhwc -> bchw folded into the store
        p.out_nchw, p.nchw_r, p.Hc, p.Wc = out_nchw.data_ptr(), nchw_r, out_nchw.shape[2], out_nchw.shape[3]
        p.post_scale = post_scale
        for i in range(4):
            p.post_shift[i] = float(post_shift[i]) if post_shift is not None and i < len(post_shift) else 0.0
    capi.check(capi.lib().grl_tc_gemm(ctypes.byref(p), capi.stream()))


def mlp(x16, w1, b1, w2, b2, *, M, C, out_f32, out_bf16, res_f32, gamma, beta, eps=1e-5, res_scale=1.0):
    """out = res + res_scale * LayerNorm(fc2(GELU(fc1(x)))) in one launch (grl_tc_mlp): x16 (M, cpad), w1 (hpad, cpad),
    w2 (n_ln, hpad) as packed by BlockPlan; out_f32 (M, C) fp32 and out_bf16 (M, ldo) 16-bit, zero beyond C."""
    if not (x16.dtype == w1.dtype == w2.dtype == out_bf16.dtype):
        raise RuntimeError("grl_b200: activation / weight operand formats differ")
    if w1.shape[1] != x16.shape[-1] or w2.shape[1] != w1.shape[0]:
        raise RuntimeError("grl_b200: MLP weight shapes do not chain")
    p = capi.GrlTcMlp()
    p.fmt = fmt_of(x16)
    p.x, p.w1, p.b1, p.w2, p.b2 = x16.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr()
    p.M, p.C, p.cpad, p.hpad, p.n_ln = M, C, x16.shape[-1], w1.shape[0], w2.shape[0]
    p.gamma, p.beta, p.eps, p.res_scale = gamma.data_ptr(), beta.data_ptr(), eps, res_scale
    p.res_f32, p.ldr = res_f32.data_ptr(), res_f32.shape[-1]
    p.out_f32, p.ldo_f32 = out_f32.data_ptr(), out_f32.shape[-1]
    p.out_bf16, p.ldo_bf16 = out_bf16.data_ptr(), out_bf16.shape[-1]
    capi.check(capi.lib().grl_tc_mlp(ctypes.byref(p), capi.stream()))


def attention(gq, gk, q, q_off, k, k_off, v, v_off, out, o_off, B, heads, bias, use_mask, v_dense=False,
              o_dense=False, tag="attn", ones_col=False):
    p = capi.GrlTcAttn()
    p.fmt = fmt_of(q)
    p.gq, p.gk = gq, gk
    p.q, p.ldq, p.q_off = q.data_ptr(), q.shape[-1], q_off
    p.k, p.ldk, p.k_off = k.data_ptr(), k.shape[-1], k_off
    p.v, p.ldv, p.v_off, p.v_dense = v.data_ptr(), v.shape[-1], v_off, int(v_dense)
    p.out, p.ldo, p.o_off, p.o_dense = out.data_ptr(), out.shape[-1], o_off, int(o_dense)
    if bias.dim() != 3 or bias.shape[1] != 4:
        raise RuntimeError("grl_b200: attention bias must be the (heads, 4, rows_pad) table of bias_table_log2 / shifted_copies")
    p.B, p.heads, p.bias, p.use_mask = B, heads, bias.data_ptr(), int(use_mask)
    p.rows, p.rows_pad = (gq.wh + gk.wh - 1) * (gq.ww + gk.ww - 1), bias.shape[2]
    p.ones_col = int(ones_col)
    K._timed(tag, lambda: capi.check(capi.lib().grl_tc_attn(ctypes.byref(p), capi.stream())))


def bias_rows_pad(rows):
    return round_up(rows + 16, 4)  # slack for the aligned over-reads of the shifted copies (16: staged rows, variant 4)


def shifted_copies(table_hr):
    """(heads, rows) fp32 -> (heads, 4, rows_pad): copy c shifted right by c entries (layout grl_tc_attn reads)."""
    heads, rows = table_hr.shape
    out = torch.zeros(heads, 4, bias_rows_pad(rows), device=table_hr.device, dtype=torch.float32)
    for c in range(4):
        out[:, c, c:c + rows] = table_hr
    return out


def bias_table_log2(transform, table):
    """16*sigmoid(cpb_mlp(table))*log2(e) as the 4-copy table of the attention kernel."""
    t = table.reshape(-1, 2)
    w1, b1, w2 = transform.cpb_mlp[0].weight, transform.cpb_mlp[0].bias, transform.cpb_mlp[2].weight
    heads, hidden = w2.shape
    rows_pad = bias_rows_pad(t.shape[0])
    out = torch.zeros(heads, 4, rows_pad, device=t.device, dtype=torch.float32)
    capi.check(capi.lib().grl_tc_bias_table4(capi.ptr(t), t.shape[0], capi.ptr(w1), capi.ptr(b1), capi.ptr(w2), hidden,
                                             heads, LOG2E, rows_pad, capi.ptr(out), capi.stream()))
    return out


def conv3x3(x16, wpack, bias, cin_pad, npad, *, n_store, n_real=0, act=K.ACT_NONE, slope=0.0, out_bf16=None,
            out_f32=None, res_f32=None, **tail):
    """x16 bf16 (B, H, W, cin_pad) channels-last.  tail: ps_r / out_nchw / nchw_r / post_scale / post_shift (head-tail fusion)."""
    B, H, W, _ = x16.shape
    gemm(x16, wpack, bias, image=(B, H, W), kpad=cin_pad, npad=npad, taps=9, epi=EPI_BIAS_ACT, n_store=n_store,
         n_real=n_real, out_bf16=out_bf16, out_f32=out_f32, res_f32=res_f32, act=act, slope=slope, **tail)


def _version_key(module):
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


class BlockPlan:
    """Packed weights + launch sequence of one EfficientMixAttnTransformerBlock."""

    def __init__(self, blk, fmt):
        self.key = (_version_key(blk), fmt)
        self.fmt = fmt
        self._const_key, self._consts = None, None
        at = blk.attn
        C = blk.dim
        c = C // 2
        hw, hs = at.window_attn.num_heads, at.stripe_attn.num_heads
        dw, ds = c // hw, c // hs
        self.C, self.cpad, self.hw, self.hs = C, round_up(C, 64), hw, hs
        self.nslots = 3 * hw + 3 * hs
        # --- QKV: dest row = slot*32 + e
        rmap = []
        for half, (h, d) in enumerate(((hw, dw), (hs, ds))):
            slot_base = 0 if half == 0 else 3 * hw
            for t in range(3):
                for head in range(h):
                    for e in range(d):
                        rmap.append((slot_base + t * h + head) * SLOT + e)
        # source rows are already ordered (half, t, head, e) in the reference layout (efficient.py:150,:251,:362)
        self.n_qkv = self.nslots * SLOT
        self.w_qkv = _pad_matrix(at.qkv.body.weight, self.n_qkv, self.cpad, row_map=rmap, fmt=fmt)
        self.b_qkv = _pad_vector(at.qkv.body.bias if at.qkv.body.bias is not None else torch.zeros(3 * C, device=at.qkv.body.weight.device), self.n_qkv, rmap)
        # ones-column (attn_tc.cu): with head_dim < 32 the last slot column of every VALUE slot is 1 (set through the
        # bias; its weight row is zero), so the P V MMA also produces the softmax denominator.  The stripe pass-1 output
        # X1 inherits it (O[:, 31] / O[:, 31] == 1) and is the value operand of pass 2.
        self.ones_w, self.ones_s = dw < SLOT, ds < SLOT
        for half, (hh, on) in enumerate(((hw, self.ones_w), (hs, self.ones_s))):
            if on:
                base = (0 if half == 0 else 3 * hw) + 2 * hh
                for head in range(hh):
                    self.b_qkv[(base + head) * SLOT + SLOT - 1] = 1.0
        # --- anchor projection: dest row = head*32 + e
        amap = [head * SLOT + e for head in range(hs) for e in range(ds)]
        red = at.anchor.body[0].reduction
        self.n_anc = hs * SLOT
        self.w_anc = _pad_matrix(red.weight, round_up(self.n_anc, 32), self.cpad, row_map=amap, fmt=fmt)
        self.b_anc = _pad_vector(red.bias, round_up(self.n_anc, 32), amap)
        self.anc_scale = torch.ones(hs, device=red.weight.device, dtype=torch.float32)
        self.df = at.anchor.body[0].down_factor
        # --- output projection: K index = slot*32 + e over [window heads | stripe heads]
        cmap = [head * SLOT + e for head in range(hw) for e in range(dw)] + \
               [(hw + head) * SLOT + e for head in range(hs) for e in range(ds)]
        self.k_proj = round_up((hw + hs) * SLOT, 64)
        self.n_ln = 64 if C <= 64 else 128 if C <= 128 else 192 if C <= 192 else 256
        self.w_proj = _pad_matrix(at.proj.weight, self.n_ln, self.k_proj, col_map=cmap, fmt=fmt)
        self.b_proj = _pad_vector(at.proj.bias, self.n_ln)
        # --- MLP
        hid = blk.mlp.fc1.weight.shape[0]
        self.hid, self.hpad = hid, round_up(hid, 64)
        self.w_fc1 = _pad_matrix(blk.mlp.fc1.weight, self.hpad, self.cpad, fmt=fmt)
        self.b_fc1 = _pad_vector(blk.mlp.fc1.bias, self.hpad)
        self.w_fc2 = _pad_matrix(blk.mlp.fc2.weight, self.n_ln, self.hpad, fmt=fmt)
        self.b_fc2 = _pad_vector(blk.mlp.fc2.bias, self.n_ln)
        # --- CAB
        self.cab = bool(blk.args.local_connection)
        if self.cab:
            c0, c2 = blk.conv.cab[0], blk.conv.cab[2]
            self.cmid = c0.weight.shape[0]
            self.cmid_pad = round_up(self.cmid, 64)
            self.w_cab1, self.b_cab1 = pack_conv(c0, self.cpad, self.cmid_pad, fmt)
            self.w_cab2, self.b_cab2 = pack_conv(c2, self.cmid_pad, self.cpad, fmt)
            a1, a3 = blk.conv.cab[3].attention[1], blk.conv.cab[3].attention[3]
            self.ca = (a1.weight.detach().reshape(a1.weight.shape[0], -1).contiguous(), a1.bias.detach(),
                       a3.weight.detach().reshape(a3.weight.shape[0], -1).contiguous(), a3.bias.detach())

    @torch.no_grad()
    def run(self, blk, x32, x16, x_size, t):
        """x32 fp32 (B, L, C), x16 bf16 (B, L, cpad) or None -> (x32', x16')."""
        B, L, C = x32.shape
        H, W = x_size
        dev = x32.device
        at = blk.attn
        hw, hs, cpad = self.hw, self.hs, self.cpad
        fmt = self.fmt
        if x16 is None or x16.dtype != DTYPE[fmt]:
            x16 = pack_rows(x32, cpad, fmt)
        lib = capi.lib()
        wa, sa = at.window_attn, at.stripe_attn
        # attention constants of this block (slot scales + activated bias tables): functions of the parameters and
        # the coordinate tables only, so they are cached until a parameter or the resolution changes
        ckey = (self.key, t["table_w"].data_ptr(), t["table_s"].data_ptr(), t["table_s"].shape)
        if self._const_key != ckey:
            slot_scale = torch.empty(self.nslots, device=dev, dtype=torch.float32)
            capi.check(lib.grl_tc_slot_scale(capi.ptr(wa.attn_transform.logit_scale),
                                             capi.ptr(sa.attn_transform1.logit_scale),
                                             capi.ptr(sa.attn_transform2.logit_scale), hw, hs, capi.ptr(slot_scale),
                                             capi.stream()))
            self._consts = (slot_scale, bias_table_log2(wa.attn_transform, t["table_w"]),
                            bias_table_log2(sa.attn_transform1, t["table_s"]),
                            bias_table_log2(sa.attn_transform2, t["table_s"]))
            self._const_key = ckey
        slot_scale, bias_w, bias_1, bias_2 = self._consts
        # projections
        qkv = _h16(B * L, self.n_qkv, device=dev, fmt=fmt)
        gemm(x16, self.w_qkv, self.b_qkv, M=B * L, kpad=cpad, npad=self.n_qkv, epi=EPI_QKV, n_store=self.n_qkv,
             out_bf16=qkv, slot_scale=slot_scale)
        df = self.df
        pooled = _h16(B, H // df, W // df, cpad, device=dev, fmt=fmt)
        capi.check(lib.grl_tc_avgpool16(capi.ptr(x16), capi.ptr(pooled), B, H, W, cpad, df, fmt, capi.stream()))
        La = (H // df) * (W // df)
        n_anc = self.w_anc.shape[0]
        anchor = _h16(B * La, n_anc, device=dev, fmt=fmt)
        gemm(pooled, self.w_anc, self.b_anc, M=B * La, kpad=cpad, npad=n_anc, epi=EPI_QKV, n_store=n_anc, out_bf16=anchor,
             slot_scale=self.anc_scale)
        # attention
        merged = _h16(B * L, self.k_proj, device=dev, fmt=fmt, zero=self.k_proj != (hw + hs) * SLOT)
        s = wa.shift_size
        gw = G.token_grid(x_size, wa.window_size, (s, s))
        attention(gw, gw, qkv, 0, qkv, hw * SLOT, qkv, 2 * hw * SLOT, merged, 0, B, hw, bias_w, t["mask_w"] is not None,
                  tag="window_attn", ones_col=self.ones_w)
        tok, anc = sa.grids(x_size)
        nW = (tok.H // tok.wh) * (tok.W // tok.ww)
        x1 = _h16(B * nW * hs * anc.wh * anc.ww, SLOT, device=dev, fmt=fmt)
        use_mask = t["mask_a2w"] is not None
        attention(anc, tok, anchor, 0, qkv, (3 * hw + hs) * SLOT, qkv, (3 * hw + 2 * hs) * SLOT, x1, 0, B, hs, bias_1,
                  use_mask, o_dense=True, tag="stripe_attn", ones_col=self.ones_s)
        attention(tok, anc, qkv, 3 * hw * SLOT, anchor, 0, x1, 0, merged, hw * SLOT, B, hs, bias_2, use_mask,
                  v_dense=True, tag="stripe_attn", ones_col=self.ones_s)
        # CAB
        cab_y = gate = None
        if self.cab:
            t1 = _h16(B, H, W, self.cmid_pad, device=dev, fmt=fmt)
            conv3x3(x16.view(B, H, W, cpad), self.w_cab1, self.b_cab1, cpad, self.cmid_pad, n_store=self.cmid_pad,
                    act=K.ACT_GELU, out_bf16=t1)
            cab_y = _h16(B * L, cpad, device=dev, fmt=fmt)
            conv3x3(t1, self.w_cab2, self.b_cab2, self.cmid_pad, cpad, n_store=cpad, out_bf16=cab_y)
            nbytes = lib.grl_tc_channel_gate_workspace(B, L, C)
            ws = torch.empty(max(nbytes, 4) // 4, device=dev, dtype=torch.float32)
            gate = torch.empty(B, C, device=dev, dtype=torch.float32)
            w1, b1, w2, b2 = self.ca
            capi.check(lib.grl_tc_channel_gate(capi.ptr(cab_y), cpad, fmt, B, L, C, capi.ptr(w1), capi.ptr(b1), capi.ptr(w2),
                                               capi.ptr(b2), w1.shape[0], capi.ptr(gate), capi.ptr(ws), nbytes,
                                               capi.stream()))
        # proj + LN1 + residual (+ CAB)
        y32 = torch.empty(B, L, C, device=dev, dtype=torch.float32)
        y16 = _h16(B, L, cpad, device=dev, fmt=fmt)
        gemm(merged, self.w_proj, self.b_proj, M=B * L, kpad=self.k_proj, npad=self.n_ln, epi=EPI_LN, n_store=self.n_ln,
             n_real=C, out_bf16=y16, out_f32=y32, res_f32=x32, C=C, gamma=blk.norm1.weight, beta=blk.norm1.bias,
             eps=blk.norm1.eps, res_scale=blk.res_scale, cab_y=cab_y, cab_gate=gate, L=L)
        # MLP + LN2 + residual in one launch (the hidden activation stays on the SM)
        z32 = torch.empty(B, L, C, device=dev, dtype=torch.float32)
        z16 = _h16(B, L, cpad, device=dev, fmt=fmt)
        mlp(y16, self.w_fc1, self.b_fc1, self.w_fc2, self.b_fc2, M=B * L, C=C, out_f32=z32, out_bf16=z16, res_f32=y32,
            gamma=blk.norm2.weight, beta=blk.norm2.bias, eps=blk.norm2.eps, res_scale=blk.res_scale)
        return z32, z16


def block_plan(blk, fmt):
    plan = getattr(blk, "_tc_plan", None)
    if plan is None or plan.key != (_version_key(blk), fmt):
        plan = BlockPlan(blk, fmt)
        blk._tc_plan = plan
    return plan


class ConvPlan:
    """One packed 3x3 conv (stage conv / head convs)."""

    def __init__(self, conv, cin_pad, fmt, ps_r=0):
        self.key = (_version_key(conv), fmt, ps_r)
        self.cout = conv.weight.shape[0]
        self.cin_pad = cin_pad
        self.npad = round_up(self.cout, 64)
        self.w, self.b = pack_conv(conv, cin_pad, self.npad, fmt, ps_r)


def conv_plan(owner, name, conv, cin_pad, fmt, ps_r=0):
    cache = owner.__dict__.setdefault("_tc_convs", {})
    plan = cache.get(name)
    if plan is None or plan.key != (_version_key(conv), fmt, ps_r) or plan.cin_pad != cin_pad:
        plan = ConvPlan(conv, cin_pad, fmt, ps_r)
        cache[name] = plan
    return plan
