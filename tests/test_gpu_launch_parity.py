"""Every kernel launch of the benchmarked tensor-core forwards, compared with a float64 reference of that launch.

The whole-network tests compare fp16 outputs after ~250 launches with loose bounds, so a kernel that is wrong on one tile, one
window type, one head or one batch item can hide under them.  Here the real forward runs eagerly with every `monai_b200._kernels`
entry point that the network calls replaced by a checking wrapper.  The wrapper snapshots the launch's operands, runs the original,
and compares what it wrote with a float64 torch computation of the same operation on those operands, per batch item and with a bound
per entry point.  The reference never calls a monai_b200 kernel: NC8 buffers are unpacked with permute / reshape here.

- Fresh NC8 buffers are NaN-filled and callers that pass no `out` get a NaN-filled one, so an element a kernel leaves unwritten
  fails the check; after a call that writes a channel slice of a larger buffer, the other channels must be bit-for-bit unchanged.
- `K._call` is wrapped as well: a launch outside a checked wrapper fails the test (weight / bias packing excepted), and each
  configuration has a coverage list of variants that must have been seen.
- Weights reach the kernels as fp16 images: the reference uses the packed weight rounded to fp16, as the tensor core reads it.

Run with -s to see the report (entry point, launches, worst max / rms error relative to the item's max / rms, bound)."""
from __future__ import annotations

import contextlib
import functools
import inspect
import io
import math
import time
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from monai_b200 import _kernels as K
from monai_b200 import _lib as L
from weights import fill_state_dict

pytestmark = pytest.mark.gpu
DEV = "cuda"
LOG2E = 1.4426950408889634

# Bounds per entry point: (max |got - ref| / max |ref|, rms(got - ref) / rms(ref)), per batch item.
TOL = {
    "conv3x3x3_tc": (3e-3, 1e-3),
    "gemm_tc": (3e-3, 1e-3),
    "window_attention_tc": (4e-3, 1e-3),
    "mlp_fused_tc": (3e-3, 1e-3),
    "layernorm_nc8": (3e-3, 1e-3),
    "patch_merge_ln_nc8": (3e-3, 1e-3),
    "norm_act_nc8": (3e-3, 1e-3),
    "norm_act_cin1res_nc8": (3e-3, 1e-3),
    "head_conv_norm_nc8": (3e-3, 1e-3),
    "conv_cin1_nc8": (3e-3, 1e-3),
    "conv_gather_tc": (3e-3, 1e-3),
    "convt3s2_head_nc8": (3e-3, 1e-3),
    "pack_nc8": (0.0, 0.0),
    "copy_channels": (0.0, 0.0),
}
# statistics outputs {sum, sum of squares} per (n, c): |d sum| / sum |y| and |d sumsq| / sum y^2
STATS_TOL = (1e-3, 2e-3)
# entry points that only prepare weights / biases (their products are checked through the launches that read them)
PREP = ("conv3x3x3_tc_pack_weight", "gemm_tc_pack_weight", "conv_gather_tc_pack_weight", "window_attention_tc_pack_bias")


# ----------------------------------------------------------------------------------------------------- helpers
def _nc(buf: torch.Tensor, items) -> torch.Tensor:
    """NC8 buffer [N, C/8, D, H, W, 8] -> NCDHW [len(items), C, D, H, W] (same dtype)."""
    t = buf[items]
    n, c8 = t.shape[:2]
    return t.permute(0, 1, 5, 2, 3, 4).reshape(n, c8 * 8, *t.shape[2:5])


def _act(x: torch.Tensor, act: int, slope: float) -> torch.Tensor:
    if act == L.ACT_NONE:
        return x
    if act == L.ACT_LEAKY:
        return torch.where(x >= 0, x, x * slope)
    if act == L.ACT_RELU:
        return x.clamp_min(0)
    if act == L.ACT_GELU:
        return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))
    raise AssertionError(f"activation {act} has no reference here")


def _inorm(x: torch.Tensor, stats: torch.Tensor, items, eps: float) -> torch.Tensor:
    """Instance norm of x [n, C, *sp] (float64) with mean / biased variance from the GIVEN {sum, sumsq} statistics [N*C, 2]."""
    n, c = x.shape[:2]
    st = stats.reshape(-1, c, 2)[items].double()
    S = x[0, 0].numel()
    mean = st[..., 0] / S
    var = (st[..., 1] / S - mean * mean).clamp_min(0)
    rstd = 1.0 / torch.sqrt(var + eps)
    shape = (n, c) + (1,) * (x.dim() - 2)
    return (x - mean.reshape(shape)) * rstd.reshape(shape)


def _f16(w: torch.Tensor) -> torch.Tensor:
    """A weight as the tensor core reads it: rounded to fp16, then widened to float64."""
    return w.float().half().double()


def _rel_index(ws) -> torch.Tensor:
    """relative_position_index of a WindowAttention module with window ws (swin_unetr.py:449-461)."""
    coords = torch.stack(torch.meshgrid(*(torch.arange(w) for w in ws), indexing="ij")).flatten(1)
    rel = (coords[:, :, None] - coords[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += ws[0] - 1
    rel[:, :, 1] += ws[1] - 1
    rel[:, :, 2] += ws[2] - 1
    rel[:, :, 0] *= (2 * ws[1] - 1) * (2 * ws[2] - 1)
    rel[:, :, 1] *= 2 * ws[2] - 1
    return rel.sum(-1)


def _snap(v):
    if isinstance(v, K.NC8):
        return K.NC8(v.N, v.C, v.sp, None, buf=v.buf.clone())
    if torch.is_tensor(v):
        return v.clone()
    if isinstance(v, tuple):
        return tuple(_snap(e) for e in v)
    return v


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


class Harness:
    def __init__(self, items, inject=None):
        self.items = items
        self.inject = inject
        self.rows: list[dict] = []
        self.launched: list[tuple[str, str | None]] = []   # (entry point, checked wrapper it ran under or None)
        self.seen: set[str] = set()
        self.weights: dict = {}       # packed weight data_ptr -> (packed tensor, source weight float32)
        self.biases: dict = {}        # packed attention bias data_ptr -> (packed, table, heads, n, window, region_types, ntypes)
        self.concat: set = set()      # data_ptrs of buffers written slice by slice (decoder concat buffers)
        self.active: str | None = None
        self.launch_id = 0

    # -- reporting
    def cmp(self, op, what, got, ref, tol=None):
        """One output of one launch: per batch item relative max and rms error (NaN / Inf anywhere fails)."""
        tmax, trms = TOL[op] if tol is None else tol
        worst_m = worst_r = 0.0
        for i in range(ref.shape[0]):
            g, r = got[i].double(), ref[i]
            if not (torch.isfinite(g).all() and torch.isfinite(r).all()):
                worst_m = worst_r = math.inf
                continue
            d = g - r
            amax, rrms = float(r.abs().max()), float(r.pow(2).mean().sqrt())
            worst_m = max(worst_m, float(d.abs().max()) / (amax if amax > 0 else 1.0))
            worst_r = max(worst_r, float(d.pow(2).mean().sqrt()) / (rrms if rrms > 0 else 1.0))
        self._row(op, what, tuple(got.shape), worst_m, worst_r, (tmax, trms))

    def cmp_stats(self, op, what, stats, y_ref):
        """{sum, sumsq} statistics [N*C, 2] against those of the float64 reference output y_ref [n_items, C, ...]."""
        c = y_ref.shape[1]
        g = stats.reshape(-1, c, 2)[self.items].double()
        y = y_ref.reshape(y_ref.shape[0], c, -1)
        s, q, a = y.sum(-1), (y * y).sum(-1), y.abs().sum(-1)
        if not torch.isfinite(g).all():
            e1 = e2 = math.inf
        else:
            e1 = float(((g[..., 0] - s).abs() / a.clamp_min(1e-30)).max())
            e2 = float(((g[..., 1] - q).abs() / q.clamp_min(1e-30)).max())
        self._row(op, what, tuple(stats.shape), e1, e2, STATS_TOL)

    def untouched(self, op, before: torch.Tensor, after: torch.Tensor, c0: int, c1: int):
        """Channels [0, c0) and [c1, C) of a destination must keep their bits (dim 1 indexes channels or 8-channel blocks)."""
        ok = all(torch.equal(_bits(before[:, sl]), _bits(after[:, sl])) for sl in (slice(0, c0), slice(c1, None)))
        self._row(op, "untouched", tuple(after.shape), 0.0 if ok else math.inf, 0.0 if ok else math.inf, (0.0, 0.0))

    def finite(self, op, what, t: torch.Tensor):
        """Every batch item (also those without a reference) holds finite values: nothing was left at the NaN poison."""
        ok = bool(torch.isfinite(t).all())
        self._row(op, what + " finite", tuple(t.shape), 0.0 if ok else math.inf, 0.0 if ok else math.inf, (0.0, 0.0))

    def _row(self, op, what, shape, m, r, tol):
        ok = m <= tol[0] and r <= tol[1]
        self.rows.append(dict(id=self.launch_id, op=op, what=what, shape=shape, max=m, rms=r, tol=tol, ok=ok))

    def tag(self, op, *tags):
        for t in tags:
            self.seen.add(f"{op}:{t}")

    def nc8_out(self, N, C, sp, dev):
        nc8 = K.NC8(N, C, sp, dev)
        nc8.buf.fill_(float("nan"))
        return nc8

    def report(self, title, seconds):
        lines = [f"\n{title}: {self.launch_id} checked launches, {seconds:.1f} s",
                 f"{'entry point':24s} {'launches':>8s} {'worst max':>10s} {'worst rms':>10s} {'bound':>16s}"]
        ops: dict = {}
        for r in self.rows:
            if r["what"] in ("untouched",) or r["what"].endswith("finite"):
                continue
            key = r["op"] + (" stats" if "stats" in r["what"] else "")
            d = ops.setdefault(key, dict(ids=set(), m=0.0, r=0.0, tol=r["tol"]))
            d["ids"].add(r["id"])
            d["m"], d["r"] = max(d["m"], r["max"]), max(d["r"], r["rms"])
        for k in sorted(ops):
            d = ops[k]
            lines.append(f"{k:24s} {len(d['ids']):8d} {d['m']:10.2e} {d['r']:10.2e} {d['tol'][0]:7.0e}/{d['tol'][1]:7.0e}")
        print("\n".join(lines))


# ----------------------------------------------------------------------------------- per entry point references
def _chk_conv3x3x3_tc(h, pre, a, ret):
    it = h.items
    x, cin, cout, coff = pre["x"], a["Cin"], a["Cout"], a["in_coff"]
    xin = _nc(x.buf, it)[:, coff: coff + cin].double()
    tags = ["plain"]
    if a["x"].buf.data_ptr() in h.concat:   # the buffer the launch read, not its snapshot
        tags.append("concat_in")
    if coff:
        tags.append("in_coff")
    if pre["in_norm"] is not None:
        st, eps, act, slope = pre["in_norm"]
        xin = _act(_inorm(xin, st, it, eps), act, slope).half().double()   # the fp16 operand the kernel feeds the tensor core
        tags.append("in_norm")
    w = _f16(h.weights[a["packed_w"].data_ptr()][1])
    b = None if a["bias"] is None else a["bias"].double()
    y = F.conv3d(xin, w, b, padding=1)
    out, oc = ret[0], a["out_coff"]
    h.cmp("conv3x3x3_tc", "out", _nc(out.buf, it)[:, oc: oc + cout], y)
    h.finite("conv3x3x3_tc", "out", out.buf[:, oc // 8: (oc + cout) // 8])
    if ret[1] is not None:
        h.cmp_stats("conv3x3x3_tc", "stats", ret[1], y)
        tags.append("want_stats")
    if a["res_w"] is not None:
        w3 = _f16(h.weights[a["res_w"].data_ptr()][1]).reshape(cout, cin, 1, 1, 1)
        y3 = F.conv3d(xin, w3)
        h.cmp("conv3x3x3_tc", "res_out", _nc(ret[2].buf, it), y3)
        h.finite("conv3x3x3_tc", "res_out", ret[2].buf)
        if ret[3] is not None:
            h.cmp_stats("conv3x3x3_tc", "res_stats", ret[3], y3)
        tags.append("res_w")
    return tags


def _chk_gemm_tc(h, pre, a, ret):
    it = h.items
    x, kd, n, mode = pre["x"], a["Kd"], a["N"], a["mode"]
    xin = _nc(x.buf, it)[:, a["in_coff"]: a["in_coff"] + kd].double().reshape(len(it), kd, -1)
    w = _f16(h.weights[a["packed_w"].data_ptr()][1])             # [N, K]
    y = torch.einsum("nks,ok->nos", xin, w)
    if a["bias"] is not None:
        y = y + a["bias"].double()[None, :, None]
    y = _act(y, a["act"], 0.0)
    out = ret[0]
    cout = n // 8 if mode == 2 else n
    tags = [f"mode{mode}"]
    if mode == 0:
        dst = y.reshape(len(it), n, *x.sp)
    elif mode == 1:
        rm = pre["row_map"].long()
        valid = rm >= 0
        cover = torch.bincount(rm[valid], minlength=out.S)
        h._row("gemm_tc", "row_map covers destination", (out.S,), 0.0 if bool((cover == 1).all()) else math.inf, 0.0, (0.0, 0.0))
        dst = torch.zeros((len(it), n, out.S), dtype=torch.float64, device=y.device)
        dst[:, :, rm[valid]] = y[:, :, valid]
        dst = dst.reshape(len(it), n, *out.sp)
    else:
        D, H, W = x.sp
        dst = y.reshape(len(it), 2, 2, 2, cout, D, H, W).permute(0, 4, 5, 1, 6, 2, 7, 3).reshape(len(it), cout, 2 * D, 2 * H, 2 * W)
    if pre["res"] is not None:
        dst = dst + _nc(pre["res"].buf, it)[:, a["res_coff"]: a["res_coff"] + cout].double()
        tags.append("res")
    if a["act"] != L.ACT_NONE:
        tags.append("act")
    oc = a["out_coff"]
    h.cmp("gemm_tc", f"out mode {mode}", _nc(out.buf, it)[:, oc: oc + cout], dst)
    h.finite("gemm_tc", "out", out.buf[:, oc // 8: (oc + cout) // 8])
    if ret[1] is not None:
        assert mode == 0, "column statistics are only referenced for mode 0"
        h.cmp_stats("gemm_tc", "stats", ret[1], dst)
        tags.append("want_stats")
    return tags


def _chk_window_attention_tc(h, pre, a, ret):
    it = h.items
    qkv, C, heads, nW, n, ntypes = pre["qkv"], a["Cc"], a["heads"], a["nW"], a["n"], a["ntypes"]
    packed, table, b_heads, b_n, window, reps, b_ntypes = h.biases[a["packed_bias"].data_ptr()]
    assert (b_heads, b_n, b_ntypes) == (heads, n, ntypes)
    q, k, v = _nc(qkv.buf, it)[:, : 3 * C].double().reshape(len(it), 3, heads, 16, nW, n).permute(1, 0, 2, 4, 5, 3)
    idx = _rel_index(window)[:n, :n].reshape(-1).to(table.device)
    bias = table.double()[idx].reshape(n, n, heads).permute(2, 0, 1)   # [heads, n, n]
    sched = pre["sched"].cpu().numpy()
    ref = torch.zeros((len(it), heads, nW, n, 16), dtype=torch.float64, device=q.device)
    for t in range(ntypes):
        ids = torch.from_numpy(sched[16 + sched[8 + t]: 16 + sched[8 + t] + sched[t]].astype(np.int64)).to(q.device)
        mask = 0.0
        if reps is not None:
            lab = reps[t]
            mask = torch.where(lab[None, :] != lab[:, None], -100.0, 0.0).double()
        # the kernel reads log2(e) * (bias + mask) as an fp16 operand
        bt = ((bias + mask) * LOG2E).half().double() / LOG2E
        for i in range(len(it)):
            s = q[i][:, ids] @ k[i][:, ids].transpose(-1, -2) / LOG2E + bt[:, None]
            ref[i][:, ids] = s.softmax(-1) @ v[i][:, ids]
    ref = ref.permute(0, 1, 4, 2, 3).reshape(len(it), C, 1, nW, n)
    h.cmp("window_attention_tc", f"out n={n} types={ntypes}", _nc(ret.buf, it), ref)
    h.finite("window_attention_tc", "out", ret.buf)
    return ["ntypes1" if ntypes == 1 else "ntypes>1", f"n{n}"]


def _chk_mlp_fused_tc(h, pre, a, ret):
    it = h.items
    x, hid = pre["x"], a["hidden"]
    C = x.C
    t = _nc(x.buf, it).double().reshape(len(it), C, -1).transpose(1, 2)
    g = None if a["gamma"] is None else a["gamma"].double()
    b = None if a["beta"] is None else a["beta"].double()
    w1, w2 = _f16(h.weights[a["packed_w1"].data_ptr()][1]), _f16(h.weights[a["packed_w2"].data_ptr()][1])
    u = F.layer_norm(t, (C,), g, b, a["eps"]) @ w1.T + a["b1"].double()
    y = t + _act(u, L.ACT_GELU, 0.0) @ w2.T + a["b2"].double()
    h.cmp("mlp_fused_tc", "out", _nc(ret.buf, it), y.transpose(1, 2).reshape(len(it), C, *x.sp))
    h.finite("mlp_fused_tc", "out", ret.buf)
    return ["plain"]


def _chk_layernorm_nc8(h, pre, a, ret):
    it = h.items
    x = pre["x"]
    t = _nc(x.buf, it).double().reshape(len(it), x.C, -1).transpose(1, 2)
    g = None if a["gamma"] is None else a["gamma"].double()
    b = None if a["beta"] is None else a["beta"].double()
    y = F.layer_norm(t, (x.C,), g, b, a["eps"])
    tags = ["affine" if g is not None else "no_affine"]
    if pre["src"] is not None:
        src = pre["src"].long()
        valid = src >= 0
        z = torch.zeros((len(it), src.numel(), x.C), dtype=torch.float64, device=y.device)
        z[:, valid] = y[:, src[valid]]
        y = z
        tags.append("src")
    out = ret
    h.cmp("layernorm_nc8", "out", _nc(out.buf, it), y.transpose(1, 2).reshape(len(it), x.C, *out.sp))
    h.finite("layernorm_nc8", "out", out.buf)
    return tags


MERGE_V1 = [(0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, 1, 1)]
MERGE_V2 = [(i, j, k) for i in range(2) for j in range(2) for k in range(2)]


def _chk_patch_merge_ln_nc8(h, pre, a, ret):
    it = h.items
    x = pre["x"]
    t = _nc(x.buf, it).double().permute(0, 2, 3, 4, 1)
    D, H, W = x.sp
    t = F.pad(t, (0, 0, 0, W % 2, 0, H % 2, 0, D % 2))
    cat = torch.cat([t[:, i::2, j::2, k::2, :] for i, j, k in (MERGE_V2 if a["v2"] else MERGE_V1)], -1)
    y = F.layer_norm(cat, (8 * x.C,), a["gamma"].double(), a["beta"].double(), a["eps"]).permute(0, 4, 1, 2, 3)
    h.cmp("patch_merge_ln_nc8", "out", _nc(ret.buf, it), y)
    h.finite("patch_merge_ln_nc8", "out", ret.buf)
    return ["v2" if a["v2"] else "v1"] + (["odd"] if any(s % 2 for s in x.sp) else [])


def _chk_norm_act_nc8(h, pre, a, ret):
    it = h.items
    x, c = pre["x"], a["C_"]
    y = _nc(x.buf, it)[:, a["x_coff"]: a["x_coff"] + c].double()
    tags = []
    if pre["stats"] is not None:
        y = _inorm(y, pre["stats"], it, a["eps"])
        tags.append("norm")
    else:
        tags.append("copy")
    if pre["res"] is not None:
        r = _nc(pre["res"].buf, it)[:, a["res_coff"]: a["res_coff"] + c].double()
        if pre["res_stats"] is not None:
            r = _inorm(r, pre["res_stats"], it, a["eps"])
            tags.append("res_norm")
        else:
            tags.append("res")
        y = y + r
    y = _act(y, a["act"], a["slope"])
    oc = a["out_coff"]
    if oc:
        tags.append("out_coff")
    h.cmp("norm_act_nc8", "out", _nc(ret.buf, it)[:, oc: oc + c], y)
    h.finite("norm_act_nc8", "out", ret.buf[:, oc // 8: (oc + c) // 8])
    return tags


def _chk_norm_act_cin1res_nc8(h, pre, a, ret):
    it = h.items
    x, c, eps = pre["x"], a["C_"], a["eps"]
    y = _inorm(_nc(x.buf, it)[:, :c].double(), pre["stats"], it, eps)
    u = pre["raw"][it].double()                                  # [n, 1, *sp]
    rs = pre["raw_stats"].reshape(-1, 2)[it].double()
    S = u[0, 0].numel()
    mu = rs[:, 0] / S
    var = (rs[:, 1] / S - mu * mu).clamp_min(0)
    w = pre["raw_weight"].reshape(-1).float().double()           # conv3 weights, one per output channel
    sh = (len(it), 1, 1, 1, 1)
    r = (w[None, :, None, None, None] * (u - mu.reshape(sh))) / torch.sqrt(w[None, :, None, None, None] ** 2 * var.reshape(sh) + eps)
    y = _act(y + r, a["act"], a["slope"])
    oc = a["out_coff"]
    h.cmp("norm_act_cin1res_nc8", "out", _nc(ret.buf, it)[:, oc: oc + c], y)
    h.finite("norm_act_cin1res_nc8", "out", ret.buf[:, oc // 8: (oc + c) // 8])
    return ["plain"] + (["out_coff"] if oc else [])


def _chk_head_conv_norm_nc8(h, pre, a, ret):
    it = h.items
    x, eps = pre["x"], a["eps"]
    t = _inorm(_nc(x.buf, it).double(), pre["stats"], it, eps)
    tags = []
    if pre["res"] is not None:
        r = _nc(pre["res"].buf, it)[:, a["res_coff"]: a["res_coff"] + x.C].double()
        if pre["res_stats"] is not None:
            r = _inorm(r, pre["res_stats"], it, eps)
            tags.append("res_norm")
        else:
            tags.append("res")
        t = t + r
    t = _act(t, L.ACT_LEAKY, a["slope"])
    w = a["weight"].float().double().reshape(a["weight"].shape[0], -1)
    y = torch.einsum("nc...,oc->no...", t, w)
    if a["bias"] is not None:
        y = y + a["bias"].float().double().reshape(1, -1, 1, 1, 1)
    h.cmp("head_conv_norm_nc8", "out", ret[it], y)
    h.finite("head_conv_norm_nc8", "out", ret)
    return tags


def _chk_instnorm_stats(h, pre, a, ret):
    h.cmp_stats("instnorm_stats", "stats", ret, pre["x"][h.items].double())
    return ["plain"]


def _chk_conv_cin1_nc8(h, pre, a, ret, entry):
    it = h.items
    x, k, s, p = pre["x"], a["k"], a["stride"], a["pad"]
    w, b = pre["weight"].float(), pre["bias"]
    xin = x[it].double()
    if entry == "conv_cin1_tc":   # tensor-core stem: fp16 operands (input and weights rounded on the way into shared memory)
        xin, w = xin.float().half().double(), w.half()
    y = F.conv3d(xin, w.double(), None if b is None else b.float().double(), stride=s, padding=p)
    out, oc, cout = ret[0], a["out_coff"], pre["weight"].shape[0]
    h.cmp("conv_cin1_nc8", f"out {entry}", _nc(out.buf, it)[:, oc: oc + cout], y)
    h.finite("conv_cin1_nc8", "out", out.buf[:, oc // 8: (oc + cout) // 8])
    if ret[1] is not None:
        h.cmp_stats("conv_cin1_nc8", "stats", ret[1], y)
    return [f"{entry}_k{k}s{s}", f"{entry}_k{k}s{s}_{'f16' if x.dtype == torch.float16 else 'f32'}"]


def _chk_conv_gather_tc(h, pre, a, ret):
    it = h.items
    x, cin, cout, k, s, p, tr = pre["x"], a["Cin"], a["Cout"], a["k"], a["stride"], a["pad"], a["transposed"]
    xin = _nc(x.buf, it)[:, a["in_coff"]: a["in_coff"] + cin].double()
    w = _f16(h.weights[a["packed_w"].data_ptr()][1])
    b = None if a["bias"] is None else a["bias"].float().double()
    if tr:
        y = F.conv_transpose3d(xin, w, b, stride=s, padding=p, output_padding=a["output_padding"])
    else:
        y = F.conv3d(xin, w, b, stride=s, padding=p)
    out = ret[0]
    tags = [f"{'convT' if tr else 'conv'}_k{k}s{s}"]
    if isinstance(out, K.NC8):
        oc = a["out_coff"]
        h.cmp("conv_gather_tc", "out nc8", _nc(out.buf, it)[:, oc: oc + cout], y)
        h.finite("conv_gather_tc", "out", out.buf[:, oc // 8: (oc + cout) // 8])
        tags.append("nc8")
    else:
        h.cmp("conv_gather_tc", "out ncdhw", out[it], y)
        h.finite("conv_gather_tc", "out", out)
        tags.append("ncdhw")
    if a["in_coff"] or cin != x.C:
        tags.append("in_slice")
    if ret[1] is not None:
        h.cmp_stats("conv_gather_tc", "stats", ret[1], y)
        tags.append("want_stats")
    return tags


def _chk_convt3s2_head_nc8(h, pre, a, ret):
    it = h.items
    x, cin = pre["x"], a["Cin"]
    xin = _nc(x.buf, it)[:, a["in_coff"]: a["in_coff"] + cin].double()
    b = None if a["bias"] is None else a["bias"].float().double()
    y = F.conv_transpose3d(xin, a["weight"].float().double(), b, stride=2, padding=1, output_padding=1)
    h.cmp("convt3s2_head_nc8", "out", ret[it], y)
    h.finite("convt3s2_head_nc8", "out", ret)
    return ["plain"]


def _chk_pack_nc8(h, pre, a, ret):
    it = h.items
    x, c0 = pre["x"], a["c_off"]
    got = _nc(ret.buf, it)[:, c0: c0 + x.shape[1]]
    h.cmp("pack_nc8", "out", got.reshape(got.shape[0], got.shape[1], -1), x[it].half().double().reshape(len(it), x.shape[1], -1))
    h.finite("pack_nc8", "out", ret.buf[:, c0 // 8: (c0 + x.shape[1]) // 8])
    return ["plain"]


def _chk_copy_channels(h, pre, a, ret):
    it = h.items
    x, dst, c0 = pre["x"], a["dst"], a["c_off"]
    Di, Hi, Wi = x.shape[2:]
    Do, Ho, Wo = dst.shape[2:]
    ix = [torch.arange(o, device=x.device).clamp_max(i - 1) for i, o in ((Di, Do), (Hi, Ho), (Wi, Wo))]
    want = x[it][:, :, ix[0]][:, :, :, ix[1]][:, :, :, :, ix[2]]
    h.cmp("copy_channels", "out", dst[it][:, c0: c0 + x.shape[1]], want.double())
    return ["plain"]


def _make_out_conv3(a):
    x = a["x"]
    return K.NC8(x.N, a["Cout"], x.sp, x.buf.device)


def _make_out_gemm(a):
    x, mode = a["x"], a["mode"]
    sp = tuple(a["out_sp"]) if a["out_sp"] is not None else (tuple(2 * s for s in x.sp) if mode == 2 else x.sp)
    return K.NC8(x.N, a["N"] // 8 if mode == 2 else a["N"], sp, x.buf.device)


def _make_out_ln(a):
    x = a["x"]
    return K.NC8(x.N, x.C, tuple(a["out_sp"]) if a["out_sp"] is not None else x.sp, x.buf.device)


def _make_out_norm(a):
    x = a["x"]
    return K.NC8(x.N, a["C_"], x.sp, x.buf.device)


def _make_out_cin1(a):
    x = a["x"]
    sp = tuple((s + 2 * a["pad"] - a["k"]) // a["stride"] + 1 for s in x.shape[2:])
    return K.NC8(x.shape[0], a["weight"].shape[0], sp, x.device)


def _make_out_gather(a):
    x = a["x"]
    sp = K.conv_out_shape(x.sp, (a["k"],) * 3, (a["stride"],) * 3, (a["pad"],) * 3, a["transposed"], (a["output_padding"],) * 3)
    if a["ncdhw_dtype"] is None:
        return K.NC8(x.N, a["Cout"], sp, x.buf.device)
    return torch.full((x.N, a["Cout"], *sp), float("nan"), device=x.buf.device, dtype=a["ncdhw_dtype"])


def _make_out_pack(a):
    x = a["x"]
    return K.NC8(x.shape[0], x.shape[1], x.shape[2:], x.device)


# entry point -> (check, maker of the NaN-filled `out` when the caller passes none, name of that argument, written channels)
CHECKED = {
    "conv3x3x3_tc": (_chk_conv3x3x3_tc, _make_out_conv3, "out", lambda a: (a["out_coff"], a["Cout"])),
    "gemm_tc": (_chk_gemm_tc, _make_out_gemm, "out", lambda a: (a["out_coff"], a["N"] // 8 if a["mode"] == 2 else a["N"])),
    "window_attention_tc": (_chk_window_attention_tc, None, None, None),
    "mlp_fused_tc": (_chk_mlp_fused_tc, None, None, None),
    "layernorm_nc8": (_chk_layernorm_nc8, _make_out_ln, "out", lambda a: (0, a["x"].C)),
    "patch_merge_ln_nc8": (_chk_patch_merge_ln_nc8, None, None, None),
    "norm_act_nc8": (_chk_norm_act_nc8, _make_out_norm, "out", lambda a: (a["out_coff"], a["C_"])),
    "norm_act_cin1res_nc8": (_chk_norm_act_cin1res_nc8, _make_out_norm, "out", lambda a: (a["out_coff"], a["C_"])),
    "head_conv_norm_nc8": (_chk_head_conv_norm_nc8, None, None, None),
    "instnorm_stats": (_chk_instnorm_stats, None, None, None),
    "conv_cin1_nc8": (_chk_conv_cin1_nc8, _make_out_cin1, "out", lambda a: (a["out_coff"], a["weight"].shape[0])),
    "conv_gather_tc": (_chk_conv_gather_tc, _make_out_gather, "out", lambda a: (a["out_coff"], a["Cout"])),
    "convt3s2_head_nc8": (_chk_convt3s2_head_nc8, None, None, None),
    "pack_nc8": (_chk_pack_nc8, _make_out_pack, "dst", lambda a: (a["c_off"], a["x"].shape[1])),
    "copy_channels": (_chk_copy_channels, None, "dst", lambda a: (a["c_off"], a["x"].shape[1])),
}


def _checked(h: Harness, name: str, orig):
    check, make_out, out_arg, written = CHECKED[name]
    sig = inspect.signature(orig)

    @functools.wraps(orig)
    def wrapper(*args, **kwargs):
        if h.active is not None:   # nested inside another checked call: that call's check covers it
            return orig(*args, **kwargs)
        ba = sig.bind(*args, **kwargs)
        ba.apply_defaults()
        a = dict(ba.arguments)
        passed_out = out_arg is not None and a.get(out_arg) is not None
        if make_out is not None and not passed_out:
            out = make_out(a)
            if isinstance(out, K.NC8):
                out.buf.fill_(float("nan"))
            a[out_arg] = out
        pre = {k: _snap(v) for k, v in a.items()}
        first = len(h.launched)
        h.active = name
        try:
            ret = orig(**a)
        finally:
            h.active = None
        torch.cuda.synchronize()
        entries = {e for e, _ in h.launched[first:]}
        if h.inject is not None:
            h.inject(h, name, a, ret)
        if name == "conv_cin1_nc8":
            tags = check(h, pre, a, ret, entries.pop())
        else:
            tags = check(h, pre, a, ret)
        h.tag(name, *tags)
        if passed_out:   # a pre-existing destination: only the written channel slice may change
            dst = a[out_arg]
            c0, c = written(a)
            before, after = (pre[out_arg].buf, dst.buf) if isinstance(dst, K.NC8) else (pre[out_arg], dst)
            blk = 8 if isinstance(dst, K.NC8) else 1
            h.untouched(name, before, after, c0 // blk, (c0 + c) // blk)
            if c0 or c != (dst.C if isinstance(dst, K.NC8) else dst.shape[1]):
                h.concat.add(dst.buf.data_ptr() if isinstance(dst, K.NC8) else dst.data_ptr())
        h.launch_id += 1
        return ret

    return wrapper


def install(h: Harness, monkeypatch) -> None:
    """Wrap K._call (launch log), the weight / bias packers (recorded for the references) and every checked entry point.
    Must run before the network's first forward: packed weights are cached on first use."""
    orig_call = K._call

    def call(name, *args, **kwargs):
        h.launched.append((name, h.active))
        return orig_call(name, *args, **kwargs)

    monkeypatch.setattr(K, "_call", call)

    orig_init = K.NC8.__init__

    def nc8_init(self, N, C_, sp, device, buf=None):
        orig_init(self, N, C_, sp, device, buf)
        if buf is None:
            self.buf.fill_(float("nan"))   # fresh buffers start poisoned: unwritten elements show up as NaN

    monkeypatch.setattr(K.NC8, "__init__", nc8_init)

    def rec_weight(orig, src_arg):
        @functools.wraps(orig)
        def wrapper(*args, **kwargs):
            ba = inspect.signature(orig).bind(*args, **kwargs)
            src = ba.arguments[src_arg].detach().float().clone()
            packed = orig(*args, **kwargs)
            h.weights[packed.data_ptr()] = (packed, src)
            return packed

        return wrapper

    monkeypatch.setattr(K, "conv3x3x3_tc_pack_weight", rec_weight(K.conv3x3x3_tc_pack_weight, "weight"))
    monkeypatch.setattr(K, "gemm_tc_pack_weight", rec_weight(K.gemm_tc_pack_weight, "w2d"))
    monkeypatch.setattr(K, "conv_gather_tc_pack_weight", rec_weight(K.conv_gather_tc_pack_weight, "weight"))
    orig_bias = K.window_attention_tc_pack_bias

    def pack_bias(table, heads, n, window, region_types, ntypes):
        packed = orig_bias(table, heads, n, window, region_types, ntypes)
        h.biases[packed.data_ptr()] = (packed, table.detach().float().clone(), heads, n, tuple(int(w) for w in window),
                                       None if region_types is None else region_types.clone(), ntypes)
        return packed

    monkeypatch.setattr(K, "window_attention_tc_pack_bias", pack_bias)
    for name in CHECKED:
        monkeypatch.setattr(K, name, _checked(h, name, getattr(K, name)))


# ------------------------------------------------------------------------------------------------ configurations
def _build(kind: str, half: bool):
    from monai_b200.networks.nets import SwinUNETR, UNet

    with contextlib.redirect_stdout(io.StringIO()):
        if kind == "swin48":
            net = SwinUNETR(in_channels=1, out_channels=2, feature_size=48)
        elif kind == "swin48_in4_v2":
            net = SwinUNETR(in_channels=4, out_channels=3, feature_size=48, use_v2=True)
        elif kind == "unet_c2":
            net = UNet(3, 1, 2, (16, 32, 64, 128, 256), (2, 2, 2, 2))
        else:
            raise ValueError(kind)
    net.load_state_dict(fill_state_dict(net.state_dict(), 1))   # the weights bench.py uses
    net = net.eval().to(DEV)
    net = net.half() if half else net
    net._graph_enabled = False   # eager launches: a replayed CUDA graph would bypass the wrappers
    return net


SWIN = [
    "gemm_tc:mode0", "gemm_tc:mode1", "gemm_tc:mode2", "gemm_tc:want_stats", "gemm_tc:act", "gemm_tc:res",
    "window_attention_tc:ntypes1", "window_attention_tc:ntypes>1",
    "conv3x3x3_tc:res_w", "conv3x3x3_tc:in_norm", "conv3x3x3_tc:concat_in", "conv3x3x3_tc:want_stats",
    "mlp_fused_tc:plain", "patch_merge_ln_nc8:v1", "layernorm_nc8:src", "layernorm_nc8:no_affine",
    "norm_act_cin1res_nc8:out_coff", "norm_act_nc8:copy", "norm_act_nc8:out_coff", "norm_act_nc8:res_norm",
    "head_conv_norm_nc8:res_norm", "instnorm_stats:plain",
    "conv_cin1_nc8:conv_cin1_tc_k2s2", "conv_cin1_nc8:conv_cin1_tc_k3s1",
]
SWIN_F32 = [c for c in SWIN if not c.startswith("norm_act_cin1res_nc8") and c != "instnorm_stats:plain"] + [
    "conv_cin1_nc8:conv_cin1_tc_k2s2_f32", "conv_cin1_nc8:conv_cin1_tc_k3s1_f32", "conv_cin1_nc8:conv_cin1_nc8_k1s1_f32",
]
SWIN_IN4_V2 = [
    "copy_channels:plain", "pack_nc8:plain", "conv_gather_tc:conv_k2s2", "conv3x3x3_tc:plain", "conv3x3x3_tc:res_w",
    "conv3x3x3_tc:in_norm", "gemm_tc:mode0", "gemm_tc:mode1", "gemm_tc:mode2", "gemm_tc:want_stats",
    "window_attention_tc:ntypes1", "window_attention_tc:ntypes>1", "window_attention_tc:n64", "mlp_fused_tc:plain",
    "patch_merge_ln_nc8:v1", "layernorm_nc8:src", "norm_act_nc8:res", "norm_act_nc8:res_norm", "norm_act_nc8:out_coff",
    "head_conv_norm_nc8:res_norm",
]
UNET = [
    "conv_cin1_nc8:conv_cin1_nc8_k3s2", "conv_gather_tc:conv_k3s2", "conv_gather_tc:conv_k3s1", "conv_gather_tc:convT_k3s2",
    "conv_gather_tc:want_stats", "conv_gather_tc:in_slice", "norm_act_nc8:norm", "norm_act_nc8:out_coff", "convt3s2_head_nc8:plain",
]

CONFIGS = {
    # id: (network, fp16 weights, input shape, input dtype, batch items with a reference, coverage list)
    "swin48_96": ("swin48", True, (2, 1, 96, 96, 96), torch.float16, [0, 1], SWIN + ["window_attention_tc:n343", "window_attention_tc:n216"]),
    "swin48_96x64x64_f32": ("swin48", False, (1, 1, 96, 64, 64), torch.float32, [0], SWIN_F32),
    "swin48_in4_v2_64": ("swin48_in4_v2", True, (1, 4, 64, 64, 64), torch.float16, [0], SWIN_IN4_V2),
    "unet_c2_96": ("unet_c2", True, (2, 1, 96, 96, 96), torch.float16, [0, 1], UNET),
    "swin48_96_b25": ("swin48", True, (25, 1, 96, 96, 96), torch.float16, [0, 12, 24], SWIN),
    "unet_c2_96_b25": ("unet_c2", True, (25, 1, 96, 96, 96), torch.float16, [0, 12, 24], UNET),
}


def _run(cfg: str, monkeypatch, inject=None, shape=None, items=None):
    kind, half, in_shape, dtype, its, _ = CONFIGS[cfg]
    h = Harness(items if items is not None else its, inject)
    install(h, monkeypatch)
    net = _build(kind, half)
    x = torch.randn(shape or in_shape, generator=torch.Generator().manual_seed(0)).to(dtype).to(DEV)
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")   # the fp32-input notice of SwinUNETR
        y = net(x)
    torch.cuda.synchronize()
    return h, y, time.perf_counter() - t0


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_every_launch_matches_float64(cfg, monkeypatch):
    h, y, secs = _run(cfg, monkeypatch)
    h.report(cfg, secs)
    in_shape = CONFIGS[cfg][2]
    assert tuple(y.shape[2:]) == in_shape[2:] and bool(torch.isfinite(y).all())
    escaped = sorted({e for e, op in h.launched if op is None and e not in PREP})
    assert not escaped, f"launched outside a checked wrapper: {escaped}"
    missing = [c for c in CONFIGS[cfg][5] if c not in h.seen]
    assert not missing, f"variants never launched: {missing} (seen: {sorted(h.seen)})"
    bad = [r for r in h.rows if not r["ok"]]
    assert not bad, "\n".join(f"launch {r['id']} {r['op']} {r['what']} {r['shape']}: max {r['max']:.3e} rms {r['rms']:.3e} bound {r['tol']}"
                              for r in bad[:40])


def test_launch_check_catches_injected_faults(monkeypatch):
    """Corrupt three launches of a 64^3, N = 2 forward after the kernel ran and before the comparison; each must be reported,
    against the entry point that wrote it, and nothing may be reported before the first corruption."""
    done: dict = {}

    def inject(h, name, a, ret):
        if name == "gemm_tc" and a["mode"] == 1 and "tile" not in done:
            b = ret[0].buf.view(ret[0].N, ret[0].C // 8, -1, 8)
            b[1, :, 128:256] = b[0, :, 128:256]   # item 1's second 128-row tile replaced by item 0's
            done["tile"] = (h.launch_id, "gemm_tc")
        elif name == "window_attention_tc" and "elem" not in done:
            b = ret.buf
            b[1, 0, 0, 0, 5, 3] += 0.01 * float(b[1].float().abs().max())
            done["elem"] = (h.launch_id, "window_attention_tc")
        elif name == "conv3x3x3_tc" and "nan" not in done:
            ret[0].buf[0, 0, 1, 2, 3, 4] = float("nan")
            done["nan"] = (h.launch_id, "conv3x3x3_tc")

    h, _, _ = _run("swin48_96", monkeypatch, inject=inject, shape=(2, 1, 64, 64, 64), items=[0, 1])
    assert set(done) == {"tile", "elem", "nan"}
    for kind, (lid, op) in done.items():
        rows = [r for r in h.rows if r["id"] == lid]
        assert rows and all(r["op"] == op for r in rows)
        assert any(not r["ok"] for r in rows), (kind, rows)
    first = min(lid for lid, _ in done.values())
    early = [r for r in h.rows if r["id"] < first and not r["ok"]]
    assert not early, early
