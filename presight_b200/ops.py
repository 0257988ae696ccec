"""Autograd-aware Python wrappers over the C-ABI kernels (libpresight_b200.so).

Every function here allocates outputs with torch, passes raw device pointers + the current CUDA stream
through ctypes, and fails loudly when the library is missing or the tensors are not on a CUDA device.
There is no CPU / PyTorch fallback.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import call, host_floats, host_ints, host_ptrs, ptr, stream

ACT_NONE, ACT_RELU, ACT_SIGMOID = 0, 1, 2
PREC_TF32X3, PREC_BF16 = 0, 1


class KernelProbe:
    """Optional per-kernel timing with CUDA events on the launching stream (used by bench.py for the roofline
    line).  `with probe("name"):` brackets one launch; `summary()` returns {name: (launches, mean ms)}."""

    def __init__(self) -> None:
        self.events = {}

    def __call__(self, name: str):
        return _ProbeCtx(self, name)

    def summary(self):
        torch.cuda.synchronize()
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v) / len(v)) for k, v in self.events.items()}


class _ProbeCtx:
    def __init__(self, probe, name):
        self.probe, self.name = probe, name

    def __enter__(self):
        if self.probe is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()

    def __exit__(self, *exc):
        if self.probe is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            self.probe.events.setdefault(self.name, []).append((self.start, end))
        return False


PROBE: Optional[KernelProbe] = None


def _probe(name: str):
    return _ProbeCtx(PROBE, name)


def new_tminmax(dev) -> Tensor:
    """[+inf, -inf] built on the device (fill kernels only, so it can be captured into a CUDA graph)."""
    t = torch.full((2,), float("inf"), device=dev, dtype=torch.float32)
    t[1:].fill_(float("-inf"))
    return t


def zeros_like_many(tensors: Sequence[Tensor]) -> List[Tensor]:
    """Zero-filled fp32 buffers shaped like `tensors`, carved out of ONE allocation (one fill kernel instead of one each)."""
    sizes = [((t.numel() + 3) // 4) * 4 for t in tensors]          # keep every view 16-byte aligned
    flat = torch.zeros(sum(sizes), device=tensors[0].device, dtype=torch.float32)
    out, off = [], 0
    for t, n in zip(tensors, sizes):
        out.append(flat[off:off + t.numel()].view(t.shape))
        off += n
    return out


def _f32c(t: Tensor) -> Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# --------------------------------------------------------------------------------------------------
# kernel #1: hash encoding
# --------------------------------------------------------------------------------------------------
class _HashEncode(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x01: Tensor, table: Tensor, scalings: Tuple[float, ...], log2_T: int):
        x = _f32c(x01.detach()).view(-1, 3)
        tab = table.detach()
        assert tab.dtype == torch.float32 and tab.is_contiguous()
        L, F = len(scalings), tab.shape[1]
        P = x.shape[0]
        out = torch.empty(P, L * F, device=x.device, dtype=torch.float32)
        with _probe(f"hash_fwd_L{L}F{F}T{log2_T}"):
            call("ps_hash_fwd", ptr(x), P, ptr(tab), host_floats(scalings), L, F, log2_T, ptr(out), stream())
        ctx.save_for_backward(x, table)
        ctx.meta = (scalings, log2_T, x01.shape, x01.requires_grad)
        return out.view(*x01.shape[:-1], L * F)

    @staticmethod
    def backward(ctx, dout: Tensor):
        x, table = ctx.saved_tensors
        scalings, log2_T, xshape, need_dx = ctx.meta
        L, F = len(scalings), table.shape[1]
        P = x.shape[0]
        dout = _f32c(dout).view(P, L * F)
        dtable = torch.zeros_like(table) if ctx.needs_input_grad[1] else None
        dx = torch.zeros_like(x) if (need_dx and ctx.needs_input_grad[0]) else None
        if dtable is None and dx is None:
            return None, None, None, None
        if dtable is None:  # the kernel always scatters; give it a scratch target
            dtable = torch.zeros_like(table)
        with _probe(f"hash_bwd_L{L}F{F}T{log2_T}"):
            call("ps_hash_bwd", ptr(x), P, ptr(table.detach()), host_floats(scalings), L, F, log2_T, ptr(dout),
                 ptr(dtable), ptr(dx), stream())
        return (dx.view(xshape) if dx is not None else None), (dtable if ctx.needs_input_grad[1] else None), None, None


def hash_encode(x01: Tensor, table: Tensor, scalings: Sequence[float], log2_T: int) -> Tensor:
    """[..., 3] -> [..., L*F]; replaces HashEncoding.pytorch_fwd (encodings.py:343-384)."""
    return _HashEncode.apply(x01, table, tuple(float(s) for s in scalings), int(log2_T))


def hash_indices(x01: Tensor, scalings: Sequence[float], log2_T: int) -> Tuple[Tensor, Tensor]:
    """Parity probe: ([P,L,8] int64 rows incl. level offset, [P,L,3] offsets)."""
    x = _f32c(x01).view(-1, 3)
    P, L = x.shape[0], len(scalings)
    idx = torch.empty(P, L, 8, device=x.device, dtype=torch.int64)
    off = torch.empty(P, L, 3, device=x.device, dtype=torch.float32)
    call("ps_hash_indices", ptr(x), P, host_floats(scalings), L, int(log2_T), ptr(idx), ptr(off), stream())
    return idx, off


# --------------------------------------------------------------------------------------------------
# position prologue
# --------------------------------------------------------------------------------------------------
def normalize_positions(pos: Tensor, aabb: Sequence[float], contract: bool = True) -> Tuple[Tensor, Tensor]:
    """World positions [...,3] -> (unit-cube positions, uint8 selector [...]); no gradient
    (ingp_field.py:169-177).  `aabb` = 6 host floats (min xyz, max xyz)."""
    p = _f32c(pos.detach()).view(-1, 3)
    P = p.shape[0]
    x01 = torch.empty_like(p)
    sel = torch.empty(P, device=p.device, dtype=torch.uint8)
    call("ps_normalize_positions", ptr(p), P, host_floats(aabb), 1 if contract else 0, ptr(x01), ptr(sel), stream())
    return x01.view(pos.shape), sel.view(pos.shape[:-1])


def sample_positions(origins: Tensor, dirs: Tensor, eu_bins: Tensor) -> Tensor:
    """Frustum mid-points [N,S,3] (cameras/rays.py:49-58)."""
    N, S = eu_bins.shape[0], eu_bins.shape[1] - 1
    pos = torch.empty(N, S, 3, device=eu_bins.device, dtype=torch.float32)
    # converted copies bound to names: ptr() keeps only an address, and a copy freed before the launch may be handed to
    # the next one of the argument list
    o, d, eu = _f32c(origins), _f32c(dirs), _f32c(eu_bins)
    call("ps_sample_positions", ptr(o), ptr(d), ptr(eu), N, S, ptr(pos), stream())
    return pos


def sh4(dirs: Tensor, mapped: bool = False) -> Tensor:
    """[...,3] -> 16 SH components (math.py:27-74); no gradient.  mapped=False: raw directions, the kernel
    applies the (d+1)/2 mapping of base_field.py:136-142; mapped=True: input already mapped."""
    d = _f32c(dirs.detach()).view(-1, 3)
    out = torch.empty(d.shape[0], 16, device=d.device, dtype=torch.float32)
    call("ps_sh4", ptr(d), d.shape[0], 1 if mapped else 0, ptr(out), stream())
    return out.view(*dirs.shape[:-1], 16)


def nearest_centroid(pos: Tensor, centroids: Tensor) -> Tensor:
    """[P,3],[nf,3] -> int32 [P] (ingp_field_ms.py:97)."""
    p = _f32c(pos.detach()).view(-1, 3)
    c = _f32c(centroids)
    out = torch.empty(p.shape[0], device=p.device, dtype=torch.int32)
    call("ps_nearest_centroid", ptr(p), p.shape[0], ptr(c), c.shape[0], ptr(out), stream())
    return out


# --------------------------------------------------------------------------------------------------
# kernel #2: fused MLP, trunc_exp
# --------------------------------------------------------------------------------------------------
class _Mlp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, out_act: int, precision: int, n_layers: int, *params: Tensor):
        ws, bs = params[:n_layers], params[n_layers:]
        xs = _f32c(x.detach())
        lead = xs.shape[:-1]
        x2 = xs.view(-1, xs.shape[-1])
        dims = [x2.shape[1]] + [w.shape[0] for w in ws]
        for i, w in enumerate(ws):
            assert w.shape[1] == dims[i], f"layer {i}: weight {tuple(w.shape)} does not match input width {dims[i]}"
        y = torch.empty(x2.shape[0], dims[-1], device=x2.device, dtype=torch.float32)
        wd = [w.detach().contiguous() for w in ws]
        bd = [None if b is None else b.detach().contiguous() for b in bs]
        with _probe("mlp_fwd_" + "x".join(map(str, dims))):
            call("ps_mlp_fwd", ptr(x2), x2.shape[0], host_ptrs(wd), host_ptrs(bd), host_ints(dims), n_layers, out_act,
                 precision, ptr(y), stream())
        ctx.save_for_backward(x2, *wd, *[b for b in bd if b is not None])
        ctx.meta = (out_act, precision, n_layers, dims, [b is not None for b in bd], x.shape)
        return y.view(*lead, dims[-1])

    @staticmethod
    def backward(ctx, dy: Tensor):
        out_act, precision, n_layers, dims, has_b, xshape = ctx.meta
        saved = ctx.saved_tensors
        x2, wd = saved[0], list(saved[1:1 + n_layers])
        rest = list(saved[1 + n_layers:])
        bd = [rest.pop(0) if hb else None for hb in has_b]
        dy2 = _f32c(dy).view(-1, dims[-1])
        dx = torch.empty_like(x2) if ctx.needs_input_grad[0] else None
        zs = zeros_like_many([*wd, *[b for b in bd if b is not None]])      # one fill kernel for all gradients
        dW, zb = zs[:n_layers], zs[n_layers:]
        db = [None if b is None else zb.pop(0) for b in bd]
        with _probe("mlp_bwd_" + "x".join(map(str, dims))):
            call("ps_mlp_bwd", ptr(x2), None, ptr(dy2), x2.shape[0], host_ptrs(wd), host_ptrs(bd), host_ints(dims),
                 n_layers, out_act, precision, ptr(dx), host_ptrs(dW), host_ptrs(db), stream())
        return (None if dx is None else dx.view(xshape), None, None, None, *dW, *db)


class _MlpSelect(torch.autograd.Function):
    """y[n] = MLP_{sf[n]}(x[n]) for nf networks of one shape: every network runs on all rows (the per-ray sky networks are
    tiny) and each row keeps its own network's output — one autograd node, one gather, instead of nf nodes and 4 nf
    element-wise launches.  params: the networks' weights, then their biases, network by network."""

    @staticmethod
    def forward(ctx, x: Tensor, sf: Tensor, out_act: int, precision: int, n_layers: int, nf: int, *params: Tensor):
        xs = _f32c(x.detach())
        x2 = xs.view(-1, xs.shape[-1])
        N = x2.shape[0]
        per = 2 * n_layers
        nets = [([p.detach().contiguous() for p in params[k * per:k * per + n_layers]],
                 [p.detach().contiguous() for p in params[k * per + n_layers:(k + 1) * per]]) for k in range(nf)]
        dims = [x2.shape[1]] + [w.shape[0] for w in nets[0][0]]
        Y = torch.empty(nf, N, dims[-1], device=x2.device, dtype=torch.float32)
        hd, st = host_ints(dims), stream()
        with _probe("mlp_fwd_" + "x".join(map(str, dims))):
            for k, (ws, bs) in enumerate(nets):
                call("ps_mlp_fwd", ptr(x2), N, host_ptrs(ws), host_ptrs(bs), hd, n_layers, out_act, precision,
                     ptr(Y[k]), st)
        idx = sf.view(1, N, 1).expand(1, N, dims[-1])
        y = Y.gather(0, idx).squeeze(0)
        ctx.save_for_backward(x2, sf, *params)
        ctx.meta = (out_act, precision, n_layers, nf, dims, x.shape)
        return y.view(*x.shape[:-1], dims[-1])

    @staticmethod
    def backward(ctx, dy: Tensor):
        out_act, precision, n_layers, nf, dims, xshape = ctx.meta
        x2, sf, *params = ctx.saved_tensors
        N, per = x2.shape[0], 2 * n_layers
        nets = [([p.detach().contiguous() for p in params[k * per:k * per + n_layers]],
                 [p.detach().contiguous() for p in params[k * per + n_layers:(k + 1) * per]]) for k in range(nf)]
        idx = sf.view(1, N, 1).expand(1, N, dims[-1])
        dY = torch.zeros(nf, N, dims[-1], device=x2.device, dtype=torch.float32)
        dY.scatter_(0, idx, _f32c(dy).view(1, N, dims[-1]))              # rows of other networks' rays stay zero
        zs = zeros_like_many([t for ws, bs in nets for t in (*ws, *bs)])     # one fill for every gradient
        need_dx = ctx.needs_input_grad[0]
        dX = torch.empty(nf, N, dims[0], device=x2.device, dtype=torch.float32) if need_dx else None
        hd, st = host_ints(dims), stream()
        with _probe("mlp_bwd_" + "x".join(map(str, dims))):
            for k, (ws, bs) in enumerate(nets):
                g = zs[k * per:(k + 1) * per]
                call("ps_mlp_bwd", ptr(x2), None, ptr(dY[k]), N, host_ptrs(ws), host_ptrs(bs), hd, n_layers, out_act, precision,
                     None if dX is None else ptr(dX[k]), host_ptrs(g[:n_layers]), host_ptrs(g[n_layers:]), st)
        dx = None
        if need_dx:
            dx = dX.gather(0, sf.view(1, N, 1).expand(1, N, dims[0])).squeeze(0).view(xshape)
        return (dx, None, None, None, None, None, *zs)


def mlp_select(x: Tensor, sf: Tensor, nets: Sequence[Tuple[Sequence[Tensor], Sequence[Tensor]]], out_act: int = ACT_NONE,
               precision: int = PREC_BF16) -> Tensor:
    """Row n through network sf[n] (all networks of one shape, biases present): see _MlpSelect."""
    n_layers = len(nets[0][0])
    flat = [t for ws, bs in nets for t in (*ws, *bs)]
    return _MlpSelect.apply(x, sf, int(out_act), int(precision), n_layers, len(nets), *flat)


def mlp(x: Tensor, weights: Sequence[Tensor], biases: Sequence[Optional[Tensor]], out_act: int = ACT_NONE,
        precision: int = PREC_BF16) -> Tensor:
    """Linear+ReLU stack with optional output activation (mlp.py:157-174) in ONE kernel per direction."""
    return _Mlp.apply(x, int(out_act), int(precision), len(weights), *weights, *biases)


class _TruncExp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, sel: Optional[Tensor]):
        xs = _f32c(x.detach())
        y = torch.empty_like(xs)
        s = None if sel is None else sel.contiguous()
        call("ps_trunc_exp_fwd", ptr(xs), ptr(s), xs.numel(), 1, ptr(y), stream())
        ctx.save_for_backward(xs)
        ctx.sel = s
        return y

    @staticmethod
    def backward(ctx, dy: Tensor):
        (xs,) = ctx.saved_tensors
        dx = torch.empty_like(xs)
        call("ps_trunc_exp_bwd", ptr(xs), ptr(ctx.sel), ptr(_f32c(dy)), xs.numel(), 1, ptr(dx), 1, stream())
        return dx, None


def trunc_exp(x: Tensor, selector: Optional[Tensor] = None) -> Tensor:
    """exp(x) * selector with the clamped backward of activations.py:28-41 (selector: uint8, same numel)."""
    return _TruncExp.apply(x, selector)


# --------------------------------------------------------------------------------------------------
# kernel #3: samplers
# --------------------------------------------------------------------------------------------------
def spaced_bins(nears: Tensor, fars: Tensor, num_samples: int, thr: float, t_rand: Optional[Tensor]):
    """-> (spacing bins [N,S+1], euclidean bins [N,S+1]); ray_samplers.py:98-128 with PreSight's spacing."""
    n = _f32c(nears).view(-1)
    f = _f32c(fars).view(-1)
    N = n.shape[0]
    lin = torch.linspace(0.0, 1.0, num_samples + 1, device=n.device)
    sp = torch.empty(N, num_samples + 1, device=n.device, dtype=torch.float32)
    eu = torch.empty_like(sp)
    tr = None if t_rand is None else _f32c(t_rand).view(-1)
    call("ps_spaced_bins", ptr(n), ptr(f), ptr(lin), ptr(tr), N, num_samples, float(thr), ptr(sp), ptr(eu), stream())
    return sp, eu


def pdf_resample(weights: Tensor, sp_in: Tensor, num_samples: int, rand: Optional[Tensor], nears: Tensor, fars: Tensor,
                 thr: float, padding: float = 0.01, eps: float = 1e-5, anneal: float = 1.0, probes: bool = False):
    """Inverse-CDF resampling (ray_samplers.py:305-362).  weights [N,S_in], sp_in [N,S_in+1].
    -> (sp_out, eu_out[, inds, cdf, u])."""
    w = _f32c(weights.detach())
    N, S_in = w.shape
    nb = num_samples + 1
    dev = w.device
    u_base = torch.linspace(0.0, 1.0 - (1.0 / nb), steps=nb, device=dev)
    sp_out = torch.empty(N, nb, device=dev, dtype=torch.float32)
    eu_out = torch.empty_like(sp_out)
    inds = torch.empty(N, nb, device=dev, dtype=torch.int64) if probes else None
    cdf = torch.empty(N, S_in + 1, device=dev, dtype=torch.float32) if probes else None
    u = torch.empty(N, nb, device=dev, dtype=torch.float32) if probes else None
    r = None if rand is None else _f32c(rand).view(-1)
    sp, nr, fr = _f32c(sp_in.detach()), _f32c(nears).view(-1), _f32c(fars).view(-1)     # alive until the launch
    call("ps_pdf_resample", ptr(w), ptr(sp), ptr(u_base), ptr(r), ptr(nr), ptr(fr), N, S_in, num_samples,
         float(padding), float(eps), float(anneal), float(thr), ptr(sp_out), ptr(eu_out), ptr(inds), ptr(cdf), ptr(u), stream())
    return (sp_out, eu_out, inds, cdf, u) if probes else (sp_out, eu_out)


def searchsorted_right(cdf: Tensor, u: Tensor) -> Tensor:
    c, v = _f32c(cdf), _f32c(u)
    out = torch.empty(v.shape, device=v.device, dtype=torch.int64)
    call("ps_searchsorted_right", ptr(c), ptr(v), c.shape[0], c.shape[1], v.shape[1], ptr(out), stream())
    return out


# --------------------------------------------------------------------------------------------------
# kernel #4: compositing
# --------------------------------------------------------------------------------------------------
class _Weights(torch.autograd.Function):
    @staticmethod
    def forward(ctx, deltas: Tensor, density: Tensor):
        d, s = _f32c(deltas.detach()), _f32c(density.detach())
        N, S = d.shape[0], d.shape[1]
        w = torch.empty_like(s)
        call("ps_weights_fwd", ptr(d), ptr(s), N, S, ptr(w), stream())
        ctx.save_for_backward(d, s)
        return w

    @staticmethod
    def backward(ctx, dw: Tensor):
        d, s = ctx.saved_tensors
        ds = torch.empty_like(s)
        call("ps_weights_bwd", ptr(d), ptr(s), ptr(_f32c(dw)), d.shape[0], d.shape[1], ptr(ds), stream())
        return None, ds


def get_weights(deltas: Tensor, density: Tensor) -> Tensor:
    """[N,S,1] x [N,S,1] -> [N,S,1] (cameras/rays.py:128-150)."""
    return _Weights.apply(deltas, density)


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(ctx, weights: Tensor, values: Optional[Tensor]):
        w = _f32c(weights.detach())
        N, S = w.shape[0], w.shape[1]
        v = None if values is None else _f32c(values.detach())
        C = 1 if v is None else v.shape[-1]
        out = torch.empty(N, C, device=w.device, dtype=torch.float32)
        call("ps_render_fwd", ptr(w), ptr(v), N, S, C, ptr(out), stream())
        ctx.save_for_backward(w, *(() if v is None else (v,)))
        ctx.has_v = v is not None
        return out

    @staticmethod
    def backward(ctx, dout: Tensor):
        w = ctx.saved_tensors[0]
        v = ctx.saved_tensors[1] if ctx.has_v else None
        N, S = w.shape[0], w.shape[1]
        C = 1 if v is None else v.shape[-1]
        dw = torch.zeros_like(w)
        dv = torch.empty_like(v) if (v is not None and ctx.needs_input_grad[1]) else None
        call("ps_render_bwd", ptr(w), ptr(v), ptr(_f32c(dout)), N, S, C, ptr(dw), ptr(dv), stream())
        return dw, dv


def render(weights: Tensor, values: Optional[Tensor]) -> Tensor:
    """sum_s w[n,s] * v[n,s,:] -> [N,C]; values=None gives the accumulation (renderers.py:102-103,313)."""
    return _Render.apply(weights, values)


def depth_threshold(weights: Tensor, eu_bins: Tensor, threshold: float = 0.5) -> Tuple[Tensor, Tensor]:
    """-> (depth [N,1], index [N,1] int64); renderers.py:352-362."""
    w = _f32c(weights.detach())
    N, S = w.shape[0], w.shape[1]
    depth = torch.empty(N, 1, device=w.device, dtype=torch.float32)
    index = torch.empty(N, 1, device=w.device, dtype=torch.int64)
    call("ps_depth_threshold", ptr(w), ptr(_f32c(eu_bins)), N, S, float(threshold), ptr(depth), ptr(index), stream())
    return depth, index


class _Composite(torch.autograd.Function):
    """One-pass compositing: weights, rgb, accumulation, expected depth (unclipped), threshold depth, semantics."""

    @staticmethod
    def forward(ctx, eu_bins: Tensor, density: Tensor, rgb: Optional[Tensor], sem: Optional[Tensor], threshold: float):
        b, s = _f32c(eu_bins.detach()), _f32c(density.detach())
        N, S = s.shape[0], s.shape[1]
        dev = s.device
        r = None if rgb is None else _f32c(rgb.detach())
        m = None if sem is None else _f32c(sem.detach())
        C = 0 if m is None else m.shape[-1]
        w = torch.empty(N, S, device=dev, dtype=torch.float32)
        rgb_out = torch.empty(N, 3, device=dev, dtype=torch.float32) if r is not None else None
        acc = torch.empty(N, 1, device=dev, dtype=torch.float32)
        dexp = torch.empty(N, 1, device=dev, dtype=torch.float32)
        dthr = torch.empty(N, 1, device=dev, dtype=torch.float32)
        sem_out = torch.empty(N, C, device=dev, dtype=torch.float32) if m is not None else None
        tmm = new_tminmax(dev)
        call("ps_composite_fwd", ptr(b), ptr(s), ptr(r), ptr(m), N, S, C, float(threshold), ptr(w), ptr(rgb_out),
             ptr(acc), ptr(dexp), ptr(dthr), ptr(sem_out), ptr(tmm), stream())
        ctx.save_for_backward(b, s, acc, dexp, *(t for t in (r, m) if t is not None))
        ctx.flags = (r is not None, m is not None, C)
        ctx.mark_non_differentiable(dthr, tmm)
        outs = (w, rgb_out if rgb_out is not None else torch.empty(0, device=dev), acc, dexp, dthr,
                sem_out if sem_out is not None else torch.empty(0, device=dev), tmm)
        return outs

    @staticmethod
    def backward(ctx, dw, drgb, dacc, ddexp, _dthr, dsem, _dtmm):
        has_rgb, has_sem, C = ctx.flags
        saved = list(ctx.saved_tensors)
        b, s, acc, dexp = saved[:4]
        rest = saved[4:]
        r = rest.pop(0) if has_rgb else None
        m = rest.pop(0) if has_sem else None
        N, S = s.shape[0], s.shape[1]
        d_density = torch.empty_like(s)
        d_rgb = torch.empty_like(r) if (r is not None and ctx.needs_input_grad[2]) else None
        d_sem = torch.empty_like(m) if (m is not None and ctx.needs_input_grad[3]) else None

        def opt(t):
            return None if t is None else _f32c(t)
        # converted upstream gradients bound to names: alive until the launch (see sample_positions)
        g = [opt(dw), opt(drgb) if has_rgb else None, opt(dacc), opt(ddexp), opt(dsem) if has_sem else None]
        call("ps_composite_bwd", ptr(b), ptr(s), ptr(r), ptr(m), None, ptr(acc), ptr(dexp), N, S, C, *map(ptr, g),
             ptr(d_density), ptr(d_rgb), ptr(d_sem), stream())
        return None, d_density, d_rgb, d_sem, None


def composite(eu_bins: Tensor, density: Tensor, rgb: Optional[Tensor], sem: Optional[Tensor], threshold: float = 0.5):
    """eu_bins [N,S+1], density [N,S], rgb [N,S,3], sem [N,S,C] ->
    (weights [N,S], rgb [N,3], acc [N,1], depth_expected_unclipped [N,1], depth_threshold [N,1], sem [N,C],
     tminmax [2])."""
    return _Composite.apply(eu_bins, density, rgb, sem, float(threshold))


# --------------------------------------------------------------------------------------------------
# loss stack: proposal (interlevel) loss
# --------------------------------------------------------------------------------------------------
# Cross-stream hand-off of gradients: a producer may publish "this gradient tensor is complete at event E" so that a
# consumer running its backward on a side stream (presight_b200/fused.py: the proposal levels' backward overlaps the
# final level's hash scatter) waits for E instead of for everything queued on the main stream.
#
# The hand-off is keyed by an explicit token, not by an address: the consumer's forward (`fused.prop_level_weights`)
# creates a key and tags its output tensor with it (`_ps_grad_key`); a loss Function that receives that tensor remembers
# the key and publishes under it in its backward; the consumer's backward pops ITS key and checks that the gradient it was
# handed is the very tensor that was published (same address, shape and version counter — autograd's in-place
# accumulation of a second consumer's gradient bumps the version, a summed gradient has another address).  Anything
# else — no key, no entry, a mismatch — means "no hand-off": the consumer stays on the main stream, which is always
# correct.  Entries of one step never survive into the next (`clear_grad_events`, called at the start of every forward).
_GRAD_EVENTS = {}
_GRAD_KEY_COUNTER = [0]


def new_grad_key() -> int:
    _GRAD_KEY_COUNTER[0] += 1
    return _GRAD_KEY_COUNTER[0]


def clear_grad_events() -> None:
    _GRAD_EVENTS.clear()


def publish_grad_event(t: Tensor, key) -> None:
    if key is None:
        return
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream())
    _GRAD_EVENTS[key] = (ev, t.data_ptr(), tuple(t.shape), t._version)


def pop_grad_event(t: Tensor, key):
    entry = _GRAD_EVENTS.pop(key, None) if key is not None else None
    if entry is None:
        return None
    ev, addr, shape, version = entry
    if t.data_ptr() != addr or tuple(t.shape) != shape or t._version != version:
        return None
    return ev


_SIDE_STREAMS = {}


def side_stream(device) -> "torch.cuda.Stream":
    """The device's cached side stream (created on first use)."""
    key = torch.device(device).index
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


class _InterlevelLoss(torch.autograd.Function):
    """mean(lossfun_outer(c, w, t_env, w_env)) (model_components/losses.py:80-126) with the gradient w.r.t. the
    proposal weights produced in the same kernel; c and w are constants (the reference detaches them)."""

    @staticmethod
    def forward(ctx, c, w, t_env, w_env):
        c, w, t_env, we = _f32c(c.detach()), _f32c(w.detach()), _f32c(t_env.detach()), _f32c(w_env.detach())
        N, S = w.shape[0], w.shape[1]
        Sp = we.shape[1]
        loss = torch.zeros(1, device=w.device, dtype=torch.float32)
        need = ctx.needs_input_grad[3]
        grad = torch.empty_like(we) if need else None
        with _probe("interlevel_loss"):
            call("ps_interlevel_loss", ptr(c), ptr(w), ptr(t_env), ptr(we), N, S, Sp, ptr(loss), ptr(grad), stream())
        ctx.scale = 1.0 / float(N * S)
        ctx.grad_key = getattr(w_env, "_ps_grad_key", None)
        ctx.wshape = w_env.shape
        if need:
            ctx.save_for_backward(grad)
        return loss[0] * ctx.scale

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        out = (grad * (g * ctx.scale)).view(ctx.wshape)
        publish_grad_event(out, ctx.grad_key)
        return None, None, None, out


class _ZaaInterlevelLoss(torch.autograd.Function):
    """One proposal level's term of z_anti_anliasing_interlevel_loss (model_components/PreSight/losses.py:166-206) with
    the gradient w.r.t. the proposal weights produced in the same kernel; c and w are constants (detached there)."""

    @staticmethod
    def forward(ctx, c, w, t_env, w_env, pulse_width):
        c, w, t_env, we = _f32c(c.detach()), _f32c(w.detach()), _f32c(t_env.detach()), _f32c(w_env.detach())
        N, S = w.shape[0], w.shape[1]
        Sp = we.shape[1]
        assert c.shape == (N, S + 1) and t_env.shape == (N, Sp + 1) and we.numel() == N * Sp
        loss = torch.zeros(1, device=w.device, dtype=torch.float32)
        need = ctx.needs_input_grad[3]
        grad = torch.empty(N, Sp, device=w.device, dtype=torch.float32) if need else None
        with _probe("zaa_interlevel_loss"):
            call("ps_zaa_interlevel_loss", ptr(c), ptr(w), N, S, ptr(t_env), ptr(we.view(N, Sp)), Sp, float(pulse_width),
                 ptr(loss), ptr(grad), stream())
        ctx.scale = 1.0 / float(N * Sp)
        ctx.wshape = w_env.shape
        ctx.grad_key = getattr(w_env, "_ps_grad_key", None)
        if need:
            ctx.save_for_backward(grad)
        return loss[0] * ctx.scale

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        out = (grad * (g * ctx.scale)).view(ctx.wshape)
        publish_grad_event(out, ctx.grad_key)
        return None, None, None, out, None


def zaa_interlevel_loss_level(c: Tensor, w: Tensor, t_env: Tensor, w_env: Tensor, pulse_width: float) -> Tensor:
    """c [N,S+1], w [N,S] final level (constants); t_env [N,Sp+1], w_env [N,Sp] or [N,Sp,1] -> scalar."""
    return _ZaaInterlevelLoss.apply(c, w, t_env, w_env, float(pulse_width))


class _DistortionLoss(torch.autograd.Function):
    """mean over rays of lossfun_distortion(c, w) (model_components/losses.py:130-149) with the gradient w.r.t. the
    weights produced in the same kernel; c (bin edges) is a constant."""

    @staticmethod
    def forward(ctx, c, w):
        cc, wc = _f32c(c.detach()), _f32c(w.detach())
        N, S = wc.shape[0], wc.shape[1]
        assert cc.shape == (N, S + 1) and wc.numel() == N * S, "distortion_loss: c must be [N,S+1], w [N,S] or [N,S,1]"
        loss = torch.zeros(1, device=wc.device, dtype=torch.float32)
        need = ctx.needs_input_grad[1]
        grad = torch.empty(N, S, device=wc.device, dtype=torch.float32) if need else None
        with _probe("distortion_loss"):
            call("ps_distortion_loss", ptr(cc), ptr(wc.view(N, S)), N, S, ptr(loss), ptr(grad), stream())
        ctx.scale = 1.0 / float(max(N, 1))
        ctx.wshape = w.shape
        if need:
            ctx.save_for_backward(grad)
        return loss[0] * ctx.scale

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return None, (grad * (g * ctx.scale)).view(ctx.wshape)


def distortion_loss(c: Tensor, w: Tensor) -> Tensor:
    """c [N,S+1] spacing-domain bin edges, w [N,S] or [N,S,1] weights of the final level -> scalar."""
    return _DistortionLoss.apply(c, w)


def interlevel_loss_level(c: Tensor, w: Tensor, t_env: Tensor, w_env: Tensor) -> Tensor:
    """One proposal level's term of interlevel_loss: c [N,S+1], w [N,S], t_env [N,Sp+1], w_env [N,Sp] or [N,Sp,1]
    (the gradient comes back in w_env's shape) -> scalar."""
    return _InterlevelLoss.apply(c, w, t_env, w_env)


# --------------------------------------------------------------------------------------------------
# loss stack: model epilogue (sky blending) and the rendered-output loss terms, one kernel per direction
# --------------------------------------------------------------------------------------------------
class _SkyBlend(torch.autograd.Function):
    """nerfacto_nusc_ms.py:512-532: (rgb_f [N,3], acc_raw [N,1], sem_f [N,C]|None, sky_rgb|None, sky_sem|None) ->
    (rgb, accumulation [N,1], semantics|None)."""

    @staticmethod
    def forward(ctx, rgb_f, acc_raw, sem_f, sky_rgb, sky_sem, clamp_rgb):
        r, a = _f32c(rgb_f.detach()), _f32c(acc_raw.detach())
        s = None if sem_f is None else _f32c(sem_f.detach())
        kr = None if sky_rgb is None else _f32c(sky_rgb.detach())
        ks = None if (sky_sem is None or s is None) else _f32c(sky_sem.detach())
        N = r.shape[0]
        C = 0 if s is None else s.shape[1]
        rgb, acc = torch.empty_like(r), torch.empty_like(a)
        sem = None if s is None else torch.empty_like(s)
        call("ps_sky_blend_fwd", ptr(r), ptr(a), ptr(s), ptr(kr), ptr(ks), N, C, 1 if clamp_rgb else 0, ptr(rgb), ptr(acc),
             ptr(sem), stream())
        ctx.save_for_backward(r, a, kr, ks)
        ctx.meta = (N, C, bool(clamp_rgb), s is not None)
        ctx.set_materialize_grads(False)
        if sem is None:
            sem = torch.empty(0, device=r.device)
            ctx.mark_non_differentiable(sem)
        return rgb, acc, sem

    @staticmethod
    def backward(ctx, d_rgb, d_acc, d_sem):
        N, C, clamp_rgb, has_sem = ctx.meta
        r, a, kr, ks = ctx.saved_tensors
        dr = None if d_rgb is None else _f32c(d_rgb)
        da = None if d_acc is None else _f32c(d_acc)
        ds = None if (d_sem is None or not has_sem) else _f32c(d_sem)
        need = ctx.needs_input_grad
        d_acc_raw = torch.empty_like(a)
        d_rgb_f = torch.empty_like(r) if (clamp_rgb and need[0]) else None
        d_kr = torch.empty_like(kr) if (kr is not None and need[3]) else None
        d_ks = torch.empty_like(ks) if (ks is not None and need[4]) else None
        call("ps_sky_blend_bwd", ptr(r), ptr(a), ptr(kr), ptr(ks), ptr(dr), ptr(da), ptr(ds), N, C, 1 if clamp_rgb else 0,
             ptr(d_rgb_f), ptr(d_acc_raw), ptr(d_kr), ptr(d_ks), stream())
        g_rgb_f = d_rgb_f if clamp_rgb else dr          # identity paths hand the upstream gradient through
        return g_rgb_f, d_acc_raw, ds, d_kr, d_ks, None


def sky_blend(rgb_f: Tensor, acc_raw: Tensor, sem_f: Optional[Tensor], sky_rgb: Optional[Tensor],
              sky_sem: Optional[Tensor], clamp_rgb: bool = False):
    """-> (rgb [N,3], accumulation [N,1], semantics [N,C] or None)."""
    rgb, acc, sem = _SkyBlend.apply(rgb_f, acc_raw, sem_f, sky_rgb, sky_sem, clamp_rgb)
    return rgb, acc, (None if sem_f is None else sem)


class _RenderLosses(torch.autograd.Function):
    """[rgb MSE, sky BCE, semantic MSE] (nerfacto_nusc_ms.py:560-576, PreSight/losses.py:106-125) and their gradients
    in one kernel; absent terms are zero."""

    @staticmethod
    def forward(ctx, rgb, gt_rgb, acc, sky_mask, sem, gt_sem, eps):
        ref = rgb if rgb is not None else (acc if acc is not None else sem)
        c = lambda t: None if t is None else _f32c(t.detach())
        r, gr, a, km, s, gs = c(rgb), c(gt_rgb), c(acc), c(sky_mask), c(sem), c(gt_sem)
        N = ref.shape[0]
        C = 0 if s is None else s.shape[1]
        need = ctx.needs_input_grad
        losses = torch.zeros(3, device=ref.device, dtype=torch.float32)
        g_r = torch.empty_like(r) if (r is not None and need[0]) else None
        g_a = torch.empty_like(a) if (a is not None and need[2]) else None
        g_s = torch.empty_like(s) if (s is not None and need[4]) else None
        with _probe("render_losses"):
            call("ps_render_losses", ptr(r), ptr(gr), ptr(a), ptr(km), ptr(s), ptr(gs), N, C, float(eps), ptr(losses),
                 ptr(g_r), ptr(g_a), ptr(g_s), stream())
        ctx.has = tuple(t is not None for t in (g_r, g_a, g_s))
        ctx.save_for_backward(*(t for t in (g_r, g_a, g_s) if t is not None))
        return losses

    @staticmethod
    def backward(ctx, g):
        rest = list(ctx.saved_tensors)
        g_r, g_a, g_s = (rest.pop(0) if h else None for h in ctx.has)
        return (None if g_r is None else g_r * g[0], None, None if g_a is None else g_a * g[1], None,
                None if g_s is None else g_s * g[2], None, None)


def render_losses(rgb: Optional[Tensor], gt_rgb: Optional[Tensor], acc: Optional[Tensor], sky_mask: Optional[Tensor],
                  sem: Optional[Tensor], gt_sem: Optional[Tensor], eps: float = 1e-7) -> Tensor:
    """-> [3] = (rgb_loss, sky_loss, semantic_loss), each a mean; pass None pairs to skip a term."""
    return _RenderLosses.apply(rgb, gt_rgb, acc, sky_mask, sem, gt_sem, eps)


class _DepthLosses(torch.autograd.Function):
    """[expected-depth loss, line-of-sight loss] (model_components/PreSight/losses.py:28-103 as called from
    nerfacto_nusc_ms.py:577-629): means over the rays passing the depth mask, with both gradients produced by the same
    kernel.  The number of masked rays stays on the device (no host sync); an empty mask gives NaN like torch's mean."""

    @staticmethod
    def forward(ctx, weights, expected_depth, eu_bins, steps_m, target_m, sky_mask, pose_scale, sigma, upper_bound, mode):
        c = lambda t: None if t is None else _f32c(t.detach())
        w, e, b, st, tg, sk = c(weights), c(expected_depth), c(eu_bins), c(steps_m), c(target_m), c(sky_mask)
        N = tg.numel()
        S = 0 if w is None else w.numel() // max(N, 1)
        if w is not None:
            assert w.numel() == N * S and (b is None or b.shape == (N, S + 1)) and (st is None or st.numel() == N * S)
        sums = torch.zeros(3, device=tg.device, dtype=torch.float32)
        g_e = torch.empty(N, device=tg.device, dtype=torch.float32) if (e is not None and ctx.needs_input_grad[1]) else None
        g_w = torch.empty(N, S, device=tg.device, dtype=torch.float32) if (w is not None and ctx.needs_input_grad[0]) else None
        scale_dev = _f32c(pose_scale.detach()).reshape(-1)[:1] if torch.is_tensor(pose_scale) else None
        with _probe("depth_losses"):
            call("ps_depth_losses", ptr(w), ptr(b), ptr(st), ptr(e), ptr(tg), ptr(sk), N, S,
                 1.0 if scale_dev is not None else float(pose_scale), ptr(scale_dev), float(sigma), float(upper_bound),
                 int(mode), ptr(sums), ptr(g_e), ptr(g_w), stream())
        inv = 1.0 / sums[0]
        ctx.save_for_backward(inv, *(t for t in (g_e, g_w) if t is not None))
        ctx.has = (g_e is not None, g_w is not None)
        ctx.shapes = (None if weights is None else weights.shape, None if expected_depth is None else expected_depth.shape)
        return sums[1:] * inv

    @staticmethod
    def backward(ctx, g):
        inv, *rest = ctx.saved_tensors
        g_e = rest.pop(0) if ctx.has[0] else None
        g_w = rest.pop(0) if ctx.has[1] else None
        d_w = None if g_w is None else (g_w * (g[1] * inv)).view(ctx.shapes[0])
        d_e = None if g_e is None else (g_e * (g[0] * inv)).view(ctx.shapes[1])
        return d_w, d_e, None, None, None, None, None, None, None, None


def depth_losses(weights: Optional[Tensor], expected_depth: Optional[Tensor], target_depth_m: Tensor,
                 sky_mask: Optional[Tensor], pose_scale, sigma: float, upper_bound: float, inverse: bool = False,
                 eu_bins: Optional[Tensor] = None, steps_m: Optional[Tensor] = None) -> Tensor:
    """-> [2] = (expected-depth loss, line-of-sight loss) before their multipliers.  weights [N,S(,1)] final-level
    weights with their bin edges `eu_bins` [N,S+1] (scene units) or mid-points `steps_m` [N,S(,1)] (metres);
    expected_depth [N(,1)] rendered depth in scene units; target_depth_m [N(,1)] metres; sky_mask [N(,1)] or None;
    pose_scale: a float, or a CUDA tensor whose first element is read on the device (no host sync)."""
    return _DepthLosses.apply(weights, expected_depth, eu_bins, steps_m, target_depth_m, sky_mask,
                              pose_scale if torch.is_tensor(pose_scale) else float(pose_scale), float(sigma), float(upper_bound), 1 if inverse else 0)


def launch_count() -> int:
    return _lib.launch_count()
