"""Level-fused fast paths: one autograd node per sampling level, a fixed chain of libpresight_b200 kernels inside.

The drop-in modules (`HashEncoding`, `MLP`, `get_weights`, renderers) compose through torch autograd like the
reference does; these two Functions are what the model driver uses when a level is served by a single sub-field:

  proposal level (ray_samplers.py:600-609):   ray_points -> hash_fwd -> mlp(+density epilogue) -> weights
  field level (nerfacto_nusc_ms.py:497-530):  ray_points -> hash_fwd -> base mlp(+density) -> semantic head ->
                                              sh4 -> colour head -> one-pass compositing

No torch.cat / split / expand copies: the heads read column windows of the base MLP's output `h` and per-ray vectors
(SH of the view direction, appearance embedding) through segmented row descriptors, and their input gradients are
written straight into the matching windows of one `dh` buffer (the appearance gradient is reduced per ray in-kernel).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import ops
from ._lib import call, host_floats, host_ints, host_ptrs, host_segments, ptr, stream

_f32c = ops._f32c
OVERLAP_PROP_BWD = True


def set_overlap_prop_bwd(on: bool) -> bool:
    """Scheduling policy of the proposal levels' backward: True = early, on a side stream beside the final level's
    kernels (single GPU); False = on the main stream behind them (what a data-parallel run wants, so that the main
    table's all-reduce has compute to hide under).  The caller decides (bench.py does, per world size); nothing in
    the library flips it behind the caller's back.  -> the previous value."""
    global OVERLAP_PROP_BWD
    prev, OVERLAP_PROP_BWD = OVERLAP_PROP_BWD, bool(on)
    return prev

# Partial-gradient sinks (data-parallel training, presight_b200/parallel.py): the main hash table is ONE parameter of 512 MiB
# whose gradient is complete only when the last level has been scattered — the last kernel of the backward.  A sink registered
# for the table receives every level group's rows as soon as that group's scatter has been launched (called with the scatter's
# stream current, so a collective issued inside it is ordered behind exactly that kernel) and can start reducing them while
# the remaining levels and the proposal networks are still being differentiated.
# device index -> [event recorded where the step's field backward kernel becomes launchable, proposal backwards launched
# since] (autograd runs the field level's backward first).  The first proposal backward of a step starts at once; later ones
# wait for that event, so they queue behind the field kernel without waiting for its end (two kernels launched microseconds
# apart on different streams would otherwise race for the SMs).
_FIELD_BWD_ORDER = {}

_PARTIAL_SINKS = {}          # table.data_ptr() -> (callable(dtable, row_lo, row_hi), level groups [(l0, l1), ...], alloc)


def register_partial_grad_sink(table: Tensor, fn, level_groups, alloc=None) -> None:
    """`alloc` (optional): () -> the zero-filled gradient buffer to scatter into (called with the scatter's stream current),
    for exchanges that need the gradient in memory of their own (peer_exchange.py); default torch.zeros_like(table)."""
    _PARTIAL_SINKS[table.data_ptr()] = (fn, [tuple(g) for g in level_groups], alloc)


def unregister_partial_grad_sink(table: Tensor) -> None:
    _PARTIAL_SINKS.pop(table.data_ptr(), None)


@dataclass(frozen=True)
class GridMeta:
    scalings: Tuple[float, ...]
    log2_T: int
    F: int

    @property
    def L(self) -> int:
        return len(self.scalings)

    @property
    def level_major(self) -> bool:
        """Store features [L][P][F] when a thread's levels-per-thread x F floats would not fill a 32-byte sector of
        the row-major [P][L*F] layout (C2 main grid: 1 level x 2 floats per thread); small grids keep row-major."""
        from ._lib import hash_levels_per_thread
        return hash_levels_per_thread(self.L, self.F, self.log2_T) * self.F < 8


@dataclass(frozen=True)
class MlpMeta:
    dims: Tuple[int, ...]
    out_act: int

    @property
    def n_layers(self) -> int:
        return len(self.dims) - 1


def _mlp_fwd(segs, P, ws, bs, meta: MlpMeta, prec, y, sel=None, density_out=None, name="mlp"):
    with ops._probe(f"mlp_fwd_{name}"):
        call("ps_mlp_fwd_ex", host_segments(segs), len(segs), P, host_ptrs(ws), host_ptrs(bs), host_ints(meta.dims),
             meta.n_layers, meta.out_act, prec, ptr(y), ptr(sel), ptr(density_out), stream())


def _mlp_bwd(segs, dy, P, ws, bs, meta: MlpMeta, prec, dW, db, sel=None, d_density=None, name="mlp"):
    with ops._probe(f"mlp_bwd_{name}"):
        call("ps_mlp_bwd_ex", host_segments(segs), len(segs), ptr(dy), P, host_ptrs(ws), host_ptrs(bs),
             host_ints(meta.dims), meta.n_layers, meta.out_act, prec, host_ptrs(dW), host_ptrs(db), ptr(sel),
             ptr(d_density), stream())


def _ray_points(origins, dirs, eu, aabb, contract):
    N, S = eu.shape[0], eu.shape[1] - 1
    x01 = torch.empty(N * S, 3, device=eu.device, dtype=torch.float32)
    sel = torch.empty(N * S, device=eu.device, dtype=torch.uint8)
    call("ps_ray_points", ptr(origins), ptr(dirs), ptr(eu), N, S, host_floats(aabb), 1 if contract else 0, ptr(x01),
         ptr(sel), stream())
    return x01, sel


def _hash_fwd(x01, table, g: GridMeta, level_major: Optional[bool] = None):
    """-> features as a flat tensor of P*L*F floats: level-major [L][P][F] (ps_hash_fwd_lm) when `level_major`
    (default `g.level_major`; the fused field kernels read only this layout), else the reference's row-major [P][L*F]."""
    lm = g.level_major if level_major is None else level_major
    P = x01.shape[0]
    out = torch.empty(P * g.L * g.F, device=x01.device, dtype=torch.float32)
    with ops._probe(f"hash_fwd_L{g.L}F{g.F}T{g.log2_T}"):
        call("ps_hash_fwd_lm" if lm else "ps_hash_fwd", ptr(x01), P, ptr(table), host_floats(g.scalings), g.L, g.F, g.log2_T, ptr(out), stream())
    return out


def _feat_seg(feat, dfeat, g: GridMeta):
    """Row-segment descriptor of level-major hash features (and their gradient buffer)."""
    return (feat, dfeat, g.L * g.F, 0, g.L * g.F, 1, g.F if g.level_major else 0)


def _hash_bwd(x01, dfeat, table, g: GridMeta, level_major: Optional[bool] = None):
    """-> the table gradient of features `dfeat` laid out as `_hash_fwd` writes them."""
    lm = g.level_major if level_major is None else level_major
    dtable = torch.zeros_like(table)
    with ops._probe(f"hash_bwd_L{g.L}F{g.F}T{g.log2_T}"):
        call("ps_hash_bwd_lm" if lm else "ps_hash_bwd", ptr(x01), x01.shape[0], None, host_floats(g.scalings), g.L, g.F, g.log2_T, ptr(dfeat),
             ptr(dtable), None, stream())
    return dtable


def _split_params(params: Sequence[Tensor], counts: Sequence[int]):
    """params = [W..., b...] per network, concatenated; counts = layers per network."""
    nets, i = [], 0
    for n in counts:
        ws = [p.detach() for p in params[i:i + n]]
        bs = [p.detach() for p in params[i + n:i + 2 * n]]
        nets.append((ws, bs))
        i += 2 * n
    return nets


class _PropLevel(torch.autograd.Function):
    """weights of one proposal level from bin edges (prop_density_field.py:129-153 + rays.py:128-150)."""

    @staticmethod
    def forward(ctx, origins, dirs, eu_bins, table, aabb, contract, grid: GridMeta, net: MlpMeta, prec, *params):
        o, d, eu = _f32c(origins.detach()), _f32c(dirs.detach()), _f32c(eu_bins.detach())
        N, S = eu.shape[0], eu.shape[1] - 1
        P = N * S
        (ws, bs), = _split_params(params, [net.n_layers])
        x01, sel = _ray_points(o, d, eu, aabb, contract)
        feat = _hash_fwd(x01, table.detach(), grid)
        density = torch.empty(P, device=eu.device, dtype=torch.float32)
        _mlp_fwd([_feat_seg(feat, None, grid)], P, ws, bs, net, prec, None, sel, density, "prop")
        w = torch.empty(N, S, device=eu.device, dtype=torch.float32)
        call("ps_composite_fwd", ptr(eu), ptr(density), None, None, N, S, 0, 0.5, ptr(w), None, None, None, None, None,
             None, stream())
        ctx.save_for_backward(eu, x01, sel, feat, density, table, *params)
        ctx.meta = (grid, net, prec, N, S)
        return w.view(N, S, 1)

    @staticmethod
    def backward(ctx, dw):
        grid, net, prec, N, S = ctx.meta
        eu, x01, sel, feat, density, table, *params = ctx.saved_tensors
        P = N * S
        (ws, bs), = _split_params(params, [net.n_layers])
        d_density = torch.empty(P, device=eu.device, dtype=torch.float32)
        call("ps_composite_bwd", ptr(eu), ptr(density), None, None, None, None, None, N, S, 0,
             ptr(_f32c(dw).view(N, S)), None, None, None, None, ptr(d_density), None, None, stream())
        dfeat = torch.empty_like(feat)
        dW = [torch.zeros_like(w) for w in ws]
        db = [torch.zeros_like(b) for b in bs]
        _mlp_bwd([_feat_seg(feat, dfeat, grid)], None, P, ws, bs, net, prec, dW, db, sel, d_density, "prop")
        dtable = _hash_bwd(x01, dfeat, table, grid)
        return (None, None, None, dtable, None, None, None, None, None, *dW, *db)


# ---------------------------------------------------------------------------------------------------------------
# tcgen05 proposal level: positions + hash gather + MLP + weights in ONE kernel per direction (csrc/prop_tc5.cu)
# ---------------------------------------------------------------------------------------------------------------
def tc5_prop_supported(grid: GridMeta, net: MlpMeta, prec, S: int) -> bool:
    return (prec == ops.PREC_BF16 and grid.F in (1, 2) and grid.L * grid.F <= 16 and S in (32, 64, 96, 128)
            and net.n_layers == 2 and net.dims[1] in (16, 64) and net.dims[2] == 1 and net.out_act == ops.ACT_NONE)


class _PropLevelTc5(torch.autograd.Function):
    @staticmethod
    def forward(ctx, origins, dirs, eu_bins, table, aabb, contract, grid: GridMeta, grad_key, w0, b0, w1, b1):
        import ctypes as C
        ctx.grad_key = grad_key
        from ._lib import host_prop_net, load
        o, d, eu = _f32c(origins.detach()), _f32c(dirs.detach()), _f32c(eu_bins.detach())
        N, S = eu.shape[0], eu.shape[1] - 1
        need_grad = any(ctx.needs_input_grad)
        stride = int(load().ps_prop_level_feat_stride(grid.L, grid.F))
        feat = torch.empty(N * S, stride, device=eu.device, dtype=torch.bfloat16) if need_grad else None
        w = torch.empty(N, S, device=eu.device, dtype=torch.float32)
        net = host_prop_net([w0.detach(), w1.detach()], [b0.detach(), b1.detach()])
        with ops._probe(f"prop_level_fwd_S{S}"):
            call("ps_prop_level_fwd", C.byref(net), ptr(o), ptr(d), ptr(eu), N, S, host_floats(aabb), 1 if contract else 0,
                 ptr(table.detach()), host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(w), ptr(feat), stream())
        if need_grad:
            ctx.save_for_backward(o, d, eu, feat, table, w0, b0, w1, b1)
        ctx.meta = (grid, tuple(aabb), contract, N, S)
        return w.view(N, S, 1)

    @staticmethod
    def backward(ctx, dw):
        import ctypes as C
        from ._lib import host_prop_net
        grid, aabb, contract, N, S = ctx.meta
        o, d, eu, feat, table, w0, b0, w1, b1 = ctx.saved_tensors
        ws, bs = [w0.detach(), w1.detach()], [b0.detach(), b1.detach()]
        main = torch.cuda.current_stream()
        # The proposal levels' gradients depend only on the interlevel loss, not on the final level's backward: when
        # the producer of `dw` published its completion event, run this backward on a side stream so that it overlaps
        # the field kernels / main hash scatter already queued on the main stream.
        ev_in = ops.pop_grad_event(dw, ctx.grad_key) if OVERLAP_PROP_BWD else None
        run_on = ops.side_stream(eu.device) if ev_in is not None else main
        with torch.cuda.stream(run_on):
            if ev_in is not None:
                run_on.wait_event(ev_in)
                # Order against the final level's backward (see _FIELD_BWD_ORDER): the first proposal backward since then
                # starts at once; a later one queues behind the field kernel — which needs whole SMs and all of tensor
                # memory, so cannot share them with this kernel's persistent CTAs — and co-runs with the main hash
                # scatter once the field kernel retires.
                order = _FIELD_BWD_ORDER.get(eu.device.index)
                if order is not None:
                    if order[1] >= 1:
                        run_on.wait_event(order[0])
                    order[1] += 1
            dwc = _f32c(dw).view(N, S)
            zs = _zeros_like_many([*ws, *bs])
            dws, dbs = zs[:2], zs[2:]
            dtable = torch.zeros_like(table)
            net = host_prop_net(ws, bs, dws, dbs)
            with ops._probe(f"prop_level_bwd_S{S}"):
                call("ps_prop_level_bwd", C.byref(net), ptr(o), ptr(d), ptr(eu), N, S, host_floats(aabb),
                     1 if contract else 0, host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(feat), ptr(dwc),
                     ptr(dtable), run_on.cuda_stream)
            if ev_in is not None:
                done = torch.cuda.Event()
                done.record(run_on)
        if ev_in is not None:
            # Join before returning: everything later on the main stream is ordered behind the side-stream kernel, so
            # `dw` (a main-stream block read on the side stream) may be freed by autograd right away, and the outputs
            # (side-stream blocks) are only ever reused by a later backward on the same side stream, which first waits
            # for a later main-stream event.  No Tensor.record_stream: its deferred frees make the caching allocator fall
            # back to cudaMalloc (a device-wide sync) whenever the host runs several steps ahead of the GPU.
            main.wait_event(done)
        return (None, None, None, dtable, None, None, None, None, dws[0], dbs[0], dws[1], dbs[1])


def prop_level_weights(origins, dirs, eu_bins, table, aabb, contract, grid: GridMeta, net: MlpMeta, prec,
                       weights: Sequence[Tensor], biases: Sequence[Tensor]) -> Tensor:
    if tc5_prop_supported(grid, net, prec, eu_bins.shape[1] - 1) and all(b is not None for b in biases):
        # hand-off key: a loss that consumes this tensor publishes its gradient's completion event under it (ops.py)
        key = ops.new_grad_key() if (OVERLAP_PROP_BWD and torch.is_grad_enabled()) else None
        out = _PropLevelTc5.apply(origins, dirs, eu_bins, table, aabb, contract, grid, key, weights[0], biases[0],
                                  weights[1], biases[1])
        if key is not None:
            out._ps_grad_key = key
        return out
    return _PropLevel.apply(origins, dirs, eu_bins, table, aabb, contract, grid, net, prec, *weights, *biases)


class _FieldLevel(torch.autograd.Function):
    """Final level: field evaluation + one-pass compositing (ingp_field.py:163-251, nerfacto_nusc_ms.py:497-530)."""

    @staticmethod
    def forward(ctx, origins, dirs, eu_bins, app, table, aabb, contract, grid: GridMeta, base: MlpMeta,
                sem: Optional[MlpMeta], rgb: MlpMeta, geo_dim: int, prec, threshold, *params):
        o, d, eu = _f32c(origins.detach()), _f32c(dirs.detach()), _f32c(eu_bins.detach())
        N, S = eu.shape[0], eu.shape[1] - 1
        P = N * S
        dev = eu.device
        counts = [base.n_layers] + ([sem.n_layers] if sem is not None else []) + [rgb.n_layers]
        nets = _split_params(params, counts)
        (bw, bb) = nets[0]
        (rw, rb) = nets[-1]
        A = 0 if app is None else app.shape[1]
        app_c = None if app is None else _f32c(app.detach())
        hd = base.dims[-1]
        sem_dim = 0 if sem is None else sem.dims[0]

        x01, sel = _ray_points(o, d, eu, aabb, contract)
        feat = _hash_fwd(x01, table.detach(), grid)
        h = torch.empty(P, hd, device=dev, dtype=torch.float32)
        density = torch.empty(P, device=dev, dtype=torch.float32)
        _mlp_fwd([_feat_seg(feat, None, grid)], P, bw, bb, base, prec, h, sel, density, "base")
        sem_s = None
        if sem is not None:
            sw, sb = nets[1]
            sem_s = torch.empty(P, sem.dims[-1], device=dev, dtype=torch.float32)
            _mlp_fwd([(h, None, hd, 1 + geo_dim, sem_dim, 1)], P, sw, sb, sem, prec, sem_s, name="sem")
        sh = ops.sh4(d)                                                   # [N,16], per ray
        segs = [(sh, None, 16, 0, 16, S), (h, None, hd, 1, geo_dim, 1)]
        if app_c is not None:
            segs.append((app_c, None, A, 0, A, S))
        rgb_s = torch.empty(P, 3, device=dev, dtype=torch.float32)
        _mlp_fwd(segs, P, rw, rb, rgb, prec, rgb_s, name="rgb")

        C = 0 if sem_s is None else sem_s.shape[1]
        w = torch.empty(N, S, device=dev, dtype=torch.float32)
        rgb_out = torch.empty(N, 3, device=dev, dtype=torch.float32)
        acc = torch.empty(N, 1, device=dev, dtype=torch.float32)
        dexp = torch.empty(N, 1, device=dev, dtype=torch.float32)
        dthr = torch.empty(N, 1, device=dev, dtype=torch.float32)
        sem_out = torch.empty(N, C, device=dev, dtype=torch.float32) if C else torch.empty(0, device=dev)
        tmm = ops.new_tminmax(dev)
        with ops._probe("composite_fwd"):
            call("ps_composite_fwd", ptr(eu), ptr(density), ptr(rgb_s), ptr(sem_s), N, S, C, float(threshold), ptr(w),
                 ptr(rgb_out), ptr(acc), ptr(dexp), ptr(dthr), ptr(sem_out) if C else None, ptr(tmm), stream())
        saved = [eu, x01, sel, feat, h, density, rgb_s, sh, acc, dexp, table]
        if sem_s is not None:
            saved.append(sem_s)
        if app_c is not None:
            saved.append(app_c)
        ctx.save_for_backward(*saved, *params)
        ctx.meta = (grid, base, sem, rgb, geo_dim, prec, N, S, A, len(saved), app is not None and app.requires_grad)
        ctx.mark_non_differentiable(dthr, tmm)
        return w.view(N, S, 1), rgb_out, acc, dexp, dthr, sem_out, tmm

    @staticmethod
    def backward(ctx, dw, drgb, dacc, ddexp, _dthr, dsem, _dtmm):
        grid, base, sem, rgb, geo_dim, prec, N, S, A, n_saved, app_grad = ctx.meta
        saved = list(ctx.saved_tensors)
        params = saved[n_saved:]
        eu, x01, sel, feat, h, density, rgb_s, sh, acc, dexp, table = saved[:11]
        rest = saved[11:n_saved]
        sem_s = rest.pop(0) if sem is not None else None
        app_c = rest.pop(0) if A else None
        P = N * S
        dev = eu.device
        counts = [base.n_layers] + ([sem.n_layers] if sem is not None else []) + [rgb.n_layers]
        nets = _split_params(params, counts)
        (bw, bb) = nets[0]
        (rw, rb) = nets[-1]
        hd = base.dims[-1]
        C = 0 if sem_s is None else sem_s.shape[1]

        d_density = torch.empty(P, device=dev, dtype=torch.float32)
        d_rgb_s = torch.empty(P, 3, device=dev, dtype=torch.float32)
        d_sem_s = torch.empty(P, C, device=dev, dtype=torch.float32) if C else None
        with ops._probe("composite_bwd"):
            # converted upstream gradients bound to names: ptr() keeps only an address, and a copy freed before the
            # launch may be handed to the next one of the argument list
            g = [_f32c(dw).view(N, S), _f32c(drgb), _f32c(dacc), _f32c(ddexp), _f32c(dsem) if C else None]
            call("ps_composite_bwd", ptr(eu), ptr(density), ptr(rgb_s), ptr(sem_s), None, ptr(acc), ptr(dexp), N, S, C,
                 *map(ptr, g), ptr(d_density), ptr(d_rgb_s), ptr(d_sem_s), stream())
        # dh: column 0 is driven by d_density inside the base backward; [1, 1+geo) by the colour head;
        # [1+geo, ...) by the semantic head (zero when there is none)
        dh = torch.empty(P, hd, device=dev, dtype=torch.float32) if sem is not None \
            else torch.zeros(P, hd, device=dev, dtype=torch.float32)
        dapp = torch.zeros(N, A, device=dev, dtype=torch.float32) if (A and app_grad) else None
        segs = [(sh, None, 16, 0, 16, S), (h, dh, hd, 1, geo_dim, 1)]
        if app_c is not None:
            segs.append((app_c, dapp, A, 0, A, S))
        dWr = [torch.zeros_like(w) for w in rw]
        dbr = [torch.zeros_like(b) for b in rb]
        _mlp_bwd(segs, d_rgb_s, P, rw, rb, rgb, prec, dWr, dbr, name="rgb")
        grads_sem: List[Tensor] = []
        if sem is not None:
            sw, sb = nets[1]
            dWs = [torch.zeros_like(w) for w in sw]
            dbs = [torch.zeros_like(b) for b in sb]
            _mlp_bwd([(h, dh, hd, 1 + geo_dim, sem.dims[0], 1)], d_sem_s, P, sw, sb, sem, prec, dWs, dbs, name="sem")
            grads_sem = [*dWs, *dbs]
        dfeat = torch.empty_like(feat)
        dWb = [torch.zeros_like(w) for w in bw]
        dbb = [torch.zeros_like(b) for b in bb]
        _mlp_bwd([_feat_seg(feat, dfeat, grid)], dh, P, bw, bb, base, prec, dWb, dbb, sel, d_density, "base")
        dtable = _hash_bwd(x01, dfeat, table, grid)
        return (None, None, None, dapp, dtable, None, None, None, None, None, None, None, None, None,
                *dWb, *dbb, *grads_sem, *dWr, *dbr)


# ---------------------------------------------------------------------------------------------------------------
# tcgen05 field level: base + semantic + colour networks and the compositing in ONE kernel per direction
# (csrc/field_tc5_fwd.cu / field_tc5_bwd.cu).  bf16 parity class only.
# ---------------------------------------------------------------------------------------------------------------
def tc5_field_supported(grid: GridMeta, base: MlpMeta, sem: Optional[MlpMeta], rgb: MlpMeta, geo_dim: int, prec,
                        S: int, A: int) -> bool:
    """The fused kernels implement exactly the reference field's architecture (ingp_field.py:118-161)."""
    return (prec == ops.PREC_BF16 and sem is not None and grid.F in (2, 4) and grid.L * grid.F <= 48
            and S in (32, 64, 96, 128) and geo_dim == 15 and 0 <= A <= 16
            and base.dims == (grid.L * grid.F, 64, 80) and sem.dims == (64, 64, 64, 64)
            and rgb.dims == (16 + 15 + A, 64, 64, 3) and rgb.out_act == ops.ACT_SIGMOID
            and base.out_act == ops.ACT_NONE and sem.out_act == ops.ACT_NONE)


def tc5_field_forward(o, d, eu, app_c, table, aabb, contract, grid: GridMeta, ws, bs, A, threshold):
    """-> (x01, sel, feat, w [N,S], rgb [N,3], acc [N,1], dexp [N,1], dthr [N,1], sem [N,64], tmm [2])."""
    from ._lib import host_field_net
    import ctypes as C
    N, S = eu.shape[0], eu.shape[1] - 1
    dev = eu.device
    x01, sel = _ray_points(o, d, eu, aabb, contract)
    w = torch.empty(N, S, device=dev, dtype=torch.float32)
    rgb_out = torch.empty(N, 3, device=dev, dtype=torch.float32)
    acc = torch.empty(N, 1, device=dev, dtype=torch.float32)
    dexp = torch.empty(N, 1, device=dev, dtype=torch.float32)
    dthr = torch.empty(N, 1, device=dev, dtype=torch.float32)
    sem_out = torch.empty(N, 64, device=dev, dtype=torch.float32)
    tmm = ops.new_tminmax(dev)
    net = host_field_net(ws, bs, A)
    feat = _hash_fwd(x01, table, grid, level_major=True)
    with ops._probe("field_level_fwd"):
        call("ps_field_level_fwd", C.byref(net), ptr(feat), grid.L, grid.F, ptr(sel), ptr(eu), ptr(d), ptr(app_c), N, S,
             float(threshold), ptr(w), ptr(rgb_out), ptr(acc), ptr(dexp), ptr(dthr), ptr(sem_out), ptr(tmm), stream())
    return x01, sel, feat, w, rgb_out, acc, dexp, dthr, sem_out, tmm


_zeros_like_many = ops.zeros_like_many


def _chunk_bounds(N: int, S: int) -> List[Tuple[int, int]]:
    """Ray ranges of the final level's hash and field kernels: the whole batch, one range.  bench.py's timing of the
    main-grid scatter alone reads it, so that the scatter is launched over the same ranges as in the step."""
    return [(0, N)]


class _FieldLevelTc5(torch.autograd.Function):
    """Final level on the fused tcgen05 kernels: ray_points -> hash gather -> ONE field+compositing kernel; backward =
    ONE kernel (recompute + all gradients) -> hash scatter.  Saved for backward: bins, unit-cube points, selector and
    the hash features only."""

    @staticmethod
    def forward(ctx, origins, dirs, eu_bins, app, table, aabb, contract, grid: GridMeta, threshold, *params):
        o, d, eu = _f32c(origins.detach()), _f32c(dirs.detach()), _f32c(eu_bins.detach())
        N, S = eu.shape[0], eu.shape[1] - 1
        ws = [p.detach() for p in params[:8]]
        bs = [p.detach() for p in params[8:]]
        A = 0 if app is None else app.shape[1]
        app_c = None if app is None else _f32c(app.detach())
        x01, sel, feat, w, rgb_out, acc, dexp, dthr, sem_out, tmm = tc5_field_forward(
            o, d, eu, app_c, table.detach(), aabb, contract, grid, ws, bs, A, threshold)
        saved = [eu, d, x01, sel, feat, acc, dexp, table]
        if app_c is not None:
            saved.append(app_c)
        ctx.n_fixed = len(saved)
        ctx.save_for_backward(*saved, *params)
        ctx.meta = (grid, N, S, A, app is not None and app.requires_grad)
        ctx.mark_non_differentiable(dthr, tmm)
        ctx.set_materialize_grads(False)
        return w.view(N, S, 1), rgb_out, acc, dexp, dthr, sem_out, tmm

    @staticmethod
    def backward(ctx, dw, drgb, dacc, ddexp, _dthr, dsem, _dtmm):
        import ctypes as C
        from ._lib import host_field_net
        grid, N, S, A, app_grad = ctx.meta
        saved = list(ctx.saved_tensors)
        eu, d, x01, sel, feat, acc, dexp, table = saved[:8]
        app_c = saved[8] if A else None
        params = saved[ctx.n_fixed:]
        dev = eu.device
        ws = [p.detach() for p in params[:8]]
        bs = [p.detach() for p in params[8:]]
        zs = _zeros_like_many([*ws, *bs])
        dW, dB = zs[:8], zs[8:]
        dapp = torch.zeros(N, A, device=dev, dtype=torch.float32) if (A and app_grad) else None
        net = host_field_net(ws, bs, A, dW, dB)

        def opt(t, shape=None):      # upstream gradients that autograd did not produce stay NULL (set_materialize_grads)
            if t is None:
                return None
            t = _f32c(t)
            return t if shape is None else t.view(shape)
        dwc, drgbc, daccc, ddexpc, dsemc = opt(dw, (N, S)), opt(drgb), opt(dacc), opt(ddexp), opt(dsem)

        sink = _PARTIAL_SINKS.get(table.data_ptr())
        dtable = sink[2]() if (sink is not None and sink[2] is not None) else torch.zeros_like(table)
        # recorded where the field kernel's inputs are complete: a proposal backward launched later this step waits for it,
        # i.e. it cannot reach the GPU before the field kernel is launchable and queues behind it
        ev_ready = torch.cuda.Event()
        ev_ready.record()
        dfeat = torch.empty_like(feat)
        with ops._probe("field_level_bwd"):
            call("ps_field_level_bwd", C.byref(net), ptr(feat), grid.L, grid.F, ptr(sel), ptr(eu), ptr(d), ptr(app_c), N, S,
                 ptr(acc), ptr(dexp), ptr(dwc), ptr(drgbc), ptr(daccc), ptr(ddexpc), ptr(dsemc), ptr(dfeat), ptr(dapp),
                 stream())
        _FIELD_BWD_ORDER[dev.index] = [ev_ready, 0]      # [field kernel launchable, proposal backwards launched since]
        # with a sink: one scatter per level group (the kernel is level-major anyway), each handed to the sink at once
        T, P = 1 << grid.log2_T, N * S
        dfl, dtl = dfeat.view(grid.L, P * grid.F), dtable.view(grid.L, T * grid.F)
        for (l0, l1) in (sink[1] if sink is not None else [(0, grid.L)]):
            with ops._probe(f"hash_bwd_L{grid.L}F{grid.F}T{grid.log2_T}"):
                call("ps_hash_bwd_lm", ptr(x01), P, None, host_floats(grid.scalings[l0:l1]), l1 - l0, grid.F, grid.log2_T,
                     ptr(dfl[l0:l1]), ptr(dtl[l0:l1]), None, stream())
            if sink is not None:
                sink[0](dtable, l0 * T, l1 * T)
        return (None, None, None, dapp, dtable, None, None, None, None, *dW, *dB)


def field_level(origins, dirs, eu_bins, app, table, aabb, contract, grid: GridMeta, base: MlpMeta,
                sem: Optional[MlpMeta], rgb: MlpMeta, geo_dim: int, prec, threshold, base_params, sem_params,
                rgb_params):
    """-> (weights [N,S,1], rgb [N,3], acc [N,1], depth_expected_unclipped [N,1], depth_threshold [N,1],
    semantics [N,C], tminmax [2]).  *_params = (weights list, biases list)."""
    A = 0 if app is None else app.shape[1]
    if tc5_field_supported(grid, base, sem, rgb, geo_dim, prec, eu_bins.shape[1] - 1, A):
        ws = [*base_params[0], *sem_params[0], *rgb_params[0]]
        bs = [*base_params[1], *sem_params[1], *rgb_params[1]]
        return _FieldLevelTc5.apply(origins, dirs, eu_bins, app, table, aabb, contract, grid, threshold, *ws, *bs)
    flat = [*base_params[0], *base_params[1]]
    if sem is not None:
        flat += [*sem_params[0], *sem_params[1]]
    flat += [*rgb_params[0], *rgb_params[1]]
    return _FieldLevel.apply(origins, dirs, eu_bins, app, table, aabb, contract, grid, base, sem, rgb, geo_dim, prec,
                             threshold, *flat)


# ---------------------------------------------------------------------------------------------------------------
# Sub-field mode (SURVEY §8 a10): nearest-centroid routing folded into the level, on the device.  Reference routers:
# fields/PreSight/ingp_field_ms.py:80-126, prop_density_field_ms.py:86-105.  One `route_points` per level groups the
# level's points by sub-field (csrc/ms_route.cu, no host sync, static bounds); the fused tcgen05 kernels then run on
# sub-field-homogeneous tiles with per-tile hash tables and per-sub-field weights (csrc/prop_tc5.cu, field_tc5_*.cu),
# and the weights along the rays come from the one-pass compositing kernel.
# ---------------------------------------------------------------------------------------------------------------
MS_PAD = 256       # a sub-field's rows are padded to whole pairs of 128-row tiles


@dataclass
class Routing:
    """A level's points in sub-field order."""
    rows: int                 # static bound: P rounded up + nf * MS_PAD
    perm: Tensor              # [rows] int32: row -> point, -1 = padding
    tile_sf: Tensor           # [rows / 128] uint8: sub-field of each tile, 255 = unused
    x01: Tensor               # [rows, 3] unit-cube positions (normalised by the row's sub-field's aabb)
    sel: Tensor               # [rows] uint8 inside-the-cube flag
    sf: Tensor                # [P] uint8 nearest centroid of every point (original order)


def route_points(centroids: Tensor, aabbs_host: Sequence[Sequence[float]], contract: bool, origins: Optional[Tensor],
                 dirs: Optional[Tensor], eu: Optional[Tensor], positions: Optional[Tensor] = None) -> Routing:
    """Group the sample points of a level (ray mid-points of `eu`, or explicit `positions` [P,3]) by nearest centroid."""
    nf = centroids.shape[0]
    if positions is not None:
        pos = _f32c(positions.detach()).view(-1, 3)
        P, S, dev = pos.shape[0], 1, pos.device
    else:
        pos = None
        N, S = eu.shape[0], eu.shape[1] - 1
        P, dev = N * S, eu.device
    rows = (P + MS_PAD - 1) // MS_PAD * MS_PAD + nf * MS_PAD
    cen = _f32c(centroids.detach())
    from ._lib import _device_table
    sig = tuple(float(v) for b in aabbs_host for v in b)
    boxes = _device_table((("aabbs", id(aabbs_host)), str(dev)), sig,
                          lambda: torch.tensor(sig, dtype=torch.float32).view(nf, 6).to(dev))
    block_hist = torch.empty((P + 255) // 256 * nf, device=dev, dtype=torch.int32)
    seg_start = torch.empty(2 * nf + 1, device=dev, dtype=torch.int32)        # nf + 1 starts | nf totals
    sf = torch.empty(P, device=dev, dtype=torch.uint8)
    perm = torch.full((rows,), -1, device=dev, dtype=torch.int32)
    tile_sf = torch.empty(rows // 128, device=dev, dtype=torch.uint8)
    x01 = torch.zeros(rows, 3, device=dev, dtype=torch.float32)
    sel = torch.zeros(rows, device=dev, dtype=torch.uint8)
    o, d, e = (None, None, None) if pos is not None else (ptr(origins), ptr(dirs), ptr(eu))
    call("ps_ms_route", ptr(pos), o, d, e, P, S, ptr(cen), nf, ptr(sf), ptr(block_hist), stream())
    call("ps_ms_plan", ptr(block_hist), P, nf, MS_PAD, 128, rows, ptr(seg_start), ptr(tile_sf), stream())
    call("ps_ms_scatter", ptr(pos), o, d, e, P, S, ptr(sf), ptr(boxes), nf, 1 if contract else 0, ptr(block_hist),
         ptr(seg_start), ptr(perm), ptr(x01), ptr(sel), stream())
    return Routing(rows, perm, tile_sf, x01, sel, sf)


def tc5_ms_prop_supported(grid: GridMeta, hidden: int, prec) -> bool:
    return prec == ops.PREC_BF16 and grid.F in (1, 2) and grid.L * grid.F <= 16 and hidden in (16, 64)


class _PropLevelMS(torch.autograd.Function):
    """weights of one proposal level whose points are routed to nf sub-fields (prop_density_field_ms.py:86-105 +
    rays.py:128-150).  params = per sub-field (table, W0, b0, W1, b1), flattened."""

    @staticmethod
    def forward(ctx, origins, dirs, eu_bins, centroids, aabbs_host, contract, grid: GridMeta, nf, *params):
        from ._lib import PropNetDev, device_ptr_array, device_struct_array, load
        o, d, eu = _f32c(origins.detach()), _f32c(dirs.detach()), _f32c(eu_bins.detach())
        N, S = eu.shape[0], eu.shape[1] - 1
        dev = eu.device
        subs = [[t.detach() for t in params[5 * k:5 * k + 5]] for k in range(nf)]
        rt = route_points(centroids, aabbs_host, contract, o, d, eu)
        need_grad = any(ctx.needs_input_grad)
        stride = int(load().ps_prop_level_feat_stride(grid.L, grid.F))
        feat = torch.empty(rt.rows, stride, device=dev, dtype=torch.bfloat16) if need_grad else None
        slot = ("prop", subs[0][0].data_ptr())
        tables = device_ptr_array([s[0] for s in subs], dev, (slot, "tables"))
        nets = device_struct_array([PropNetDev(s[1].data_ptr(), s[2].data_ptr(), s[3].data_ptr(), s[4].data_ptr(), 0, 0, 0, 0)
                                    for s in subs], dev, (slot, "nets_fwd"))
        hidden = subs[0][1].shape[0]
        density = torch.zeros(N * S, device=dev, dtype=torch.float32)
        with ops._probe(f"prop_level_fwd_ms_S{S}"):
            call("ps_prop_level_fwd_ms", ptr(nets), hidden, ptr(rt.x01), ptr(rt.sel), ptr(rt.perm), ptr(rt.tile_sf), rt.rows,
                 ptr(tables), host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(density), ptr(feat), stream())
        w = torch.empty(N, S, device=dev, dtype=torch.float32)
        call("ps_composite_fwd", ptr(eu), ptr(density), None, None, N, S, 0, 0.5, ptr(w), None, None, None, None, None,
             None, stream())
        if need_grad:
            ctx.save_for_backward(eu, density, feat, rt.perm, rt.tile_sf, rt.x01, rt.sel, *params)
        ctx.meta = (grid, N, S, nf, rt.rows, hidden)
        return w.view(N, S, 1)

    @staticmethod
    def backward(ctx, dw):
        from ._lib import PropNetDev, device_ptr_array, device_struct_array
        grid, N, S, nf, rows, hidden = ctx.meta
        eu, density, feat, perm, tile_sf, x01, sel, *params = ctx.saved_tensors
        dev = eu.device
        subs = [[t.detach() for t in params[5 * k:5 * k + 5]] for k in range(nf)]
        d_density = torch.empty(N * S, device=dev, dtype=torch.float32)
        call("ps_composite_bwd", ptr(eu), ptr(density), None, None, None, None, None, N, S, 0,
             ptr(_f32c(dw).view(N, S)), None, None, None, None, ptr(d_density), None, None, stream())
        grads = _zeros_like_many([t for s in subs for t in s])            # one fill for every table / weight gradient
        gsub = [grads[5 * k:5 * k + 5] for k in range(nf)]
        slot = ("prop", subs[0][0].data_ptr())
        dtables = device_ptr_array([g[0] for g in gsub], dev, (slot, "dtables"))
        nets = device_struct_array([PropNetDev(s[1].data_ptr(), s[2].data_ptr(), s[3].data_ptr(), s[4].data_ptr(),
                                               g[1].data_ptr(), g[2].data_ptr(), g[3].data_ptr(), g[4].data_ptr())
                                    for s, g in zip(subs, gsub)], dev, (slot, "nets_bwd"))
        with ops._probe(f"prop_level_bwd_ms_S{S}"):
            call("ps_prop_level_bwd_ms", ptr(nets), hidden, ptr(x01), ptr(sel), ptr(perm), ptr(tile_sf), rows, ptr(dtables),
                 host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(feat), ptr(d_density), stream())
        return (None, None, None, None, None, None, None, None, *grads)


def prop_level_weights_ms(origins, dirs, eu_bins, centroids, aabbs_host, contract, grid: GridMeta, fields_params) -> Tensor:
    """fields_params: per sub-field (table, W0, b0, W1, b1)."""
    flat = [t for fp in fields_params for t in fp]
    return _PropLevelMS.apply(origins, dirs, eu_bins, centroids, aabbs_host, contract, grid, len(fields_params), *flat)


class _FieldLevelMS(torch.autograd.Function):
    """Final level with nf routed sub-fields (ingp_field_ms.py:80-126 + nerfacto_nusc_ms.py:497-530): route -> per-tile
    hash gather -> ONE fused field kernel (per-point density / rgb / semantics) -> one-pass compositing; backward:
    compositing backward -> ONE fused field backward kernel -> per-tile hash scatter.
    params = per sub-field (table, 8 weights, 8 biases), flattened."""

    PER = 17

    @staticmethod
    def forward(ctx, origins, dirs, eu_bins, app, centroids, aabbs_host, contract, grid: GridMeta, threshold, nf, *params):
        from ._lib import FieldNetDev, device_ptr_array, device_struct_array
        o, d, eu = _f32c(origins.detach()), _f32c(dirs.detach()), _f32c(eu_bins.detach())
        N, S = eu.shape[0], eu.shape[1] - 1
        P, dev = N * S, eu.device
        PER = _FieldLevelMS.PER
        subs = [[t.detach() for t in params[PER * k:PER * (k + 1)]] for k in range(nf)]
        A = 0 if app is None else app.shape[1]
        app_c = None if app is None else _f32c(app.detach())
        rt = route_points(centroids, aabbs_host, contract, o, d, eu)
        slot = ("field", subs[0][0].data_ptr())
        tables = device_ptr_array([s[0] for s in subs], dev, (slot, "tables"))
        feat = torch.empty(rt.rows * grid.L * grid.F, device=dev, dtype=torch.float32)
        with ops._probe(f"hash_fwd_ms_L{grid.L}F{grid.F}T{grid.log2_T}"):
            call("ps_hash_fwd_ms", ptr(rt.x01), rt.rows, ptr(tables), ptr(rt.tile_sf), host_floats(grid.scalings), grid.L,
                 grid.F, grid.log2_T, ptr(feat), stream())

        def net_of(s, g=None):
            n = FieldNetDev()
            for i in range(8):
                n.W[i], n.B[i] = s[1 + i].data_ptr(), s[9 + i].data_ptr()
                n.dW[i] = 0 if g is None else g[1 + i].data_ptr()
                n.dB[i] = 0 if g is None else g[9 + i].data_ptr()
            n.in_dim, n.app_dim = grid.L * grid.F, A
            return n
        nets = device_struct_array([net_of(s) for s in subs], dev, (slot, "nets_fwd"))
        density = torch.zeros(P, device=dev, dtype=torch.float32)
        rgb_s = torch.empty(P, 3, device=dev, dtype=torch.float32)
        sem_s = torch.empty(P, 64, device=dev, dtype=torch.float32)
        with ops._probe("field_level_fwd_ms"):
            call("ps_field_level_fwd_ms", ptr(nets), A, ptr(feat), grid.L, grid.F, ptr(rt.sel), ptr(rt.perm), ptr(rt.tile_sf),
                 rt.rows, S, ptr(d), ptr(app_c), ptr(density), ptr(rgb_s), ptr(sem_s), stream())
        w = torch.empty(N, S, device=dev, dtype=torch.float32)
        rgb_out = torch.empty(N, 3, device=dev, dtype=torch.float32)
        acc = torch.empty(N, 1, device=dev, dtype=torch.float32)
        dexp = torch.empty(N, 1, device=dev, dtype=torch.float32)
        dthr = torch.empty(N, 1, device=dev, dtype=torch.float32)
        sem_out = torch.empty(N, 64, device=dev, dtype=torch.float32)
        tmm = ops.new_tminmax(dev)
        with ops._probe("composite_fwd"):
            call("ps_composite_fwd", ptr(eu), ptr(density), ptr(rgb_s), ptr(sem_s), N, S, 64, float(threshold), ptr(w),
                 ptr(rgb_out), ptr(acc), ptr(dexp), ptr(dthr), ptr(sem_out), ptr(tmm), stream())
        saved = [eu, d, density, rgb_s, sem_s, acc, dexp, feat, rt.perm, rt.tile_sf, rt.x01, rt.sel]
        if app_c is not None:
            saved.append(app_c)
        ctx.n_fixed = len(saved)
        ctx.save_for_backward(*saved, *params)
        ctx.meta = (grid, N, S, A, nf, rt.rows, app is not None and app.requires_grad)
        ctx.net_of = net_of
        ctx.mark_non_differentiable(dthr, tmm)
        ctx.set_materialize_grads(False)
        return w.view(N, S, 1), rgb_out, acc, dexp, dthr, sem_out, tmm

    @staticmethod
    def backward(ctx, dw, drgb, dacc, ddexp, _dthr, dsem, _dtmm):
        from ._lib import device_ptr_array, device_struct_array
        grid, N, S, A, nf, rows, app_grad = ctx.meta
        saved = list(ctx.saved_tensors)
        eu, d, density, rgb_s, sem_s, acc, dexp, feat, perm, tile_sf, x01, sel = saved[:12]
        app_c = saved[12] if A else None
        params = saved[ctx.n_fixed:]
        PER = _FieldLevelMS.PER
        P, dev = N * S, eu.device
        subs = [[t.detach() for t in params[PER * k:PER * (k + 1)]] for k in range(nf)]

        def opt(t, shape=None):
            if t is None:
                return None
            t = _f32c(t)
            return t if shape is None else t.view(shape)
        d_density = torch.empty(P, device=dev, dtype=torch.float32)
        # the compositing backward writes d_rgb_s / d_sem_s only when their upstream gradient is given, and the sub-field
        # kernel reads both: a loss without colour (or semantics) must hand it zeros
        d_rgb_s = (torch.empty if drgb is not None else torch.zeros)(P, 3, device=dev, dtype=torch.float32)
        d_sem_s = (torch.empty if dsem is not None else torch.zeros)(P, 64, device=dev, dtype=torch.float32)
        with ops._probe("composite_bwd"):
            g = [opt(dw, (N, S)), opt(drgb), opt(dacc), opt(ddexp), opt(dsem)]     # alive until the launch
            call("ps_composite_bwd", ptr(eu), ptr(density), ptr(rgb_s), ptr(sem_s), None, ptr(acc), ptr(dexp), N, S, 64,
                 *map(ptr, g), ptr(d_density), ptr(d_rgb_s), ptr(d_sem_s), stream())
        grads = _zeros_like_many([t for s in subs for t in s])
        gsub = [grads[PER * k:PER * (k + 1)] for k in range(nf)]
        slot = ("field", subs[0][0].data_ptr())
        nets = device_struct_array([ctx.net_of(s, g) for s, g in zip(subs, gsub)], dev, (slot, "nets_bwd"))
        dapp = torch.zeros(N, A, device=dev, dtype=torch.float32) if (A and app_grad) else None
        dfeat = torch.empty_like(feat)
        with ops._probe("field_level_bwd_ms"):
            call("ps_field_level_bwd_ms", ptr(nets), A, ptr(feat), grid.L, grid.F, ptr(sel), ptr(perm), ptr(tile_sf), rows, S,
                 ptr(d), ptr(app_c), ptr(d_density), ptr(d_rgb_s), ptr(d_sem_s), ptr(dfeat), ptr(dapp), stream())
        dtables = device_ptr_array([g[0] for g in gsub], dev, (slot, "dtables"))
        with ops._probe(f"hash_bwd_ms_L{grid.L}F{grid.F}T{grid.log2_T}"):
            call("ps_hash_bwd_ms", ptr(x01), rows, ptr(dtables), ptr(tile_sf), ptr(perm), host_floats(grid.scalings), grid.L,
                 grid.F, grid.log2_T, ptr(dfeat), stream())
        return (None, None, None, dapp, None, None, None, None, None, None, *grads)


def field_level_ms(origins, dirs, eu_bins, app, centroids, aabbs_host, contract, grid: GridMeta, threshold, fields_params):
    """fields_params: per sub-field (table, [8 weights], [8 biases]) in the layer order base0, base1, sem0..2, rgb0..2."""
    flat = [t for (tab, ws, bs) in fields_params for t in (tab, *ws, *bs)]
    return _FieldLevelMS.apply(origins, dirs, eu_bins, app, centroids, aabbs_host, contract, grid, threshold,
                               len(fields_params), *flat)


@torch.no_grad()
def query_priors_ms(points_scaled: Tensor, prop_routers, field_router) -> Tuple[Tensor, Tensor]:
    """The prior query (scripts/extract_priors.py:130-138) for a model with several routed sub-fields: ONE routing of the
    points (the proposal networks and the field share centroids and aabbs), then the sub-field mode of the fused kernels —
    each proposal level's density, the field's density and semantics (its colour head's output is ignored) — and the
    finalising kernel.  prop_routers: PropNetDensityFieldMS list; field_router: iNGPFieldMS."""
    from ._lib import FieldNetDev, PropNetDev, device_ptr_array, device_struct_array
    pts = _f32c(points_scaled).view(-1, 3)
    M, dev = pts.shape[0], pts.device
    nf = len(field_router.fields)
    f0 = field_router.fields[0]
    rt = route_points(field_router.centroids, field_router._aabbs_host(), f0.spatial_distortion is not None, None, None,
                      None, positions=pts)
    dens = []
    for lvl, pr in enumerate(prop_routers):
        grid = pr._ms_meta()
        subs = []
        for f in pr.fields:
            l0, l1 = list(f.mlp_base[1].layers)
            subs.append([f.encoding.hash_table.detach(), l0.weight.detach(), l0.bias.detach(), l1.weight.detach(),
                         l1.bias.detach()])
        slot = ("prop", subs[0][0].data_ptr())
        tables = device_ptr_array([s_[0] for s_ in subs], dev, (slot, "tables"))
        nets = device_struct_array([PropNetDev(s_[1].data_ptr(), s_[2].data_ptr(), s_[3].data_ptr(), s_[4].data_ptr(),
                                               0, 0, 0, 0) for s_ in subs], dev, (slot, "nets_fwd"))
        d = torch.zeros(M, device=dev, dtype=torch.float32)
        call("ps_prop_level_fwd_ms", ptr(nets), subs[0][1].shape[0], ptr(rt.x01), ptr(rt.sel), ptr(rt.perm),
             ptr(rt.tile_sf), rt.rows, ptr(tables), host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(d), None,
             stream())
        dens.append(d)
    grid = field_router._ms_meta()
    subs = []
    for f in field_router.fields:
        layers = [*f.mlp_base_mlp.layers, *f.semantic_head.layers, *f.rgb_head.layers]
        subs.append([f.mlp_base_grid.hash_table.detach(), *[l.weight.detach() for l in layers],
                     *[l.bias.detach() for l in layers]])
    slot = ("field", subs[0][0].data_ptr())
    tables = device_ptr_array([s_[0] for s_ in subs], dev, (slot, "tables"))
    feat = torch.empty(rt.rows * grid.L * grid.F, device=dev, dtype=torch.float32)
    call("ps_hash_fwd_ms", ptr(rt.x01), rt.rows, ptr(tables), ptr(rt.tile_sf), host_floats(grid.scalings), grid.L, grid.F,
         grid.log2_T, ptr(feat), stream())

    def net_of(s_):
        n = FieldNetDev()
        for i in range(8):
            n.W[i], n.B[i], n.dW[i], n.dB[i] = s_[1 + i].data_ptr(), s_[9 + i].data_ptr(), 0, 0
        n.in_dim, n.app_dim = grid.L * grid.F, 0          # no appearance: the colour head's output is not used here
        return n
    nets = device_struct_array([net_of(s_) for s_ in subs], dev, (slot, "nets_query"))
    d = torch.zeros(M, device=dev, dtype=torch.float32)
    rgb = torch.empty(M, 3, device=dev, dtype=torch.float32)
    sem = torch.zeros(M, 64, device=dev, dtype=torch.float32)
    zdir = torch.zeros(1, 3, device=dev, dtype=torch.float32)
    call("ps_field_level_fwd_ms", ptr(nets), 0, ptr(feat), grid.L, grid.F, ptr(rt.sel), ptr(rt.perm), ptr(rt.tile_sf),
         rt.rows, max(M, 1), ptr(zdir), None, ptr(d), ptr(rgb), ptr(sem), stream())        # S = M: every point is "ray 0"
    dens.append(d)
    mean = torch.empty(M, device=dev, dtype=torch.float32)
    feats = torch.empty(M, 64, device=dev, dtype=torch.float16)
    call("ps_prior_finalize", host_ptrs(dens), len(dens), ptr(sem), M, 64, ptr(mean), ptr(feats), stream())
    return mean, feats


@torch.no_grad()
def query_priors(points_scaled: Tensor, prop_fields, field) -> Tuple[Tensor, Tensor]:
    """Dense prior query for one sub-field (scripts/extract_priors.py:130-138): mean of the proposal and field
    densities [M] fp32 and the clipped semantic features [M,C] fp16.

    The reference evaluates the main hash grid + base MLP twice (density_fn, then semantic_fn,
    fields/PreSight/ingp_field.py:256); both evaluations are identical, so one pass serves both outputs.
    prop_fields: PropNetDensityField list; field: iNGPField with semantics."""
    pts = _f32c(points_scaled).view(-1, 3)
    M, dev = pts.shape[0], pts.device
    dens = []
    x01 = sel = None
    for f in [*prop_fields, field]:
        key = (tuple(f.aabb_host()), f.spatial_distortion is not None)
        if x01 is None or key != last_key:      # every network of a sub-field shares the aabb: normalise once
            x01, sel = ops.normalize_positions(pts, f.aabb_host(), f.spatial_distortion is not None)
            sel = sel.reshape(-1)
            last_key = key
        if f is field:
            enc, mlp = f.mlp_base_grid, f.mlp_base_mlp
            layers = list(mlp.layers)
            prec = mlp.precision
        else:
            enc = f.encoding
            layers = [f.linear] if f.use_linear else list(f.mlp_base[1].layers)
            prec = f._precision
        g = GridMeta(enc._scalings_host, enc.log2_hashmap_size, enc.features_per_level)
        feat = _hash_fwd(x01, enc.hash_table.detach(), g)
        meta = MlpMeta((layers[0].weight.shape[1],) + tuple(l.weight.shape[0] for l in layers), ops.ACT_NONE)
        ws, bs = [l.weight.detach() for l in layers], [l.bias.detach() for l in layers]
        d = torch.empty(M, device=dev, dtype=torch.float32)
        if f is field:
            h = torch.empty(M, meta.dims[-1], device=dev, dtype=torch.float32)
            _mlp_fwd([_feat_seg(feat, None, g)], M, ws, bs, meta, prec, h, sel, d, "base")
        else:
            _mlp_fwd([_feat_seg(feat, None, g)], M, ws, bs, meta, prec, None, sel, d, "prop")
        dens.append(d)
    sl = list(field.semantic_head.layers)
    smeta = MlpMeta((sl[0].weight.shape[1],) + tuple(l.weight.shape[0] for l in sl), ops.ACT_NONE)
    sem = torch.empty(M, smeta.dims[-1], device=dev, dtype=torch.float32)
    _mlp_fwd([(h, None, h.shape[1], 1 + field.geo_feat_dim, field.semantic_dim, 1)], M,
             [l.weight.detach() for l in sl], [l.bias.detach() for l in sl], smeta, field.semantic_head.precision, sem,
             name="sem")
    mean = torch.empty(M, device=dev, dtype=torch.float32)
    feats = torch.empty(M, smeta.dims[-1], device=dev, dtype=torch.float16)
    call("ps_prior_finalize", host_ptrs(dens), len(dens), ptr(sem), M, smeta.dims[-1], ptr(mean), ptr(feats), stream())
    return mean, feats


# ---------------------------------------------------------------------------------------------------------------
# Density level of the main field, forward only (prior extraction): the final level of `get_depth` as the fused proposal
# kernels instantiated for the field's density head (csrc/prop_tc5.cu, ps_density_level_fwd*), then the threshold depth.
# No autograd node and no saved state: these run under torch.no_grad().
# ---------------------------------------------------------------------------------------------------------------
def tc5_density_supported(grid: GridMeta, hidden: int, prec, S: int) -> bool:
    """The fused density level covers the bf16 parity class, hidden width 64, L*F <= 48 with F in {1,2,4} and
    S in {32,64,96,128}; anything else (fp32 class, S = 48, ...) keeps the per-operator path."""
    return (prec == ops.PREC_BF16 and hidden == 64 and grid.F in (1, 2, 4) and grid.L * grid.F <= 48
            and S in (32, 64, 96, 128))


@torch.no_grad()
def density_level_depth(origins, dirs, eu_bins, table, aabb, contract, grid: GridMeta, w0, b0, w1, b1,
                        threshold: float = 0.5) -> Tensor:
    """Threshold depth [N,1] of one sub-field's final level: ps_density_level_fwd -> ps_depth_threshold.
    w0 / b0: base0 weight [64, L*F] / bias; w1 / b1: base1 weight [80, 64] / bias (row 0 and bias[0] are read)."""
    import ctypes as C
    from ._lib import host_prop_net
    o, d, eu = _f32c(origins), _f32c(dirs), _f32c(eu_bins)
    N, S = eu.shape[0], eu.shape[1] - 1
    w = torch.empty(N, S, device=eu.device, dtype=torch.float32)
    net = host_prop_net([w0.detach(), w1.detach()], [b0.detach(), b1.detach()])
    with ops._probe(f"density_level_fwd_S{S}"):
        call("ps_density_level_fwd", C.byref(net), ptr(o), ptr(d), ptr(eu), N, S, host_floats(aabb), 1 if contract else 0,
             ptr(table.detach()), host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(w), stream())
    depth = torch.empty(N, 1, device=eu.device, dtype=torch.float32)
    call("ps_depth_threshold", ptr(w), ptr(eu), N, S, float(threshold), ptr(depth), None, stream())
    return depth


@torch.no_grad()
def density_level_depth_ms(origins, dirs, eu_bins, centroids, aabbs_host, contract, grid: GridMeta, fields_params,
                           threshold: float = 0.5) -> Tensor:
    """Threshold depth [N,1] of a final level routed to nf sub-fields: route_points -> ps_density_level_fwd_ms ->
    ps_composite_fwd (threshold depth only).  fields_params: per sub-field (table, w0, b0, w1, b1) as in
    density_level_depth."""
    from ._lib import PropNetDev, device_ptr_array, device_struct_array
    o, d, eu = _f32c(origins), _f32c(dirs), _f32c(eu_bins)
    N, S = eu.shape[0], eu.shape[1] - 1
    dev = eu.device
    subs = [[t.detach() for t in fp] for fp in fields_params]
    rt = route_points(centroids, aabbs_host, contract, o, d, eu)
    slot = ("density", subs[0][0].data_ptr())
    tables = device_ptr_array([s[0] for s in subs], dev, (slot, "tables"))
    nets = device_struct_array([PropNetDev(s[1].data_ptr(), s[2].data_ptr(), s[3].data_ptr(), s[4].data_ptr(), 0, 0, 0, 0)
                                for s in subs], dev, (slot, "nets_fwd"))
    density = torch.zeros(N * S, device=dev, dtype=torch.float32)
    with ops._probe(f"density_level_fwd_ms_S{S}"):
        call("ps_density_level_fwd_ms", ptr(nets), subs[0][1].shape[0], ptr(rt.x01), ptr(rt.sel), ptr(rt.perm),
             ptr(rt.tile_sf), rt.rows, ptr(tables), host_floats(grid.scalings), grid.L, grid.F, grid.log2_T, ptr(density),
             stream())
    depth = torch.empty(N, 1, device=dev, dtype=torch.float32)
    call("ps_composite_fwd", ptr(eu), ptr(density), None, None, N, S, 0, float(threshold), None, None, None, None,
         ptr(depth), None, None, stream())
    return depth
