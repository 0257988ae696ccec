"""GPU parity tests: every CUDA kernel (through the C-ABI) against the CPU oracle and the golden fixtures.

Bars (BASELINE.json north_star): bit-exact hash-corner indices and PDF bin indices; <= 1e-3 scale-relative for
fp32 results; <= 1e-2 for the bf16-MLP path.
"""
import numpy as np
import pytest
import torch

import oracle as O
from oracle import state as OS
from helpers import FAR, NEAR, THR, Fixture, assert_close, field_meta, prop_meta, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL32 = 1e-3
TOL16 = 1e-2


@pytest.fixture(scope="module")
def ops():
    from presight_b200 import ops as _ops
    return _ops


# ------------------------------------------------------------------------------------------ hash
@pytest.fixture(scope="module")
def fx_hash():
    return Fixture("hash.npz")


@pytest.mark.parametrize("name", ["kat4", "main16", "presight10", "prop8a", "prop8b", "prop5a", "prop5b",
                                  "main16_c2", "f8"])
def test_hash_indices_bit_exact_golden(ops, fx_hash, name):
    L, lo, hi, log2T, F = (int(v) for v in fx_hash.np(f"{name}/cfg"))
    s = O.hash_scalings(L, lo, hi)
    idx, off = ops.hash_indices(fx_hash["x"].to(DEV), s.tolist(), log2T)
    assert torch.equal(idx.cpu(), fx_hash[f"{name}/idx"])
    assert torch.equal(off.cpu(), fx_hash[f"{name}/offset"])


def test_hash_indices_bit_exact_random(ops):
    g = torch.Generator().manual_seed(5)
    x = torch.rand(20000, 3, generator=g) * 1.2 - 0.1        # includes out-of-cube values
    x[:100] = torch.randint(0, 65, (100, 3), generator=g).float() / 64.0   # exact lattice points
    for (L, lo, hi, log2T) in [(16, 16, 2048, 22), (10, 16, 16384, 20), (8, 16, 4096, 20), (5, 16, 128, 17)]:
        s = O.hash_scalings(L, lo, hi)
        want, woff = O.hash_corner_indices(x, s, log2T)
        got, goff = ops.hash_indices(x.to(DEV), s.tolist(), log2T)
        assert torch.equal(got.cpu(), want)
        assert torch.equal(goff.cpu(), woff)


@pytest.mark.parametrize("name", ["v_l4f2", "v_l8f1", "v_l10f4", "v_l16f2", "v_l3f8"])
def test_hash_values_and_grads_golden(ops, fx_hash, name):
    L, lo, hi, log2T, F = (int(v) for v in fx_hash.np(f"{name}/cfg"))
    s = O.hash_scalings(L, lo, hi).tolist()
    table = fx_hash[f"{name}/table"].to(DEV).requires_grad_(True)
    x = fx_hash["x"].to(DEV).requires_grad_(True)
    y = ops.hash_encode(x, table, s, log2T)
    # forward follows the reference's evaluation order with un-fused fp32 ops: bit-exact
    assert torch.equal(y.cpu(), fx_hash[f"{name}/out"])
    y.backward(fx_hash[f"{name}/dout"].to(DEV))
    assert_close(table.grad.cpu(), fx_hash[f"{name}/dtable"], TOL32, "dtable")
    assert_close(x.grad.cpu(), fx_hash[f"{name}/dx"], TOL32, "dx")


def test_hash_large_against_oracle(ops):
    """Config-2 sized levels on a smaller table; empty input; repeated points (atomic contention)."""
    g = torch.Generator().manual_seed(11)
    L, lo, hi, log2T, F = 16, 16, 2048, 16, 2
    s = O.hash_scalings(L, lo, hi)
    table = (torch.rand((1 << log2T) * L, F, generator=g) * 2 - 1)
    x = torch.rand(30000, 3, generator=g)
    x[1000:3000] = x[0]                       # 2000 identical points hammer the same entries
    x[3000:3500] = 0.0                        # masked points collapse to the origin
    dout = torch.randn(x.shape[0], L * F, generator=g)
    t_cpu = table.clone().requires_grad_(True)
    y_cpu = O.hash_encode(x, O.HashGrid(t_cpu, s, log2T))
    y_cpu.backward(dout)
    t_gpu = table.to(DEV).requires_grad_(True)
    y = ops.hash_encode(x.to(DEV), t_gpu, s.tolist(), log2T)
    assert torch.equal(y.cpu(), y_cpu.detach())
    y.backward(dout.to(DEV))
    assert_close(t_gpu.grad.cpu(), t_cpu.grad, TOL32, "dtable")
    # linearity of the scatter: grad(2*dout) == 2*grad(dout)
    t2 = table.to(DEV).requires_grad_(True)
    ops.hash_encode(x.to(DEV), t2, s.tolist(), log2T).backward(2 * dout.to(DEV))
    assert_close(t2.grad, 2 * t_gpu.grad, 1e-5, "linearity")
    empty = ops.hash_encode(torch.zeros(0, 3, device=DEV), t_gpu, s.tolist(), log2T)
    assert empty.shape == (0, L * F)


# ------------------------------------------------------------------------------------------ prologue
def test_normalize_positions_and_sh(ops):
    fx = Fixture("fields.npz")
    pos = fx["pos"]
    aabb = fx["field/aabb"]
    want, wsel = O.normalize_to_unit_cube(pos, aabb, True)
    got, gsel = ops.normalize_positions(pos.to(DEV), aabb.flatten().tolist(), True)
    assert torch.equal(gsel.cpu().bool(), wsel)
    assert_close(got.cpu(), want, 1e-6, "x01")
    want2, wsel2 = O.normalize_to_unit_cube(pos, aabb, False)
    got2, gsel2 = ops.normalize_positions(pos.to(DEV), aabb.flatten().tolist(), False)
    assert torch.equal(gsel2.cpu().bool(), wsel2)
    assert_close(got2.cpu(), want2, 1e-6, "x01 (no contraction)")
    assert_close(ops.sh4(fx["dirs"].to(DEV)).cpu(), fx["sh_out"], 1e-6, "sh4")
    assert_close(ops.sh4(((fx["dirs"] + 1) / 2).to(DEV), mapped=True).cpu(), fx["sh_out"], 1e-6, "sh4 mapped")
    assert torch.equal(ops.nearest_centroid(pos.to(DEV), fx["ms/centroids"].to(DEV)).cpu().long(), fx["ms/assign"])


# ------------------------------------------------------------------------------------------ MLP
SHAPES = [  # (in, hidden, n_layers, out, out_act)
    (8, 64, 2, 1, 0), (10, 16, 2, 1, 0), (5, 64, 2, 1, 0), (8, 0, 1, 1, 0),
    (32, 64, 2, 80, 0), (32, 64, 2, 16, 0), (40, 64, 2, 80, 0), (12, 64, 2, 80, 0),
    (64, 64, 3, 64, 0), (47, 64, 3, 3, 2), (63, 64, 3, 3, 2), (31, 64, 3, 3, 2),
    (32, 32, 3, 3, 2), (16, 32, 3, 64, 0),
]


def _make_mlp(g, n_in, hidden, n_layers, n_out):
    dims = [n_in] + [hidden] * (n_layers - 1) + [n_out]
    ws = [torch.randn(dims[i + 1], dims[i], generator=g) / np.sqrt(dims[i]) for i in range(n_layers)]
    bs = [torch.randn(dims[i + 1], generator=g) * 0.1 for i in range(n_layers)]
    return ws, bs


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("prec", [0, 1])
def test_mlp_forward_backward(ops, shape, prec):
    """prec 0 (3xTF32): everything within 1e-3 of the fp32 oracle.
    prec 1 (bf16): outputs within 1e-2 of the fp32 oracle; gradients are checked tightly against the oracle's
    bf16-operand emulation (ReLU-mask flips make a max-norm comparison with fp32 gradients meaningless) and in
    relative L2 against the fp32 oracle."""
    n_in, hidden, n_layers, n_out, act = shape
    g = torch.Generator().manual_seed(n_in * 131 + n_out)
    ws, bs = _make_mlp(g, n_in, hidden, n_layers, n_out)
    P = 1000  # not a multiple of the 128-point tile
    x = torch.randn(P, n_in, generator=g)
    dy = torch.randn(P, n_out, generator=g)

    def run_oracle(fn):
        wc = [w.clone().requires_grad_(True) for w in ws]
        bc = [b.clone().requires_grad_(True) for b in bs]
        xc = x.clone().requires_grad_(True)
        yc = fn(xc, O.Mlp(wc, bc, "sigmoid" if act == 2 else None))
        yc.backward(dy)
        return yc.detach(), xc.grad, [w.grad for w in wc], [b.grad for b in bc]

    y32, dx32, dW32, db32 = run_oracle(O.mlp_forward)
    wg = [w.to(DEV).requires_grad_(True) for w in ws]
    bg = [b.to(DEV).requires_grad_(True) for b in bs]
    xg = x.to(DEV).requires_grad_(True)
    yg = ops.mlp(xg, wg, bg, act, prec)
    yg.backward(dy.to(DEV))
    if prec == 0:
        assert_close(yg.cpu(), y32, TOL32, "y")
        assert_close(xg.grad.cpu(), dx32, TOL32, "dx")
        for i in range(n_layers):
            assert_close(wg[i].grad.cpu(), dW32[i], TOL32, f"dW{i}")
            assert_close(bg[i].grad.cpu(), db32[i], TOL32, f"db{i}")
    else:
        assert_close(yg.cpu(), y32, TOL16, "y vs fp32 oracle")
        y16, dx16, dW16, db16 = run_oracle(O.mlp_forward_bf16_emulated)
        # a value sitting on a bf16 rounding boundary may round the other way after a different fp32 summation
        # order, so deeper nets agree with the emulation to a few bf16 ulps rather than exactly
        assert_close(yg.cpu(), y16, 3e-3, "y vs bf16 emulation")
        assert rel_l2(xg.grad.cpu(), dx16) < 2e-2, f"dx vs bf16 emulation {rel_l2(xg.grad.cpu(), dx16):.2e}"
        assert rel_l2(xg.grad.cpu(), dx32) < 8e-2, "dx vs fp32 oracle"
        for i in range(n_layers):
            assert rel_l2(wg[i].grad.cpu(), dW16[i]) < 2e-2, f"dW{i} vs bf16 emulation {rel_l2(wg[i].grad.cpu(), dW16[i]):.2e}"
            assert rel_l2(bg[i].grad.cpu(), db16[i]) < 2e-2, f"db{i} vs bf16 emulation"
            assert rel_l2(wg[i].grad.cpu(), dW32[i]) < 8e-2, f"dW{i} vs fp32 oracle"


def test_mlp_multi_tile_and_empty(ops):
    g = torch.Generator().manual_seed(3)
    ws, bs = _make_mlp(g, 32, 64, 2, 80)
    # With 2.4 M hidden units a few pre-activations land within float rounding of zero and flip their ReLU against
    # the CPU oracle; their weight in dW grows like sqrt(P).  This test is about accumulation across tiles, so keep
    # every unit active (hidden bias +8); mask handling is covered at P = 1000 above.
    bs[0] = bs[0] + 8.0
    P = 128 * 300 + 17        # more tiles than the persistent grid has CTAs
    x = torch.randn(P, 32, generator=g)
    dy = torch.randn(P, 80, generator=g)
    wc = [w.clone().requires_grad_(True) for w in ws]
    bc = [b.clone().requires_grad_(True) for b in bs]
    yc = O.mlp_forward(x, O.Mlp(wc, bc))
    yc.backward(dy)
    wg = [w.to(DEV).requires_grad_(True) for w in ws]
    bg = [b.to(DEV).requires_grad_(True) for b in bs]
    yg = ops.mlp(x.to(DEV), wg, bg, 0, 0)
    assert_close(yg.cpu(), yc, TOL32, "y")
    yg.backward(dy.to(DEV))
    for i in range(2):
        # 2.4 M hidden units: the handful whose pre-activation is within 1e-6 of zero may flip their ReLU against
        # the CPU oracle, which moves single entries by ~1e-2 of the maximum -> relative L2 is the robust check
        assert rel_l2(wg[i].grad.cpu(), wc[i].grad) < TOL32, f"dW{i}: {rel_l2(wg[i].grad.cpu(), wc[i].grad):.2e}"
        assert rel_l2(bg[i].grad.cpu(), bc[i].grad) < TOL32, f"db{i}"
    assert ops.mlp(torch.zeros(0, 32, device=DEV), wg, bg, 0, 1).shape == (0, 80)


def test_mlp_unsupported_shape_fails_loudly(ops):
    g = torch.Generator().manual_seed(3)
    ws, bs = _make_mlp(g, 200, 64, 2, 1)
    with pytest.raises(RuntimeError, match="no kernel instantiated"):
        ops.mlp(torch.zeros(4, 200, device=DEV), [w.to(DEV) for w in ws], [b.to(DEV) for b in bs], 0, 1)


def test_trunc_exp(ops):
    g = torch.Generator().manual_seed(9)
    x = torch.randn(5000, 1, generator=g) * 8
    x[0] = 20.0
    x[1] = -30.0
    sel = (torch.rand(5000, generator=g) > 0.2)
    xc = x.clone().requires_grad_(True)
    yc = O.trunc_exp(xc) * sel[:, None]
    gy = torch.randn(5000, 1, generator=g)
    yc.backward(gy)
    xg = x.to(DEV).requires_grad_(True)
    yg = ops.trunc_exp(xg, sel.to(DEV).to(torch.uint8))
    assert_close(yg.cpu(), yc, 1e-5, "trunc_exp")
    yg.backward(gy.to(DEV))
    assert_close(xg.grad.cpu(), xc.grad, 1e-5, "trunc_exp grad")


# ------------------------------------------------------------------------------------------ samplers
@pytest.fixture(scope="module")
def fx_sr():
    return Fixture("sampler_render.npz")


@pytest.mark.parametrize("S", [128, 256, 48])
def test_spaced_bins_golden(ops, fx_sr, S):
    fx = fx_sr
    sp, eu = ops.spaced_bins(fx["nears"].to(DEV), fx["fars"].to(DEV), S, THR, fx[f"spaced{S}/t_rand"].to(DEV))
    assert torch.equal(sp.cpu()[:, :-1], fx[f"spaced{S}/sp_starts"])
    assert_close(eu.cpu()[:, :-1], fx[f"spaced{S}/starts"], 1e-6, "euclidean starts")
    assert_close(eu.cpu()[:, 1:], fx[f"spaced{S}/ends"], 1e-6, "euclidean ends")
    pos = ops.sample_positions(fx["origins"].to(DEV), fx["dirs"].to(DEV), eu)
    assert_close(pos.cpu(), fx[f"spaced{S}/positions"], 1e-6, "positions")
    _, eu_e = ops.spaced_bins(fx["nears"].to(DEV), fx["fars"].to(DEV), S, THR, None)
    assert_close(eu_e.cpu()[:, :-1], fx[f"spaced{S}/eval_starts"], 1e-6, "eval starts")


@pytest.mark.parametrize("S_in,S_out", [(128, 64), (64, 64), (256, 96), (96, 48)])
def test_pdf_resample_golden(ops, fx_sr, S_in, S_out):
    fx = fx_sr
    k = f"pdf{S_in}_{S_out}"
    eps = float(torch.finfo(torch.float32).eps)
    args = (fx[f"{k}/weights"].to(DEV), fx[f"{k}/existing_sp"].to(DEV), S_out)
    nf = (fx["nears"].to(DEV), fx["fars"].to(DEV), THR)
    sp, eu, inds, cdf, u = ops.pdf_resample(*args, fx[f"{k}/rand"].to(DEV), *nf, padding=0.01, eps=eps, probes=True)
    assert torch.equal(u.cpu(), fx[f"{k}/u"])
    assert_close(cdf.cpu(), fx[f"{k}/cdf"], 1e-6, "cdf")
    # (i) the bin search itself is bit-exact on identical inputs ...
    assert torch.equal(ops.searchsorted_right(fx[f"{k}/cdf"].to(DEV), fx[f"{k}/u"].to(DEV)).cpu(), fx[f"{k}/inds"])
    assert torch.equal(inds.cpu(), torch.searchsorted(cdf.cpu(), u.cpu(), side="right"))
    # (ii) ... and end to end the indices agree except where u sits within 2 ulp of a cdf entry
    ref_inds = fx[f"{k}/inds"]
    mism = inds.cpu() != ref_inds
    if mism.any():
        rc, ru = fx[f"{k}/cdf"], fx[f"{k}/u"]
        near = torch.gather(rc, 1, ref_inds.clamp(0, S_in)) - ru
        near2 = torch.gather(rc, 1, (ref_inds - 1).clamp(0, S_in)) - ru
        gap = torch.minimum(near.abs(), near2.abs())
        assert (gap[mism] <= 4 * np.finfo(np.float32).eps).all(), "bin index differs away from a cdf edge"
        assert mism.float().mean() < 0.01
    assert_close(sp.cpu()[:, :-1], fx[f"{k}/train/sp_starts"], 1e-5, "spacing bins")
    assert_close(eu.cpu()[:, 1:], fx[f"{k}/train/ends"], 1e-5, "euclidean bins")
    sp_e, eu_e = ops.pdf_resample(*args, None, *nf, padding=0.01, eps=eps)
    assert_close(sp_e.cpu()[:, :-1], fx[f"{k}/eval/sp_starts"], 1e-5, "eval spacing bins")
    assert_close(eu_e.cpu()[:, :-1], fx[f"{k}/eval/starts"], 1e-5, "eval euclidean bins")


def test_pdf_resample_anneal_and_sortedness(ops):
    g = torch.Generator().manual_seed(21)
    N, S_in, S_out = 4096, 128, 64
    w = torch.rand(N, S_in, generator=g) ** 4
    nears, fars = torch.full((N, 1), NEAR), torch.full((N, 1), FAR)
    sp0, _ = O.spaced_bins(nears, fars, S_in, THR, torch.rand(N, 1, generator=g))
    rand = torch.rand(N, 1, generator=g)
    want, winds, _, _ = O.pdf_resample(torch.pow(w, 0.37), sp0, S_out, rand, 0.01, 1e-5)
    sp, eu, inds, _, _ = ops.pdf_resample(w.to(DEV), sp0.to(DEV), S_out, rand.to(DEV), nears.to(DEV), fars.to(DEV), THR,
                                          padding=0.01, eps=1e-5, anneal=0.37, probes=True)
    assert_close(sp.cpu(), want, 1e-4, "annealed bins")
    assert (inds.cpu() != winds).float().mean() < 0.01
    assert (sp[:, 1:] >= sp[:, :-1]).all() and (eu[:, 1:] >= eu[:, :-1]).all()      # sorted without a sort
    assert (sp >= 0).all() and (sp <= 1).all()


# ------------------------------------------------------------------------------------------ compositing
def test_weights_and_renderers_golden(ops, fx_sr):
    fx = fx_sr
    deltas = fx["render/deltas"].to(DEV)
    dens = fx["render/density"][..., 0].to(DEV).requires_grad_(True)
    rgb = fx["render/rgb"].to(DEV).requires_grad_(True)
    sem = fx["render/sem"].to(DEV).requires_grad_(True)
    eu = torch.cat([fx["render/starts"], fx["render/ends"][:, -1:]], dim=-1).to(DEV)
    w = ops.get_weights(deltas, dens)
    assert_close(w.cpu(), fx["render/weights"][..., 0], 1e-5, "weights")
    img = ops.render(w, rgb)
    acc = ops.render(w, None)
    steps = ((fx["render/starts"] + fx["render/ends"]) / 2).to(DEV)
    dexp = torch.clip(ops.render(w, steps[..., None]) / (acc + 1e-10), steps.min(), steps.max())
    semo = ops.render(w, sem)
    dthr, didx = ops.depth_threshold(w, eu, 0.5)
    assert_close(img.cpu(), fx["render/img"], 1e-5, "rgb")
    assert_close(acc.cpu(), fx["render/acc"], 1e-5, "acc")
    assert_close(dexp.cpu(), fx["render/depth_expected"], 1e-5, "expected depth")
    assert_close(semo.cpu(), fx["render/sem_out"], 1e-5, "semantics")
    assert torch.equal(didx.cpu(), fx["render/depth_index"])
    assert_close(dthr.cpu(), fx["render/depth_threshold"], 1e-6, "threshold depth")
    loss = (img * fx["render/g_img"].to(DEV)).sum() + (acc * fx["render/g_acc"].to(DEV)).sum() \
        + (dexp * fx["render/g_dexp"].to(DEV)).sum() + (semo * fx["render/g_sem"].to(DEV)).sum() \
        + (w * fx["render/g_w"][..., 0].to(DEV)).sum()
    loss.backward()
    assert_close(dens.grad.cpu(), fx["render/d_density"][..., 0], TOL32, "d_density")
    assert_close(rgb.grad.cpu(), fx["render/d_rgb"], 1e-5, "d_rgb")
    assert_close(sem.grad.cpu(), fx["render/d_sem"], 1e-5, "d_sem")


def test_fused_composite_golden(ops, fx_sr):
    fx = fx_sr
    dens = fx["render/density"][..., 0].to(DEV).requires_grad_(True)
    rgb = fx["render/rgb"].to(DEV).requires_grad_(True)
    sem = fx["render/sem"].to(DEV).requires_grad_(True)
    eu = torch.cat([fx["render/starts"], fx["render/ends"][:, -1:]], dim=-1).to(DEV)
    w, img, acc, dexp_raw, dthr, semo, tmm = ops.composite(eu, dens, rgb, sem, 0.5)
    dexp = torch.clip(dexp_raw, tmm[0], tmm[1])
    assert_close(w.cpu(), fx["render/weights"][..., 0], 1e-5, "weights")
    assert_close(img.cpu(), fx["render/img"], 1e-5, "rgb")
    assert_close(acc.cpu(), fx["render/acc"], 1e-5, "acc")
    assert_close(dexp.cpu(), fx["render/depth_expected"], 1e-5, "expected depth")
    assert_close(dthr.cpu(), fx["render/depth_threshold"], 1e-6, "threshold depth")
    assert_close(semo.cpu(), fx["render/sem_out"], 1e-5, "semantics")
    steps = (fx["render/starts"] + fx["render/ends"]) / 2
    assert float(tmm[0]) == float(steps.min()) and float(tmm[1]) == float(steps.max())
    loss = (img * fx["render/g_img"].to(DEV)).sum() + (acc * fx["render/g_acc"].to(DEV)).sum() \
        + (dexp * fx["render/g_dexp"].to(DEV)).sum() + (semo * fx["render/g_sem"].to(DEV)).sum() \
        + (w * fx["render/g_w"][..., 0].to(DEV)).sum()
    loss.backward()
    assert_close(dens.grad.cpu(), fx["render/d_density"][..., 0], TOL32, "d_density")
    assert_close(rgb.grad.cpu(), fx["render/d_rgb"], 1e-5, "d_rgb")
    assert_close(sem.grad.cpu(), fx["render/d_sem"], 1e-5, "d_sem")


def test_composite_long_rays_against_oracle(ops):
    """S = 256 (8 chunks per warp) and S = 48 (ragged last chunk), random densities incl. opaque and empty rays."""
    g = torch.Generator().manual_seed(33)
    for S in (256, 48, 1):
        N = 777
        nears, fars = torch.full((N, 1), NEAR), torch.full((N, 1), FAR)
        _, eu = O.spaced_bins(nears, fars, S, THR, torch.rand(N, 1, generator=g))
        dens = torch.exp(torch.randn(N, S, generator=g) * 2)
        dens[0] = 0
        dens[1] = 1e7
        rgb = torch.rand(N, S, 3, generator=g)
        dc = dens.clone().requires_grad_(True)
        starts, ends = eu[:, :-1, None], eu[:, 1:, None]
        wc = O.get_weights(ends - starts, dc[..., None])
        imgc = O.render_rgb(rgb, wc)
        gw = torch.randn(N, S, generator=g)
        gi = torch.randn(N, 3, generator=g)
        ((wc[..., 0] * gw).sum() + (imgc * gi).sum()).backward()
        dg = dens.to(DEV).requires_grad_(True)
        w, img, acc, dexp, dthr, _, tmm = ops.composite(eu.to(DEV), dg, rgb.to(DEV), None, 0.5)
        assert_close(w.cpu(), wc[..., 0], 1e-5, f"weights S={S}")
        assert_close(img.cpu(), imgc, 1e-5, f"rgb S={S}")
        ((w * gw.to(DEV)).sum() + (img * gi.to(DEV)).sum()).backward()
        assert_close(dg.grad.cpu(), dc.grad, TOL32, f"d_density S={S}")
        dth_c, idx_c = O.render_depth_threshold(wc.detach(), starts, ends)
        assert_close(dthr.cpu(), dth_c, 1e-6, f"threshold depth S={S}")
        assert float(acc.max()) <= 1.0 + 1e-5       # sum of weights never exceeds 1


# ------------------------------------------------------------------------------------------ loss stack (8f-1)
@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_interlevel_loss_kernel_golden(ops, case):
    """ps_interlevel_loss (loss + gradient in one kernel) vs the live reference's fixture."""
    from presight_b200 import losses
    fx = Fixture("losses.npz")
    n = int(fx.np(f"{case}/n_levels"))
    c, w = fx[f"{case}/c"].to(DEV), fx[f"{case}/w"].to(DEV)
    ws = [fx[f"{case}/w{i}"].to(DEV).requires_grad_(True) for i in range(n)]
    ts = [fx[f"{case}/t{i}"].to(DEV) for i in range(n)]
    loss = losses.interlevel_loss([x[..., None] for x in ws] + [w[..., None]], ts + [c])
    assert_close(loss.cpu(), fx[f"{case}/loss"], 1e-5, "interlevel loss")
    (loss * 3.0).backward()
    for i in range(n):
        assert_close(ws[i].grad.cpu(), 3.0 * fx[f"{case}/g{i}"], TOL32, f"grad level {i}")


def test_interlevel_loss_kernel_random(ops):
    """large ragged shapes against the oracle (incl. S not a multiple of 32 and weights with exact zeros)."""
    g = torch.Generator().manual_seed(11)
    for (N, S, Sp) in [(1000, 64, 128), (513, 48, 256), (300, 33, 7)]:
        c = torch.rand(N, S + 1, generator=g).sort(-1).values
        t = torch.rand(N, Sp + 1, generator=g).sort(-1).values
        w = torch.rand(N, S, generator=g) ** 3
        w[torch.rand(N, S, generator=g) < 0.3] = 0
        we = (torch.rand(N, Sp, generator=g) ** 3 * 0.05).requires_grad_(True)
        want = O.lossfun_outer(c, w, t, we).mean()
        want.backward()
        wg = we.detach().to(DEV).requires_grad_(True)
        got = ops.interlevel_loss_level(c.to(DEV), w.to(DEV), t.to(DEV), wg)
        got.backward()
        assert_close(got.cpu(), want, 1e-5, f"loss {N}x{S}x{Sp}")
        assert_close(wg.grad.cpu(), we.grad, TOL32, f"grad {N}x{S}x{Sp}")


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_zaa_interlevel_loss_kernel_golden(ops, case):
    """ps_zaa_interlevel_loss (the reference's default proposal loss; loss + gradient in one kernel per level) vs the
    live reference's fixture, incl. the rays with near-degenerate bins whose result depends on the reference's
    argmax-on-ties interval selection."""
    from presight_b200 import losses
    fx = Fixture("zaa.npz")
    pulse = [float(v) for v in fx.np("pulse_width")]
    n = int(fx.np(f"{case}/n_levels"))
    c, w = fx[f"{case}/c"].to(DEV), fx[f"{case}/w"].to(DEV)
    ws = [fx[f"{case}/w{i}"].to(DEV).requires_grad_(True) for i in range(n)]
    ts = [fx[f"{case}/t{i}"].to(DEV) for i in range(n)]
    loss = losses.z_anti_aliasing_interlevel_loss([x[..., None] for x in ws] + [w[..., None]], ts + [c], pulse)
    assert_close(loss.cpu(), fx[f"{case}/loss"], 1e-5, "zaa interlevel loss")
    (loss * 2.0).backward()
    for i in range(n):
        assert_close(ws[i].grad.cpu(), 2.0 * fx[f"{case}/g{i}"], 2e-5, f"grad level {i}")


@pytest.mark.parametrize("case", ["a", "b", "c", "d"])
def test_distortion_loss_kernel_golden(ops, case):
    """ps_distortion_loss (loss + gradient in one kernel) vs the live reference's fixture, and on a large ragged batch vs
    the oracle."""
    from presight_b200 import losses
    fx = Fixture("distortion.npz")
    c, w = fx[f"{case}/c"].to(DEV), fx[f"{case}/w"].to(DEV).requires_grad_(True)
    loss = losses.distortion_loss([w], [c])
    assert_close(loss.cpu(), fx[f"{case}/loss"], 1e-5, "distortion loss")
    (loss * 3.0).backward()
    assert w.grad.shape == w.shape
    assert_close(w.grad.cpu(), 3.0 * fx[f"{case}/g"], 1e-5, "grad")
    if case == "a":
        g = torch.Generator().manual_seed(2)
        N, S = 3001, 64
        cc = torch.rand(N, S + 1, generator=g).sort(-1).values
        ww = (torch.rand(N, S, generator=g) ** 3 * 0.1).requires_grad_(True)
        want = O.distortion_loss([ww[..., None]], [cc])
        want.backward()
        wg = ww.detach().to(DEV).requires_grad_(True)
        got = ops.distortion_loss(cc.to(DEV), wg)
        got.backward()
        assert_close(got.cpu(), want, 1e-5, "loss (random)")
        assert_close(wg.grad.cpu(), ww.grad, 1e-5, "grad (random)")


@pytest.mark.parametrize("case", ["a", "b"])
def test_sky_blend_and_render_losses_golden(ops, case):
    """ps_sky_blend_fwd/bwd + ps_render_losses vs the live reference's fixture: blended outputs bit-exact, loss terms
    1e-5, every gradient of the weighted total 1e-5 (fp32 class)."""
    fx = Fixture("render_losses.npz")
    names = ("rgb_f", "acc_raw", "sem_f", "sky_rgb", "sky_sem")
    leaves = {k: fx[f"{case}/{k}"].to(DEV).requires_grad_(True) for k in names}
    rgb, acc, sem = ops.sky_blend(leaves["rgb_f"], leaves["acc_raw"], leaves["sem_f"], leaves["sky_rgb"], leaves["sky_sem"])
    assert torch.equal(rgb.cpu(), fx[f"{case}/rgb"]) and torch.equal(acc.cpu(), fx[f"{case}/acc"])
    assert torch.equal(sem.cpu(), fx[f"{case}/sem"])
    terms = ops.render_losses(rgb, fx[f"{case}/gt_rgb"].to(DEV), acc, fx[f"{case}/sky"].to(DEV), sem,
                              fx[f"{case}/gt_sem"].to(DEV))
    assert_close(terms.cpu(), fx[f"{case}/losses"], 1e-5, "loss terms")
    (terms[0] + 0.001 * terms[1] + 0.5 * terms[2]).backward()
    for k in names:
        assert_close(leaves[k].grad.cpu(), fx[f"{case}/g_{k}"], 1e-5, f"grad {k}")


def test_sky_blend_and_render_losses_variants(ops):
    """optional inputs (no sky model, no semantics, eval-mode rgb clamp, skipped loss terms) and a ragged large batch
    against the oracle."""
    g = torch.Generator().manual_seed(5)
    N, C = 4099, 24
    rgb_f = (torch.rand(N, 3, generator=g) * 1.4 - 0.2)
    acc_raw = torch.rand(N, 1, generator=g) * 1.4 - 0.2
    sem_f, sky_rgb, sky_sem = torch.randn(N, C, generator=g), torch.rand(N, 3, generator=g), torch.randn(N, C, generator=g)
    gt_rgb, sky, gt_sem = torch.rand(N, 3, generator=g), (torch.rand(N, 1, generator=g) < 0.5).float(), torch.randn(N, C, generator=g)
    for (use_sem, use_sky_rgb, use_sky_sem, training) in [(True, True, True, False), (True, True, False, True),
                                                         (False, True, False, True), (True, False, False, True),
                                                         (False, False, False, False)]:
        cpu = [t.clone().requires_grad_(True) for t in (rgb_f, acc_raw, sem_f, sky_rgb, sky_sem)]
        dev = [t.to(DEV).requires_grad_(True) for t in (rgb_f, acc_raw, sem_f, sky_rgb, sky_sem)]

        def pick(ts):
            return (ts[0], ts[1], ts[2] if use_sem else None, ts[3] if use_sky_rgb else None, ts[4] if use_sky_sem else None)
        r0, a0, s0 = O.sky_blend(*pick(cpu), training=training)
        r1, a1, s1 = ops.sky_blend(*pick(dev), clamp_rgb=not training)
        assert torch.equal(r1.cpu(), r0) and torch.equal(a1.cpu(), a0)
        assert (s1 is None) == (s0 is None) and (s0 is None or torch.equal(s1.cpu(), s0))
        want = O.rgb_loss(gt_rgb, r0) + 0.01 * O.sky_loss(a0, sky)
        terms = ops.render_losses(r1, gt_rgb.to(DEV), a1, sky.to(DEV), s1, None if s1 is None else gt_sem.to(DEV))
        got = terms[0] + 0.01 * terms[1]
        if s0 is not None:
            want = want + 0.5 * O.semantic_loss(s0, gt_sem)
            got = got + 0.5 * terms[2]
        else:
            assert float(terms[2]) == 0.0
        assert_close(got.cpu(), want, 1e-5, "total")
        want.backward()
        got.backward()
        for i, (c, d) in enumerate(zip(cpu, dev)):
            if c.grad is None:
                assert d.grad is None, i
            else:
                assert_close(d.grad.cpu(), c.grad, 1e-5, f"grad {i} variant {(use_sem, use_sky_rgb, use_sky_sem, training)}")
    # a skipped term: rgb only
    t = ops.render_losses(r1, gt_rgb.to(DEV), None, None, None, None)
    assert float(t[1]) == 0.0 and float(t[2]) == 0.0 and float(t[0]) > 0.0


def test_depth_losses_kernel_golden(ops):
    """ps_depth_losses vs the live reference's fixture (tests/golden/depth_losses.npz, model_components/PreSight/
    losses.py:28-103): expected mono-depth (normalised / inverse) and LiDAR depth losses with d/d predicted depth, the
    line-of-sight loss with d/d weights (with and without sky mask); then both terms from ONE launch with the sample
    mid-points derived from bin edges and a pose scale factor, against the oracle."""
    from presight_b200 import losses
    fx = Fixture("depth_losses.npz")
    depth, sky, steps = fx["depth"].cuda(), fx["sky"].cuda(), fx["steps"].cuda()
    for name, fn in {"mono": lambda p: losses.expected_monodepth_loss(depth, p, sky, 40.0, False),
                     "mono_inv": lambda p: losses.expected_monodepth_loss(depth, p, sky, 40.0, True),
                     "lidar": lambda p: losses.expected_depth_loss(depth, p, 75.0)}.items():
        pred = fx["pred"].cuda().requires_grad_(True)
        loss = fn(pred)
        assert_close(loss.cpu(), fx[f"{name}/loss"], 1e-5, name)
        loss.backward()
        assert_close(pred.grad.cpu(), fx[f"{name}/g"], 1e-5, name + " grad")
    for name, (sigma, use_sky, ub) in {"los_a": (5.0, True, 40.0), "los_b": (2.0, False, 75.0)}.items():
        w = fx["w"].cuda().requires_grad_(True)
        loss = losses.line_of_sight_loss(w, depth, steps, sigma, sky if use_sky else None, ub)
        assert_close(loss.cpu(), fx[f"{name}/loss"], 1e-5, name)
        loss.backward()
        assert_close(w.grad.cpu(), fx[f"{name}/g"], 1e-5, name + " grad")
    # one launch, mid-points from bin edges in scene units (nerfacto_nusc_ms.py:579-586)
    g = torch.Generator().manual_seed(5)
    n, S, scale = 1001, 48, 0.05
    eu = (torch.sort(torch.rand(n, S + 1, generator=g) * 70.0, dim=1).values * scale)
    wts = (torch.rand(n, S, 1, generator=g) ** 3 * 0.2)
    tgt = torch.rand(n, 1, generator=g) * 80.0
    skm = (torch.rand(n, 1, generator=g) < 0.2).float()
    exp_d = (tgt + torch.randn(n, 1, generator=g) * 3.0).clamp_min(0.01) * scale
    w_ref, e_ref = wts.clone().requires_grad_(True), exp_d.clone().requires_grad_(True)
    steps_ref = ((eu[:, :-1] + eu[:, 1:]) / 2 / scale)[..., None]
    want = [O.expected_monodepth_loss(tgt, e_ref / scale, skm, 40.0, False),
            O.line_of_sight_loss(w_ref, tgt, steps_ref, 3.5, skm, 40.0)]
    (want[0] + 0.3 * want[1]).backward()
    w_gpu, e_gpu = wts.cuda().requires_grad_(True), exp_d.cuda().requires_grad_(True)
    got = losses.depth_supervision_losses(w_gpu, e_gpu, tgt.cuda(), skm.cuda(), scale, 3.5, 40.0, False, eu_bins=eu.cuda())
    (got[0] + 0.3 * got[1]).backward()
    assert_close(got[0].cpu(), want[0].detach(), 1e-5, "expected depth (one launch)")
    assert_close(got[1].cpu(), want[1].detach(), 1e-5, "line of sight (one launch)")
    assert_close(e_gpu.grad.cpu(), e_ref.grad, 1e-5, "d expected depth")
    assert_close(w_gpu.grad.cpu(), w_ref.grad, 1e-5, "d weights")
    # an empty mask is NaN, as torch's mean over no rays
    none = losses.expected_depth_loss(torch.zeros(4, 1).cuda(), torch.ones(4, 1).cuda(), 75.0)
    assert bool(torch.isnan(none))


def test_fused_adam_matches_torch_adam(ops):
    """FusedAdam (ps_adam_step, SURVEY 8f-2) vs torch.optim.Adam — the reference's optimiser — with PreSight's
    hyper-parameters over several steps, on a table-shaped parameter and on small odd-sized ones (tail elements,
    parameters whose gradient is missing in a step)."""
    from presight_b200.optim import FusedAdam
    g = torch.Generator().manual_seed(0)
    shapes = [(1 << 16, 2), (64, 47), (3,), (1,)]
    init = [(torch.rand(*s, generator=g) * 2 - 1) * 1e-3 for s in shapes]
    ref = [torch.nn.Parameter(t.clone()) for t in init]
    dev = [torch.nn.Parameter(t.clone().to(DEV)) for t in init]
    o_ref = torch.optim.Adam(ref, lr=1e-2, eps=1e-15, weight_decay=1e-5, foreach=False)
    o_dev = FusedAdam(dev, lr=1e-2, eps=1e-15, weight_decay=1e-5)
    for step in range(6):
        for i, (a, b) in enumerate(zip(ref, dev)):
            if step == 2 and i == 1:
                a.grad, b.grad = None, None                       # a parameter that got no gradient this step
                continue
            gr = torch.randn(a.shape, generator=g) * 10.0 ** float(torch.randint(-6, 1, (1,), generator=g))
            gr[torch.rand(a.shape, generator=g) < 0.3] = 0.0
            a.grad, b.grad = gr.clone(), gr.to(DEV)
        if step == 4:
            for grp in (*o_ref.param_groups, *o_dev.param_groups):
                grp["lr"] = 2.5e-3                                # what a scheduler does
        o_ref.step()
        o_dev.step()
        for i, (a, b) in enumerate(zip(ref, dev)):
            assert_close(b.detach().cpu(), a.detach(), 1e-5, f"param {i} step {step}")
            assert_close(o_dev.state[b]["exp_avg_sq"].cpu(), o_ref.state[a]["exp_avg_sq"], 1e-5, f"exp_avg_sq {i} step {step}")
            assert int(o_dev.state[b]["step"]) == int(o_ref.state[a]["step"])


def test_generate_rays_golden(ops):
    """ps_generate_rays (pinhole RayGenerator, SURVEY 8f-3) vs the live reference's Cameras.generate_rays on nuScenes-shaped
    cameras: origins exact, unit directions and norms 1e-6, pixel area 1e-3 per ray (a product of differences of nearly
    equal unit vectors; fp32 class)."""
    from presight_b200.cameras.ray_generator import RayGenerator
    fx = Fixture("rays.npz")
    gen = RayGenerator(fx["c2w"], fx["fx"], fx["fy"], fx["cx"], fx["cy"]).to(DEV)
    rb = gen(fx["ray_indices"].to(DEV))
    assert torch.equal(rb.origins.cpu(), fx["origins"])
    assert_close(rb.directions.cpu(), fx["directions"], 1e-6, "directions")
    assert_close(rb.metadata["directions_norm"].cpu(), fx["directions_norm"], 1e-6, "directions_norm")
    rel = ((rb.pixel_area.cpu() - fx["pixel_area"]).abs() / fx["pixel_area"]).max()
    assert float(rel) < 1e-3, float(rel)
    assert torch.equal(rb.camera_indices.cpu(), fx["ray_indices"][:, :1])
    assert len(gen(torch.zeros(0, 3, dtype=torch.int64, device=DEV))) == 0


def test_tcgen05_operand_conventions(ops):
    """K-major / MN-major UMMA descriptors over one chunk-major tile (csrc/tc5.cuh): forward, input-gradient and
    weight-gradient GEMM forms against fp32 matmuls of the bf16-rounded operands."""
    from presight_b200._lib import call, ptr, stream
    g = torch.Generator().manual_seed(3)
    X, Y, W = torch.randn(128, 64, generator=g), torch.randn(128, 64, generator=g), torch.randn(64, 64, generator=g)
    Xd, Yd, Wd = X.to(DEV), Y.to(DEV), W.to(DEV)
    C = [torch.zeros(128, 64, device=DEV) for _ in range(3)]
    C4 = torch.full((128, 16), -1.0, device=DEV)
    call("ps_tc5_probe", ptr(Xd), ptr(Yd), ptr(Wd), ptr(C[0]), ptr(C[1]), ptr(C[2]), ptr(C4), stream())
    torch.cuda.synchronize()
    Xb, Yb, Wb = (t.bfloat16().float() for t in (X, Y, W))
    assert_close(C[0].cpu(), Xb @ Wb.T, 1e-5, "X W^T (K-major)")
    assert_close(C[1].cpu(), Xb @ Wb, 1e-5, "X W (MN-major B)")
    assert_close(C[2].cpu()[:64], 2.0 * (Xb.T @ Yb), 1e-5, "2 X^T Y (MN-major A and B, accumulated)")
    want4 = torch.zeros(64, 16)
    want4[:, 3] = Xb.sum(0)
    assert_close(C4.cpu()[:64], want4, 1e-5, "column sums through a one-hot operand with zero K stride")


def test_wrappers_keep_converted_inputs_alive():
    """Inputs a wrapper converts (non-contiguous or not fp32) stay referenced until the kernel is enqueued: with several
    conversions in one call, a copy freed early would have its block handed to the next one and be overwritten by it."""
    from presight_b200 import ops
    g = torch.Generator().manual_seed(0)
    N, S = 4096, 32
    o, d = torch.rand(N, 3, generator=g).to(DEV), torch.randn(N, 3, generator=g).to(DEV)
    eu = (torch.rand(N, S + 1, generator=g) * 0.1 + 0.01).cumsum(-1).to(DEV)

    def strided(t):                      # the same values as a column slice of a wider tensor: not contiguous
        return torch.cat([t, t], dim=1)[:, :t.shape[1]]
    assert torch.equal(ops.sample_positions(strided(o), strided(d), strided(eu)), ops.sample_positions(o, d, eu))
    density = (torch.rand(N, S, generator=g) * 5).to(DEV).requires_grad_(True)
    _, _, acc, dexp, _, _, _ = ops.composite(eu, density, None, None)
    # expanded upstream gradients of equal shape (what `acc.sum()` hands back) are converted one after the other
    ga, gd = torch.ones(1, 1, device=DEV).expand(N, 1), torch.full((1, 1), 0.5, device=DEV).expand(N, 1)
    got = torch.autograd.grad([acc, dexp], density, [ga, gd], retain_graph=True)[0]
    want = torch.autograd.grad([acc, dexp], density, [ga.contiguous(), gd.contiguous()])[0]
    assert torch.equal(got, want)
