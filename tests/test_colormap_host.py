"""CPU checks of the evaluation images and of LPIPS weights read from a reference checkpoint:
  - the per-pixel colormap core (presight_b200/csrc/colormap_core.h, the code the CUDA kernels run) compiled for the
    host, bit for bit against a numpy restatement of nerfstudio's colormaps in the same operation order;
  - `LPIPS.from_reference_state_dict` against `LPIPS.from_state_dicts` on the same weights, and its rejections."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
CHANNELS = (64, 192, 384, 256, 256)


# ---- colormap core ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("colormap") / "libcolormap_host.so")
    src = os.path.join(HERE, "native", "colormap_host.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", src, "-o", out], check=True)
    lib = ctypes.CDLL(out)
    lib.colormap_host.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                  ctypes.c_void_p]
    lib.colormap_host.restype = None
    return lib


def seeded_lut(seed=0):
    """Any [256,3] table in [0,1] (the project ships none; a user passes matplotlib's turbo colours)."""
    return np.random.default_rng(seed).random((256, 3)).astype(np.float32)


def boundary_values():
    """k / 255 for every LUT row and the float just below it."""
    k = (np.arange(256) / 255).astype(np.float32)
    return np.concatenate([k, np.nextafter(k, np.float32(-1))]).astype(np.float32)


def colormap_case(kind, H, W, M, seed=0):
    """(maps [M,H,W], acc [H,W]) float32 for the named case."""
    rng = np.random.default_rng(seed)
    n = H * W
    acc = rng.random(n).astype(np.float32)
    acc[: n // 7] = 0.0                                          # empty sky
    acc[n // 7: 2 * n // 7] = 1.0                                # opaque surfaces
    maps = (0.5 + 80.0 * rng.random((M, n)) ** 2).astype(np.float32)
    if kind == "constant":                                       # far == near: the divisor is 1e-10
        maps[:] = np.float32(7.25)
    elif kind == "boundaries":                                   # every LUT boundary, through both code paths
        b = boundary_values()
        reps = np.resize(b, n)
        acc = reps.copy()
        for m in range(M):                                       # near 0 and far 1: the depth map is the value itself
            maps[m] = np.resize(b, n)
            maps[m, 0], maps[m, 1] = 0.0, 1.0
    elif kind == "special":                                      # NaN and +-inf pixels, values outside [0,1]
        acc[3], acc[5] = -0.25, 1.5
        if M > 0:
            maps[0, n // 2] = np.nan
        if M > 1:
            maps[1, 7] = np.inf
        if M > 2:
            maps[2, 11] = -np.inf
    return maps.reshape(M, H, W), acc.reshape(H, W)


def np_index(x):
    x = np.clip(x, np.float32(0), np.float32(1))                 # propagates NaN, as torch.clip
    x = np.nan_to_num(x, nan=0.0)
    return (x * np.float32(255)).astype(np.int64)


def np_colormap(maps, acc, lut):
    """nerfstudio 0.3.3 apply_colormap / apply_depth_colormap with default options, in torch's operation order and
    rounding (see colormap_core.h) -> [M+1,H,W,3]."""
    out = [lut[np_index(acc)]]
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        for d in maps:
            near, far = float(np.min(d)), float(np.max(d))       # np.min / np.max propagate NaN, as torch's
            inv = np.float32(1.0 / (far - near + 1e-10))          # torch's reciprocal of a Python float
            x = (d - np.float32(near)) * inv
            c = lut[np_index(x)]
            out.append(c * acc[..., None] + (np.float32(1) - acc)[..., None])
    return np.stack(out).astype(np.float32)


def run_host(lib, maps, acc, lut):
    M, (H, W) = maps.shape[0], acc.shape
    maps, acc, lut = (np.ascontiguousarray(a, dtype=np.float32) for a in (maps, acc, lut))
    out = np.empty((M + 1, H, W, 3), np.float32)
    lib.colormap_host(maps.ctypes.data if M else None, M, H * W, acc.ctypes.data, lut.ctypes.data, out.ctypes.data)
    return out


@pytest.mark.parametrize("M", [0, 1, 3])
@pytest.mark.parametrize("kind", ["random", "constant", "boundaries", "special"])
def test_core_matches_numpy_bit_for_bit(host_lib, kind, M):
    maps, acc = colormap_case(kind, 37, 53, M, seed=M + 10)
    lut = seeded_lut(M)
    got, want = run_host(host_lib, maps, acc, lut), np_colormap(maps, acc, lut)
    assert got.shape == (M + 1, 37, 53, 3)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_special_values_follow_torch():
    """A map holding a NaN comes out as lut[0] blended with the accumulation (its min and max are NaN); an infinite
    pixel makes the range infinite, so every pixel of that map maps to 0 * inf or 0 -> lut[0]; a constant map puts
    every pixel at row 0; the accumulation image clips to the first and last rows."""
    lut = seeded_lut(5)
    maps, acc = colormap_case("special", 9, 13, 3, seed=2)
    out = np_colormap(maps, acc, lut)
    for m in range(3):
        want = lut[0] * acc[..., None] + (np.float32(1) - acc)[..., None]
        assert np.array_equal(out[1 + m], want.astype(np.float32))
    assert np.array_equal(out[0].reshape(-1, 3)[3], lut[0]) and np.array_equal(out[0].reshape(-1, 3)[5], lut[255])
    maps, acc = colormap_case("constant", 9, 13, 1, seed=2)
    assert np.array_equal(np_index(maps[0] - maps[0]), np.zeros((9, 13), np.int64))


def test_boundaries_use_every_row(host_lib):
    """The boundary case reaches all 256 rows, and the float below k / 255 lands on row k - 1 or k as fp32 rounding of
    x * 255 decides, the same in the core and the restatement."""
    maps, acc = colormap_case("boundaries", 32, 32, 1)
    idx = np_index(acc)
    assert set(np.unique(idx)) == set(range(256))
    lut = np.repeat((np.arange(256, dtype=np.float32) / 256)[:, None], 3, axis=1)
    got = run_host(host_lib, maps, acc, lut)
    assert np.array_equal(got[0][..., 0], lut[idx][..., 0])


# ---- LPIPS from a reference checkpoint -------------------------------------------------------------------------------
SLICES = {0: "net.slice1.0", 3: "net.slice2.3", 6: "net.slice3.6", 8: "net.slice4.8", 10: "net.slice5.10"}
SHIFT, SCALE = (-0.030, -0.088, -0.188), (0.458, 0.448, 0.450)


def torchvision_and_lin(seed=0):
    """Seeded weights under torchvision's AlexNet keys and the LPIPS `alex.pth` keys."""
    from presight_b200.metrics import _expected_keys
    g = torch.Generator().manual_seed(seed)
    alex, lin = {}, {}
    for k, shape in _expected_keys().items():
        (lin if k.startswith("lin") else alex)[k] = torch.randn(shape, generator=g)
    return alex, lin


def reference_checkpoint(alex, lin, prefix="_model."):
    """What a reference checkpoint holds: the model's other parameters, torchmetrics' `_LPIPS` under `lpips.net.`
    (AlexNet slices, lin layers and their `lins` aliases, the scaling layer)."""
    sd = {f"{prefix}field.mlp_head.params": torch.zeros(8), f"{prefix}lpips.total": torch.tensor(0.0)}
    for i, s in SLICES.items():
        sd[f"{prefix}lpips.net.{s}.weight"] = alex[f"features.{i}.weight"]
        sd[f"{prefix}lpips.net.{s}.bias"] = alex[f"features.{i}.bias"]
    for k in range(5):
        sd[f"{prefix}lpips.net.lin{k}.model.1.weight"] = lin[f"lin{k}.model.1.weight"]
        sd[f"{prefix}lpips.net.lins.{k}.model.1.weight"] = lin[f"lin{k}.model.1.weight"]
    sd[f"{prefix}lpips.net.scaling_layer.shift"] = torch.tensor(SHIFT)[None, :, None, None]
    sd[f"{prefix}lpips.net.scaling_layer.scale"] = torch.tensor(SCALE)[None, :, None, None]
    return sd


@pytest.mark.parametrize("prefix", ["", "_model.", "_model.module."])
def test_reference_checkpoint_packs_like_state_dicts(prefix):
    from presight_b200.metrics import LPIPS
    alex, lin = torchvision_and_lin(1)
    want = LPIPS.from_state_dicts(alex, lin, device="cpu")
    got = LPIPS.from_reference_state_dict(reference_checkpoint(alex, lin, prefix), device="cpu")
    for a, b in zip(got.conv_w + got.conv_b + got.lin, want.conv_w + want.conv_b + want.lin):
        assert torch.equal(a, b)
    # the scaling layer is optional (torchmetrics does not always persist it)
    sd = {k: v for k, v in reference_checkpoint(alex, lin, prefix).items() if "scaling_layer" not in k}
    assert torch.equal(LPIPS.from_reference_state_dict(sd, device="cpu").conv_w[2], want.conv_w[2])


def test_reference_checkpoint_rejections():
    from presight_b200.metrics import LPIPS
    alex, lin = torchvision_and_lin(2)
    good = reference_checkpoint(alex, lin)
    missing = {k: v for k, v in good.items() if k != "_model.lpips.net.net.slice4.8.bias"}
    with pytest.raises(ValueError, match=r"missing _model\.lpips\.net\.net\.slice4\.8\.bias") as e:
        LPIPS.from_reference_state_dict(missing, device="cpu")
    assert "_model.lpips.net.net.slice1.0.weight [64, 3, 11, 11]" in str(e.value)
    assert "_model.lpips.net.lin4.model.1.weight [1, 256, 1, 1]" in str(e.value)
    bad_shape = dict(good, **{"_model.lpips.net.lin2.model.1.weight": torch.zeros(384)})
    with pytest.raises(ValueError, match=r"lin2\.model\.1\.weight has shape \(384,\)"):
        LPIPS.from_reference_state_dict(bad_shape, device="cpu")
    mixed = dict(good)
    mixed["_model.module.lpips.net.net.slice3.6.bias"] = mixed.pop("_model.lpips.net.net.slice3.6.bias")
    with pytest.raises(ValueError, match="more than one prefix") as e:
        LPIPS.from_reference_state_dict(mixed, device="cpu")
    assert "_model.lpips.net.net.slice2.3.weight [192, 64, 5, 5]" in str(e.value)
    for k, v in (("shift", (-0.030, -0.088, -0.187)), ("scale", (0.458, 0.448))):
        wrong = dict(good, **{f"_model.lpips.net.scaling_layer.{k}": torch.tensor(v)[None, :, None, None]})
        with pytest.raises(ValueError, match=f"scaling_layer.{k}"):
            LPIPS.from_reference_state_dict(wrong, device="cpu")
    with pytest.raises(ValueError, match=r"missing lpips\.net\.net\.slice1\.0\.weight"):
        LPIPS.from_reference_state_dict({"field.x": torch.zeros(1)}, device="cpu")
    # a key merely ending in "lpips.net." inside a name is not a prefix
    with pytest.raises(ValueError, match="missing"):
        LPIPS.from_reference_state_dict({f"_model.xlpips.net.{k.split('lpips.net.')[1]}": v for k, v in good.items()
                                         if "lpips.net." in k}, device="cpu")
