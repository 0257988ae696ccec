"""CPU checks of LPIPS: the fp64 oracle (oracle/lpips_oracle.py) against torchvision's AlexNet, its exact properties, the
layer sizes and FLOP count the benchmark uses, and the weight packing of `presight_b200.metrics.LPIPS`."""
import pytest
import torch

from oracle import lpips_oracle as LO
from test_metrics_host import image_pair

CHANNELS = (64, 192, 384, 256, 256)


def alexnet_state_dict(seed=0):
    """torchvision's AlexNet at its own (seeded) random init: the keys and layouts of the pretrained checkpoint."""
    tv = pytest.importorskip("torchvision")
    torch.manual_seed(seed)
    return tv.models.alexnet(weights=None).state_dict()


def lin_state_dict(seed=0):
    """LPIPS v0.1 `lin` layers with non-negative weights (as the trained ones are)."""
    g = torch.Generator().manual_seed(seed)
    return {f"lin{k}.model.1.weight": torch.rand(1, c, 1, 1, generator=g) * (2.0 / c) for k, c in enumerate(CHANNELS)}


def test_oracle_features_are_torchvision_alexnet_slices():
    tv = pytest.importorskip("torchvision")
    sd = alexnet_state_dict(1)
    net = tv.models.alexnet(weights=None)
    net.load_state_dict(sd)
    feats = net.features.double().eval()
    pred, _ = image_pair("random", 67, 90, seed=4)
    x = LO.scaled_input(pred)
    assert x.shape == (1, 3, 67, 90) and x.dtype == torch.float64
    ours = LO.features(x, sd)
    with torch.no_grad():
        for f, end in zip(ours, (2, 5, 8, 10, 12)):
            want = feats[:end](x.clone())
            assert f.shape == want.shape
            torch.testing.assert_close(f, want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("kind", ["random", "smooth", "edge"])
def test_oracle_properties(kind):
    sd, lin = alexnet_state_dict(2), lin_state_dict(2)
    a, b = image_pair(kind, 45, 63, seed=5)
    total, per_layer = LO.lpips(a, b, sd, lin)
    assert total > 0 and len(per_layer) == 5 and all(v >= 0 for v in per_layer)
    assert sum(per_layer) == pytest.approx(total, rel=1e-15)
    assert LO.lpips(a, a, sd, lin)[0] == 0.0
    assert LO.lpips(b, a, sd, lin)[0] == pytest.approx(total, rel=1e-14)


def test_layer_shapes_and_flops():
    from presight_b200 import metrics
    assert metrics.lpips_layer_shapes(900, 1600) == [(224, 399), (111, 199), (55, 99), (55, 99), (55, 99)]
    assert round(metrics.lpips_flops(900, 1600) / 1e9, 3) == 41.008
    assert metrics.lpips_layer_shapes(31, 31)[-1] == (1, 1)
    with pytest.raises(ValueError, match="31 x 31"):
        metrics.lpips_layer_shapes(30, 40)
    # the oracle's feature maps have the same sizes
    sd = alexnet_state_dict(0)
    for H, W in ((31, 31), (33, 47), (64, 50)):
        fs = LO.features(LO.scaled_input(torch.rand(H, W, 3)), sd)
        assert [tuple(f.shape[2:]) for f in fs] == metrics.lpips_layer_shapes(H, W)
        assert [f.shape[1] for f in fs] == list(CHANNELS)


def test_tf32_round_is_nearest_ties_away():
    from presight_b200.metrics import tf32_round
    x = torch.tensor([1.0, 1.0 + 2 ** -11, 1.0 + 2 ** -11 - 2 ** -20, 1.0 + 2 ** -10, -(1.0 + 2 ** -11), 0.0])
    want = torch.tensor([1.0, 1.0 + 2 ** -10, 1.0, 1.0 + 2 ** -10, -(1.0 + 2 ** -10), 0.0])
    got = tf32_round(x)
    assert torch.equal(got, want)
    assert torch.equal(tf32_round(got), got)                       # TF32 values are fixed points
    r = torch.randn(10000, generator=torch.Generator().manual_seed(0))
    assert float(((tf32_round(r) - r).abs() / r.abs()).max()) <= 2 ** -11


def test_packing_round_trips_on_cpu():
    from presight_b200.metrics import LPIPS, tf32_round
    sd, lin = alexnet_state_dict(3), lin_state_dict(3)
    sd_tf32 = {k: tf32_round(v) if k.endswith("weight") else v for k, v in sd.items()}
    net = LPIPS.from_state_dicts(sd_tf32, lin, device="cpu")
    for w, c in zip(net.conv_w, CHANNELS):
        assert w.shape[0] == c and w.shape[1] % 32 == 0 and w.is_contiguous()
    assert [w.shape[1] for w in net.conv_w] == [384, 1600, 1728, 3456, 2304]
    assert torch.count_nonzero(net.conv_w[0][:, 363:]) == 0                       # zero K padding of conv1
    alex, lin2 = net.unpack()
    assert set(alex) == {k for k in sd if k.startswith("features.")} and set(lin2) == set(lin)
    for k, v in alex.items():
        assert torch.equal(v, sd_tf32[k]), k
    for k, v in lin2.items():
        assert torch.equal(v, lin[k]), k
    # (ky, kx, ci) is the packed K order
    w = sd_tf32["features.3.weight"]
    assert torch.equal(net.conv_w[1][5, (2 * 5 + 1) * 64 + 7], w[5, 7, 2, 1])
    # unrounded weights are packed rounded to TF32
    net2 = LPIPS.from_state_dicts(sd, lin, device="cpu")
    assert torch.equal(net2.unpack()[0]["features.6.weight"], sd_tf32["features.6.weight"])


def test_bad_weights_name_the_key():
    from presight_b200.metrics import LPIPS
    sd, lin = alexnet_state_dict(0), lin_state_dict(0)
    missing = {k: v for k, v in sd.items() if k != "features.8.bias"}
    with pytest.raises(ValueError, match=r"missing features\.8\.bias") as e:
        LPIPS.from_state_dicts(missing, lin, device="cpu")
    assert "lin4.model.1.weight [1, 256, 1, 1]" in str(e.value) and "features.0.weight [64, 3, 11, 11]" in str(e.value)
    flat = dict(lin, **{"lin2.model.1.weight": lin["lin2.model.1.weight"].reshape(384)})
    with pytest.raises(ValueError, match=r"lin2\.model\.1\.weight has shape \(384,\)"):
        LPIPS.from_state_dicts(sd, flat, device="cpu")
    with pytest.raises(ValueError, match=r"missing lin0\.model\.1\.weight"):
        LPIPS.from_state_dicts(sd, {"lin0.weight": lin["lin0.model.1.weight"]}, device="cpu")
    # classifier keys are ignored
    LPIPS.from_state_dicts({k: v for k, v in sd.items() if k.startswith("features.")}, lin, device="cpu")
