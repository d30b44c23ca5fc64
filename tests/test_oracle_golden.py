"""CPU: the oracle (oracle/esrgan_oracle.py) against the golden outputs recorded from the REAL
reference (tests/golden/make_golden.py).  fp32 on both sides -> tolerance 2e-5 relative."""
import os
from collections import OrderedDict

import pytest
import torch

from oracle import esrgan_oracle as O
from ref_harness import seeded_state

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(autouse=True)
def recorded_thread_count():
    """The fixtures were recorded with 8 intra-op threads (make_golden.py).  CPU convolutions split their reductions
    by thread count, and after an Adam step (-lr * sign(g)) that rounding shows in the SR output, so the oracle runs
    with the same count on every machine."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-30))


def test_rrdbnet_modes():
    fx = torch.load(os.path.join(GOLD, "modules.pt"))
    for mode in ("upconv", "pixelshuffle"):
        f = fx["rrdb_%s" % mode]
        sd = seeded_state(f["shapes"], f["seed"])
        with torch.no_grad():
            y = O.rrdbnet_forward(sd, f["x"], 2, mode)
        assert rel(y, f["y"]) < 2e-5


def test_discriminator_train_and_bn_stats():
    fx = torch.load(os.path.join(GOLD, "modules.pt"))
    for size in (32, 64):
        f = fx["disc_%d" % size]
        sd = seeded_state(f["shapes"], f["seed"])
        with torch.no_grad():
            y = O.discriminator_vgg_forward(sd, f["x"], size, training=True)
        assert rel(y, f["y_train"]) < 2e-5
        for k, v in f["bn_after"].items():
            if v.is_floating_point():
                assert rel(sd[k], v) < 2e-5, k
            else:
                assert int(sd[k]) == int(v) == 1
        with torch.no_grad():
            ye = O.discriminator_vgg_forward(sd, f["x"], size, training=False)
        assert rel(ye, f["y_eval"]) < 2e-5


def test_vgg19_conv5_4():
    import torchvision
    f = torch.load(os.path.join(GOLD, "modules.pt"))["vgg19"]
    shapes = OrderedDict((k, tuple(v.shape)) for k, v in torchvision.models.vgg19(weights=None).state_dict().items())
    fsd = O.torchvision_vgg_to_feature_net(seeded_state(shapes, f["tv_seed"]))
    with torch.no_grad():
        y = O.vgg19_features(fsd, f["x"])["conv5_4"]
    assert rel(y, f["conv5_4"]) < 2e-5


def _run_steps(fx):
    import torchvision
    g_sd = OrderedDict((k, v * (fx["g_gain"] if v.dim() > 1 else 1.0))
                       for k, v in seeded_state(fx["g_shapes"], fx["g_seed"]).items())
    d_sd = seeded_state(fx["d_shapes"], fx["d_seed"]) if fx["d_shapes"] is not None else None
    vgg_sd = None
    if fx["vgg_tv_seed"] is not None:
        shapes = OrderedDict((k, tuple(v.shape)) for k, v in
                             torchvision.models.vgg19(weights=None).state_dict().items())
        vgg_sd = O.torchvision_vgg_to_feature_net(seeded_state(shapes, fx["vgg_tv_seed"]))
    orc = O.ESRGANStepOracle(g_sd, fx["nb"], d_sd, fx["hr"] if d_sd is not None else None, vgg_sd,
                             pixel_weight=fx["pixel_weight"], feature_weight=1.0 if vgg_sd is not None else 0)
    for (lr_img, hr_img), ref_log in zip(fx["batches"], fx["logs"]):
        log = orc.optimize_parameters(lr_img, hr_img)
        for k, v in ref_log.items():
            assert abs(log[k] - v) <= 2e-5 * abs(v) + 1e-7, (k, log[k], v)
    with torch.no_grad():
        sr = orc.netG(fx["lr_test"])
    assert rel(sr, fx["sr_test"]) < 2e-5
    for k, (s, a) in fx["g_after"].items():
        assert abs(float(orc.g[k].detach().double().abs().sum()) - a) <= 1e-5 * a + 1e-9, k


def test_config1_three_steps():
    """BASELINE.json configs[0]: nb=1, 32x32 -> 128x128, L1 only, batch 1, CPU."""
    _run_steps(torch.load(os.path.join(GOLD, "config1.pt")))


def test_mini_config2_two_steps():
    """shrunk configs[1]: pix-l1 + fea-vgg19-l1 + RaGAN, D BatchNorm updated 4x per iteration."""
    fx = torch.load(os.path.join(GOLD, "mini2.pt"))
    _run_steps(fx)
    assert all(int(v) == 8 for k, v in fx["d_bn_after"].items() if k.endswith("num_batches_tracked"))
