"""Generate tests/golden/parity_full.pt, what tests/test_reference_parity_gpu.py compares against, by running the
UNMODIFIED reference on a B200.

Needs a GPU and the reference tree where baseline/reference_arm.py looks for it (tools/stage_reference.py):
    python tests/golden/make_golden_parity.py [OUT]        (default: tests/golden/parity_full.pt)

One step of the reference's own SRModel at BASELINE config 2's full size, from its own initial weights for torch
seed 0 (network_G.init_scale 0.3) and a seeded batch, twice: fp32 with TF32 off (the ground truth) and under bf16
autocast (the reference's own reduced-precision path).  The fixture keeps
  g_fingerprint, d_fingerprint   SHA-256 of the initial weights, to confirm that the test regenerates them exactly
  logs32, logs16    the log_dict of each path
  logits            D(fake) / D(real) logits of each path, repeated from the initial D on the path's own SR
  sr32_sample       a seeded sample of the fp32 SR output; sr_err16 = rel-L2 of the bf16 SR over all of it
  stats_G, stats_D  one row per state_dict key (g_shapes / d_shapes order): fp32 gradient norm, bf16 gradient
                    norm, bf16 gradient rel-L2 (NaN where the fp32 gradient is zero), sign flips of the bf16 path's
                    first Adam update, rel-L2 of its BatchNorm running-statistic change, num_batches_tracked
The fp32 step is also recomputed with oracle/esrgan_oracle.py, as the test does, and must agree with the reference's
to fp32 rounding; the agreement is printed and stored under oracle_check.
"""
import math
import os
import sys
from collections import OrderedDict

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

from baseline import reference_arm as RA  # noqa: E402
import test_reference_parity_gpu as T  # noqa: E402

NB, HR, BS = 23, 256, 16
INIT_SEED, G_INIT_SCALE, BATCH_SEED = 0, 0.3, 1234
SR_SAMPLE_SEED, SR_SAMPLE_SIZE = 5, 8192
ZERO_ABS = 1e-9


def reference_run(precision, g_sd, d_sd, batch):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = False
    model, _ = RA.create_reference_model(torch_home=T.TORCH_HOME, seed=INIT_SEED, precision=precision, nb=NB, hr_size=HR,
                                         use_gan=True, use_fea=True, pixel_weight=1e-2, feature_weight=1.0,
                                         gan_weight=5e-3, gpu=True, batch_size=BS, init_scale=G_INIT_SCALE)
    out = {"grads": {}, "g0": T._state(RA.unwrap(model.netG).state_dict()), "d0": T._state(RA.unwrap(model.netD).state_dict())}
    if g_sd is not None:
        RA.unwrap(model.netG).load_state_dict(g_sd)
        RA.unwrap(model.netD).load_state_dict(d_sd)
    T._snapshot_hooks(model, out["grads"])
    model.feed_data(batch)
    model.optimize_parameters(1)
    out["logs"] = OrderedDict((k, float(v)) for k, v in model.log_dict.items())
    out["sr"] = model.fake_H.detach().float().clone()
    out["g1"], out["d1"] = T._state(RA.unwrap(model.netG).state_dict()), T._state(RA.unwrap(model.netD).state_dict())
    del model
    torch.cuda.empty_cache()
    return out


def discriminator_logits(r32, r16, d_sd, batch):
    from models.modules.architectures import discriminators as ref_disc
    dref = ref_disc.Discriminator_VGG(HR, 3, 64).cuda()
    out = OrderedDict()
    with torch.no_grad():
        for key, x32, x16 in (("fake", r32["sr"], r16["sr"]), ("real", batch["HR"], batch["HR"])):
            dref.load_state_dict(d_sd); dref.train()
            l32 = dref(x32).float().flatten().double().cpu()
            dref.load_state_dict(d_sd)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                l16 = dref(x16).float().flatten().double().cpu()
            out[key] = (l32, l16)
    return out


def stats(sd0, r32, r16, net, k1):
    rows = []
    for k, p0 in sd0.items():
        row = [math.nan] * 6
        g32 = r32["grads"][net].get(k)
        if g32 is not None:
            g16 = r16["grads"][net][k]
            row[T.N32], row[T.N16] = float(g32.double().norm()), float(g16.double().norm())
            if row[T.N32] > ZERO_ABS * g32.numel() ** 0.5:
                row[T.E16] = T.rel(g16, g32)
        if not p0.is_floating_point():
            row[T.COUNT32] = int(r32[k1][k])
        else:
            u32 = r32[k1][k].double() - p0.double()
            if "running_" in k:
                row[T.BN_ERR16] = T.rel(r16[k1][k].double() - p0.double(), u32)
            else:
                row[T.FLIPS16] = int(((r16[k1][k].double() - p0.double() - u32).abs() > T.LR).sum())
        rows.append(row)
    return torch.tensor(rows, dtype=torch.float64)


def oracle_agreement(o32, r32, sd0s):
    """largest relative deviation of the oracle's fp32 step from the reference's, per kind of output (gradients
    that are 0 in exact arithmetic left out), and the sign flips between their first Adam updates"""
    out = OrderedDict()
    out["logs"] = max(abs(o32["logs"][0][k] - v) / abs(v) for k, v in r32["logs"].items() if k not in ("D_real", "D_fake"))
    out["sr"] = T.rel(o32["sr"], r32["sr"])
    out["grads"] = max(T.rel(o32["grads"][n][k], g) for (n, sd0) in (("G", sd0s[0][0]), ("D", sd0s[1][0]))
                       for k, g in r32["grads"][n].items() if not T.feeds_batchnorm(k, sd0))
    flips = 0
    for sd0, k1 in sd0s:
        for k, p0 in sd0.items():
            if p0.is_floating_point() and "running_" not in k:
                flips += int(((o32[k1][k].double() - r32[k1][k].double()).abs() > T.LR).sum())
    out["update_sign_flips"] = flips
    return out


def main(path):
    fx = OrderedDict(nb=NB, hr=HR, bs=BS, init_seed=INIT_SEED, g_init_scale=G_INIT_SCALE, batch_seed=BATCH_SEED,
                     sr_sample_seed=SR_SAMPLE_SEED, sr_sample_size=SR_SAMPLE_SIZE)
    batch = T._batch(BS, HR, BATCH_SEED)
    r32 = reference_run("fp32", None, None, batch)
    g_sd, d_sd = r32["g0"], r32["d0"]
    r16 = reference_run("bf16", g_sd, d_sd, batch)
    for net, sd in (("g", g_sd), ("d", d_sd)):
        fx[net + "_shapes"] = OrderedDict((k, tuple(v.shape)) for k, v in sd.items())
        fx[net + "_fingerprint"] = T.fingerprint(sd)
    for a, b in zip(T._weights(fx), (g_sd, d_sd)):
        assert all(torch.equal(v, b[k]) for k, v in a.items())
    fx["logs32"], fx["logs16"] = r32["logs"], r16["logs"]
    fx["logits"] = discriminator_logits(r32, r16, d_sd, batch)
    for key, name in (("fake", "D_fake"), ("real", "D_real")):
        l32 = fx["logits"][key][0]
        assert abs(float(l32.mean()) - r32["logs"][name]) <= 1e-4 * abs(r32["logs"][name]) + 1e-7, name
    fx["sr32_sample"] = r32["sr"].flatten()[T._sr_sample_index(r32["sr"].numel(), fx)].cpu()
    fx["sr_err16"] = T.rel(r16["sr"], r32["sr"])
    fx["stats_G"] = stats(g_sd, r32, r16, "G", "g1")
    fx["stats_D"] = stats(d_sd, r32, r16, "D", "d1")
    print("reference fp32 log_dict", dict(r32["logs"]))
    print("reference bf16 log_dict", dict(r16["logs"]))
    print("bf16 SR rel-L2 %.4e, fp32 SR std %.4e" % (fx["sr_err16"], float(r32["sr"].std())))
    o32 = T._oracle_run(g_sd, d_sd, batch, NB, HR)
    fx["oracle_check"] = oracle_agreement(o32, r32, ((g_sd, "g1"), (d_sd, "d1")))
    print("oracle fp32 step vs reference fp32 step:", dict(fx["oracle_check"]))
    assert fx["oracle_check"]["logs"] < 1e-4 and fx["oracle_check"]["sr"] < 1e-4 and fx["oracle_check"]["grads"] < 1e-3, \
        fx["oracle_check"]
    torch.save(fx, path)
    print("%s: %d KiB" % (path, os.path.getsize(path) // 1024))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "parity_full.pt"))
