"""Full-size parity on the B200 against the UNMODIFIED reference: BASELINE config 2 at its real size -- RRDBNet
nb=23, 16 x 64^2 -> 256^2, Discriminator_VGG(256), VGG19 conv5_4, L1 + perceptual + vanilla RaGAN, Adam.

The reference's own SRModel (codes/models/sr_model.py:17; feed_data :115, optimize_parameters :195) was run on a B200
through PyTorch/cuDNN twice -- fp32 (TF32 off) = the ground truth, and under bf16 autocast = the reference's own
reduced-precision path, the like-for-like yardstick -- by tests/golden/make_golden_parity.py, from the reference's own
initial weights for torch seed 0 and a seeded batch.  A full step does not fit a small fixture, so
tests/golden/parity_full.pt keeps what this test compares against:
  * of the fp32 step: its log_dict, the norm of every gradient tensor and a seeded sample of its SR output.  Here the
    fp32 step is recomputed on the GPU by oracle/esrgan_oracle.py (TF32 off) and checked against those first; the
    recomputed tensors then stand in for the reference's in the element-wise checks below;
  * of the bf16 path: its error against the fp32 step per tensor (gradient rel-L2, sign flips of Adam's first
    update, BatchNorm running statistics), its SR rel-L2 and log_dict, and the D(fake) / D(real) logits of both
    paths.
trainner_b200 runs the identical step from identical weights on the identical batch.

Tolerances (no absolute floors on the scalars):
  * the log_dict scalars pix-l1, fea-vgg19-l1, l_g_gan, l_d_real, l_d_fake, D_real:
    |v - v_ref32| <= 2e-2 |v_ref32|;
  * D_fake / D_real are MEANS of 16 raw logits that nearly cancel (measured: mean -7e-3, std 7e-3), and D(fake)
    amplifies the ~1.3e-2 relative bf16 error of the SR input through ten BatchNorm layers: the reference's OWN
    bf16 path misses 2e-2 on D_fake (measured 2.5e-2).  They are therefore checked where the noise can be
    measured, per logit: the step's D(fake) / D(real) forwards are repeated from the initial weights and
    rms(logit error) of the CUDA path must be <= 1.25 (1 + 2/sqrt(16)) x that of the reference's bf16 path (the factor
    in brackets is the scatter of an rms estimated from 16 samples); the logged means must be
    within max(2e-2 |v|, 3 sigma) with sigma = rms(reference-bf16 logit error) / sqrt(16);
  * SR (fake_H): rel-L2 vs reference-fp32 <= max(1e-2, 1.25 x the reference-bf16 rel-L2);
  * every gradient tensor of G and D: rel-L2 error vs reference-fp32 <= 1.25 x the error of the reference's
    bf16 path on that tensor, x (1 + 2/sqrt(numel)) for the scatter of an rms estimated from numel samples
    (matters for the 32-/64-element biases only; fp32-rounding-level errors <= 1e-5 pass);
  * every updated parameter tensor: Adam's first update is -lr * sign(g) wherever |g| >> eps, so the error of an
    update is a COUNT of sign flips (elements whose gradient is within the rounding noise of zero); per tensor
    flips <= 1.25 x flips of the reference-bf16 path + 3 + 3 sqrt(flips_ref) (Poisson slack for small tensors),
    and over all tensors of a network flips <= 1.1 x the reference-bf16 total; BatchNorm running statistics and
    num_batches_tracked directly.
G uses network_G.init_scale 0.3 (the reference's option, networks.py:116-120): with the default
0.1 an untrained 23-block G outputs ~1e-4 and every comparison would be vacuous (SURVEY.md 8d).
"""
import hashlib
import math
import os
import sys
import tempfile
from collections import OrderedDict

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from baseline import reference_arm as RA  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "parity_full.pt")
TORCH_HOME = os.path.join(tempfile.gettempdir(), "_parity_torch_home")
LR = 1e-4
# statistics columns of fx["stats_G"] / fx["stats_D"], one row per state_dict key (NaN where a column does not apply)
N32, N16, E16, FLIPS16, BN_ERR16, COUNT32 = range(6)


def rel(a, b):
    a, b = a.detach().double().flatten(), b.detach().double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-300))


def _batch(bs, hr, seed):
    g = torch.Generator().manual_seed(seed)
    return {"LR": torch.rand(bs, 3, hr // 4, hr // 4, generator=g).cuda(),
            "HR": torch.rand(bs, 3, hr, hr, generator=g).cuda()}


def fingerprint(sd):
    """SHA-256 of every tensor's bytes in key order: equal exactly when the tensors are bit-identical"""
    h = hashlib.sha256()
    for v in sd.values():
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def _weights(fx):
    """The reference's initial weights for torch seed fx["init_seed"] (its create_model, init_scale 0.3 for G):
    trainner_b200.networks draws them bit for bit as the reference does, which the recorded fingerprints confirm."""
    from trainner_b200 import networks
    torch.manual_seed(fx["init_seed"])
    g_sd = networks.define_G({"type": "esrgan", "nb": fx["nb"], "nf": 64, "gc": 32, "gaussian": False,
                              "upsample_mode": "upconv", "init_scale": fx["g_init_scale"]}, scale=4).state_dict()
    d_sd = networks.define_D({"type": "discriminator_vgg"}, size=fx["hr"]).state_dict()
    for net, sd in (("g", g_sd), ("d", d_sd)):
        assert list(sd) == list(fx[net + "_shapes"])
        assert fingerprint(sd) == fx[net + "_fingerprint"], "initial weights differ from the reference's"
    return (OrderedDict((k, v.cuda()) for k, v in g_sd.items()), OrderedDict((k, v.cuda()) for k, v in d_sd.items()))


def _sr_sample_index(numel, fx):
    return torch.randperm(numel, generator=torch.Generator().manual_seed(fx["sr_sample_seed"]))[:fx["sr_sample_size"]]


def _state(sd):
    return OrderedDict((k, v.detach().clone()) for k, v in sd.items())


def _oracle_run(g_sd, d_sd, batch, nb, hr):
    """The fp32 step of oracle/esrgan_oracle.py on the GPU with TF32 off: gradients as each optimizer is about to
    apply them, log_dict, SR and the weights after the step."""
    from oracle import esrgan_oracle as O
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    vgg = O.torchvision_vgg_to_feature_net(torch.load(RA.make_vgg19_checkpoint(TORCH_HOME)))
    orc = O.ESRGANStepOracle(g_sd, nb, d_sd, hr, vgg, pixel_weight=1e-2, feature_weight=1.0, gan_weight=5e-3, lr=LR,
                             device=batch["LR"].device)
    grads = {}

    def hook_for(name, sd):
        def hook(opt, args, kwargs):
            grads[name] = OrderedDict((k, v.grad.detach().clone()) for k, v in sd.items() if v.grad is not None)
        return hook
    orc.opt_g.register_step_pre_hook(hook_for("G", orc.g))
    orc.opt_d.register_step_pre_hook(hook_for("D", orc.d))
    logs = OrderedDict(orc.optimize_parameters(batch["LR"], batch["HR"]))
    out = {"grads": grads, "logs": [logs], "sr": orc.fake_H.detach().float().clone(), "g1": _state(orc.g),
           "d1": _state(orc.d)}
    del orc
    torch.cuda.empty_cache()
    return out


def _snapshot_hooks(model, store):
    """record the gradients each optimizer is about to apply (optimizer_step zeroes them afterwards)"""
    def hook_for(name, net):
        def hook(opt, args, kwargs):
            store[name] = OrderedDict((k, p.grad.detach().float().clone()) for k, p in RA.unwrap(net).named_parameters()
                                      if p.grad is not None)
        return hook
    model.optimizer_G.register_step_pre_hook(hook_for("G", model.netG))
    model.optimizer_D.register_step_pre_hook(hook_for("D", model.netD))


def _b200_opt(nb, hr):
    return {"model": "sr", "scale": 4, "is_train": True, "datasets": {"train": {"crop_size": hr}},
            "network_G": {"type": "esrgan", "nb": nb, "nf": 64, "gc": 32, "gaussian": False, "upsample_mode": "upconv"},
            "network_D": {"type": "discriminator_vgg"},
            "train": {"pixel_criterion": "l1", "pixel_weight": 1e-2, "feature_criterion": "l1", "feature_weight": 1,
                      "gan_type": "vanilla", "gan_weight": 5e-3, "lr_G": LR, "lr_D": LR,
                      "perceptual_opt": {"pretrained_path": RA.make_vgg19_checkpoint(TORCH_HOME)}}}


def _b200_run(g_sd, d_sd, batch, nb, hr, steps=1):
    from trainner_b200.models.sr_model import create_model
    model = create_model(_b200_opt(nb, hr))
    model.netG.load_state_dict(g_sd)
    model.netD.load_state_dict(d_sd)
    out = {"grads": {}, "logs": []}
    _snapshot_hooks(model, out["grads"])
    for s in range(1, steps + 1):
        model.feed_data(batch)
        model.optimize_parameters(s)
        out["logs"].append(model.get_current_log())
        if s == 1:
            out["sr"] = model.fake_H.detach().float().clone()
            model.synchronize()
            out["g1"], out["d1"] = _state(model.netG.state_dict()), _state(model.netD.state_dict())
    return out


def _stats(fx, net):
    return {k: row.tolist() for k, row in zip(fx["%s_shapes" % net.lower()], fx["stats_%s" % net])}


def feeds_batchnorm(key, shapes):
    """bias of a layer followed by BatchNorm: its gradient is 0 in exact arithmetic and rounding noise in practice"""
    head, _, leaf = key.rpartition(".")
    pre, _, idx = head.rpartition(".")
    return leaf == "bias" and idx.isdigit() and "%s.%d.running_mean" % (pre, int(idx) + 1) in shapes


def _check_recomputed_fp32_step(fx, o32):
    """the oracle's fp32 step is the reference's fp32 step, to fp32 rounding: log_dict, SR sample, gradient norms
    (except the rounding noise of gradients that are 0 in exact arithmetic)"""
    problems = []
    for k, v in fx["logs32"].items():
        # D_real / D_fake are means of logits that nearly cancel: measured against the logits' own scale
        scale = float(fx["logits"]["real" if k == "D_real" else "fake"][0].abs().mean()) if k in ("D_real", "D_fake") \
            else abs(v)
        if not abs(o32["logs"][0][k] - v) <= 1e-3 * scale:
            problems.append(("oracle log", k, o32["logs"][0][k], v))
    e = rel(o32["sr"].flatten()[_sr_sample_index(o32["sr"].numel(), fx)].cpu(), fx["sr32_sample"])
    if not e <= 1e-3:
        problems.append(("oracle SR sample", e))
    for net in ("G", "D"):
        for k, row in _stats(fx, net).items():
            if k not in o32["grads"][net] or feeds_batchnorm(k, fx["%s_shapes" % net.lower()]) or \
                    not row[N32] > 1e-9 * o32["grads"][net][k].numel() ** 0.5:
                continue
            n = float(o32["grads"][net][k].double().norm())
            if not abs(n - row[N32]) <= 1e-3 * row[N32]:
                problems.append(("oracle grad norm", net, k, n, row[N32]))
    assert not problems, problems


def _compare_tensors(what, ours, stats, ref32, zero_abs):
    """per tensor: err(ours, ref32) <= 1.25 err(ref16, ref32); numerically-zero references by absolute size"""
    bad, e_all, e_ref_all = [], [], []
    for k, t32 in ref32.items():
        if not t32.is_floating_point():
            continue
        n16, e_ref = stats[k][N16], stats[k][E16]
        if math.isnan(e_ref):
            # gradient that is exactly 0 in exact arithmetic (bias in front of BatchNorm): only rounding noise
            if float(ours[k].double().norm()) > max(4.0 * n16, zero_abs * t32.numel() ** 0.5):
                bad.append((k, "zero-ref", float(ours[k].double().norm()), n16))
            continue
        e = rel(ours[k], t32)
        e_all.append(e)
        e_ref_all.append(e_ref)
        # both errors are rms estimates over numel samples: allow the estimate's own scatter on small tensors
        if e > max(1.25 * (1.0 + 2.0 / t32.numel() ** 0.5) * e_ref, 1e-5):
            bad.append((k, e, e_ref))
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    print("%s: %d tensors, median rel-err trainner_b200 %.4f | reference bf16 %.4f; worst ratio %.2f" %
          (what, len(e_all), med(e_all), med(e_ref_all), max(a / max(b, 1e-30) for a, b in zip(e_all, e_ref_all))))
    return bad


def _discriminator_logits(fx, ours, d_sd, batch):
    """The D-step's forwards (losses.py:471-478: netD(fake.detach()), netD(real)) repeated from the initial D
    weights on each path's own fake_H: reference fp32 and reference bf16 autocast as recorded, trainner_b200 here."""
    from trainner_b200.architectures import discriminators as b200_disc
    db = b200_disc.Discriminator_VGG(fx["hr"], 3, 64).cuda()
    out = {}
    with torch.no_grad():
        for key, xb in (("fake", ours["sr"]), ("real", batch["HR"])):
            db.load_state_dict(d_sd); db.train()
            lb = db(xb).float().flatten().double().cpu()
            l32, l16 = fx["logits"][key]
            out[key] = (l32, l16, lb)
    return out


def test_full_size_step_vs_unmodified_reference():
    fx = torch.load(GOLDEN)
    batch = _batch(fx["bs"], fx["hr"], fx["batch_seed"])
    g_sd, d_sd = _weights(fx)
    r32 = _oracle_run(g_sd, d_sd, batch, fx["nb"], fx["hr"])
    _check_recomputed_fp32_step(fx, r32)
    ours = _b200_run(g_sd, d_sd, batch, fx["nb"], fx["hr"])
    logs32, logs16 = fx["logs32"], fx["logs16"]
    # ---- the 7 log_dict scalars, relative, no floor
    assert list(ours["logs"][0].keys()) == list(logs32.keys())
    rows = []
    for k, v in logs32.items():
        rows.append((k, v, logs16[k], ours["logs"][0][k]))
    print("log_dict (reference fp32 | reference bf16 | trainner_b200):")
    for k, a, b, c in rows:
        print("  %-14s % .6e  % .6e (rel %.2e)  % .6e (rel %.2e)" % (k, a, b, abs(b - a) / abs(a), c, abs(c - a) / abs(a)))
    problems = []
    for k, a, b, c in rows:
        if k in ("D_real", "D_fake"):
            continue   # checked per logit below
        if not abs(c - a) <= 2e-2 * abs(a):
            problems.append(("log", k, a, c))
    # ---- D_real / D_fake: repeat the D-step's forwards (initial D weights, the step's own fake_H) per logit
    logit_rows = _discriminator_logits(fx, ours, d_sd, batch)
    for name, key in (("D_fake", "fake"), ("D_real", "real")):
        l32, l16, lb = logit_rows[key]
        e16, eb = float((l16 - l32).pow(2).mean().sqrt()), float((lb - l32).pow(2).mean().sqrt())
        sigma = e16 / (l32.numel() ** 0.5)
        a, c = logs32[name], ours["logs"][0][name]
        print("%s logits: mean %.4e std %.3e | rms error reference-bf16 %.3e, trainner_b200 %.3e | logged mean off by "
              "%.3e (%.1f sigma)" % (name, float(l32.mean()), float(l32.std()), e16, eb, abs(c - a), abs(c - a) / sigma))
        assert abs(float(l32.mean()) - a) <= 1e-4 * abs(a) + 1e-7, "the repeated forward must reproduce the logged mean"
        if not eb <= 1.25 * (1.0 + 2.0 / l32.numel() ** 0.5) * e16:   # rms over 16 logits: +-18 % scatter of the estimate
            problems.append(("logits", name, eb, e16))
        if not abs(c - a) <= max(2e-2 * abs(a), 3.0 * sigma):
            problems.append(("log", name, a, c, sigma))
    # ---- SR
    e_sr, e_sr16 = rel(ours["sr"], r32["sr"]), fx["sr_err16"]
    print("SR rel-L2: trainner_b200 %.4e | reference bf16 %.4e; SR std %.3e" % (e_sr, e_sr16, float(r32["sr"].std())))
    assert float(r32["sr"].std()) > 1e-2, "degenerate generator output (init_scale not applied?)"
    if not e_sr <= max(1e-2, 1.25 * e_sr16):
        problems.append(("sr", e_sr, e_sr16))
    # ---- gradients, every tensor
    for net in ("G", "D"):
        bad = _compare_tensors("grad " + net, ours["grads"][net], _stats(fx, net), r32["grads"][net], 1e-9)
        if bad:
            problems.append(("grad " + net, len(bad), bad[:8]))
    # ---- every updated parameter tensor (sign flips of Adam's first update) and the BatchNorm running statistics
    for net, sd0, k1 in (("G", g_sd, "g1"), ("D", d_sd, "d1")):
        stats = _stats(fx, net)
        tot_o = tot_r = 0
        for k, p0 in sd0.items():
            if not p0.is_floating_point():
                assert int(ours[k1][k]) == int(r32[k1][k]) == int(stats[k][COUNT32]), k   # num_batches_tracked
                continue
            u32 = r32[k1][k].double() - p0.double()
            if "running_" in k:
                eo, er = rel(ours[k1][k].double() - p0.double(), u32), stats[k][BN_ERR16]
                if not eo <= max(1.25 * er, 1e-5):
                    problems.append(("bn stat", k, eo, er))
                continue
            fo = int(((ours[k1][k].double() - p0.double() - u32).abs() > LR).sum())
            fr = int(stats[k][FLIPS16])
            tot_o += fo
            tot_r += fr
            if fo > 1.25 * fr + 3 + 3 * fr ** 0.5:
                problems.append(("update " + net, k, fo, fr, p0.numel()))
        n_el = sum(v.numel() for v in sd0.values() if v.is_floating_point())
        print("update %s: sign flips of Adam's first update vs reference fp32: trainner_b200 %d | reference bf16 %d of %d "
              "elements" % (net, tot_o, tot_r, n_el))
        if tot_o > 1.1 * tot_r + 10:
            problems.append(("update total " + net, tot_o, tot_r))
    assert not problems, problems
