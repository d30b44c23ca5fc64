#!/usr/bin/env python
"""bench.py -- ESRGAN 4x G/D training-step throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference-cudnn] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): RRDBNet 23 blocks nf=64 + VGG19-conv5_4 perceptual loss +
Discriminator_VGG(256) vanilla RaGAN, 16 images / GPU, LR 64x64 -> HR 256x256, bf16 compute with
fp32 master weights, Adam.  One "step" = feed_data + SRModel.optimize_parameters (G update + D
update).  Synthetic data (torch.rand, seed 1234 + rank), random-init weights (no network here).

Prints ONE JSON line (rank 0): value = HR-pixels/s over all GPUs with inputs resident in HBM;
e2e = the same metric through the public API with pinned HOST batches (H2D inside the timed
region, loss read back every step); roofline = tensor-pipe roofline of the dominant kernel
(tcgen05 implicit-GEMM conv) from CUDA-event timings of every launch in one instrumented step;
cpu_baseline = the unmodified reference SRModel (baseline/_ref) on this box's host cores (bounded sample);
vs_cudnn = the unmodified reference SRModel on this GPU through PyTorch/cuDNN (bf16 autocast and native fp16 AMP).
--impl reference / reference-cudnn run ONLY the reference (they never import trainner_b200 or oracle/).
cpu_baseline and vs_cudnn are null when no reference tree is staged (tools/stage_reference.py).
--dump-outputs DIR writes what the last timed step computed (SR batch, losses, updated weights) as .npy files;
the inputs are seeded, so runs with the same arguments on two builds can be compared output for output.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

GFLOP_PER_IMAGE_STEP = 757.7  # SURVEY.md 8d / BASELINE.md 2: algorithmic conv FLOPs of one step, per image


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cudnn"])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--nb", type=int, default=23)
    ap.add_argument("--hr", type=int, default=256)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cudnn-ref", action="store_true", help="skip the in-run reference-cuDNN rows (vs_cudnn)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm_gbs": d["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


def vgg_checkpoint():
    """Seeded random-init torchvision VGG19 (no pretrained download possible offline)."""
    import torchvision
    path = os.path.join(tempfile.gettempdir(), "b200_bench_vgg19_seed7.pth")
    if not os.path.exists(path):
        g = torch.Generator().manual_seed(7)
        net = torchvision.models.vgg19(weights=None)
        sd = net.state_dict()
        for k, v in sd.items():
            if v.dim() > 1:
                fan_in = v[0].numel()
                v.copy_(torch.randn(v.shape, generator=g) * (2.0 / fan_in) ** 0.5)
            else:
                v.zero_()
        torch.save(sd, path + ".tmp%d" % os.getpid())
        os.replace(path + ".tmp%d" % os.getpid(), path)
    return path


def make_opt(args, vgg_path):
    return {"model": "sr", "scale": 4, "is_train": True, "datasets": {"train": {"crop_size": args.hr}},
            "network_G": {"type": "esrgan", "nb": args.nb, "nf": 64, "gc": 32, "gaussian": False,
                          "upsample_mode": "upconv"},
            "network_D": {"type": "discriminator_vgg"},
            "train": {"pixel_criterion": "l1", "pixel_weight": 1e-2, "feature_criterion": "l1",
                      "feature_weight": 1, "gan_type": "vanilla", "gan_weight": 5e-3, "lr_G": 1e-4, "lr_D": 1e-4,
                      "perceptual_opt": {"pretrained_path": vgg_path}}}


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def timed_steps(fn, steps, warmup, world):
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    return ms / steps


DUMP_MAX_ELEMENTS = 4 << 20   # per array (16 MiB of float32): the dump stays under 64 MiB at any batch size


def dump_outputs(model, out_dir):
    """Write what a caller of the timed step holds after its last step, so that two builds can be compared output
    for output: sr.npy (fake_H, float32), loss_<name>.npy (each log_dict value, float64) and netG_state.npy /
    netD_state.npy (every floating-point state_dict tensor after the optimizer step, flattened and concatenated in
    key order, float32).  An array of more than DUMP_MAX_ELEMENTS elements is replaced by the elements at a fixed
    seeded sample of its flattened positions, the same positions in every run with the same arguments."""
    import numpy as np
    model.synchronize()
    torch.cuda.synchronize()
    arrays = [("sr", model.fake_H.detach().float())]
    arrays += [("loss_" + k, torch.tensor(v, dtype=torch.float64)) for k, v in model.get_current_log().items()]
    for name, net in (("netG", model.netG), ("netD", model.netD)):
        if net is not None:
            arrays.append((name + "_state", torch.cat([v.detach().float().flatten() for v in net.state_dict().values()
                                                       if v.is_floating_point()])))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays:
        a = a.cpu()
        if a.numel() > DUMP_MAX_ELEMENTS:
            pick = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMENTS]
            a = a.flatten()[pick.sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def reference_batch(args, batch, device=None, seed=1234):
    gen = torch.Generator().manual_seed(seed)
    lr_img = torch.rand(batch, 3, args.hr // 4, args.hr // 4, generator=gen)
    hr_img = torch.rand(batch, 3, args.hr, args.hr, generator=gen)
    if device is not None:
        lr_img, hr_img = lr_img.to(device), hr_img.to(device)
    return {"LR": lr_img, "HR": hr_img}


def reference_model(args, gpu, precision, batch):
    """The UNMODIFIED reference SRModel (baseline/_ref/codes/models/sr_model.py:17) built through the
    reference's own create_model / networks / losses for BASELINE config 2."""
    from baseline import reference_arm as RA
    if gpu:
        torch.backends.cudnn.benchmark = True   # codes/train.py:482
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):   # the reference prints its option dicts; stdout carries ONE JSON line
        model, _ = RA.create_reference_model(torch_home=os.path.join(tempfile.gettempdir(), "b200_bench_ref_torch_home"),
                                             precision=precision, nb=args.nb, hr_size=args.hr, use_gan=True,
                                             use_fea=True, pixel_weight=1e-2, feature_weight=1.0, gan_weight=5e-3,
                                             gpu=gpu, batch_size=batch)
    return model


def cpu_reference_steps(args, steps, warmup, threads=None, batch=1):
    """The reference's own CPU path (gpu_ids null, fp32) on this box's host cores: feed_data +
    optimize_parameters of the unmodified SRModel at `batch` images per step."""
    from baseline import reference_arm as RA
    # oneDNN convolutions at batch 1 stop scaling (and oversubscribe badly) past a few dozen threads
    torch.set_num_threads(threads or int(os.environ.get("B200_REF_THREADS", min(os.cpu_count(), 32))))
    model = reference_model(args, False, "fp32", batch)
    ms = RA.time_reference(model, reference_batch(args, batch), steps, warmup, cuda=False)
    return batch / (ms / 1e3), ms / 1e3, torch.get_num_threads()


def run_reference_cpu(args):
    """Driver's reference arm: the unmodified reference on the host cores.  One 16-image step is
    ~12 TFLOP (~25 s on 32 cores), so each step is a bounded sample of the workload: ONE image of the
    batch (same networks, losses and sizes), K timed steps after W warm-ups."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ips, dt, threads = cpu_reference_steps(args, args.steps, args.warmup)
    val = ips * args.hr * args.hr
    sample = "1 image per step (bounded sample of the %d-image step), %d timed steps after %d warm-ups, fp32" % (
        args.batch, args.steps, args.warmup)
    line = {"impl": "reference", "metric": "hr_pixels_per_sec", "value": val, "unit": "HR-px/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "images_per_sec": ips,
            "config": {"workload": "ESRGAN 4x G/D step: RRDBNet nb=%d nf=64 + VGG19 conv5_4 L1 + Discriminator_VGG(%d) "
                                   "RaGAN, L1 pixel; LR %d^2 -> HR %d^2 -- unmodified reference SRModel on CPU" %
                                   (args.nb, args.hr, args.hr // 4, args.hr),
                       "global_batch": 1, "per_gpu_batch": 1, "parallelism": "cpu"},
            "cpu_baseline": {"value": val, "unit": "HR-px/s", "cores": threads, "kind": "reference", "sample": sample},
            "e2e": {"value": val, "unit": "HR-px/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            # this arm runs the reference only: neither the product package nor the oracle may be in the process
            "loaded": {m: any(k == m or k.startswith(m + ".") for k in sys.modules) for m in ("trainner_b200", "oracle")}}
    assert not any(line["loaded"].values()), line["loaded"]
    print(json.dumps(line))


def time_reference_cudnn(args, precision, steps, warmup):
    """ms/step of the unmodified reference SRModel on this GPU through stock PyTorch/cuDNN
    (gpu_ids [0], cudnn.benchmark as in codes/train.py:482).  precision: 'bf16' (bf16 autocast),
    'amp' (the reference's native fp16 autocast + GradScaler, base_model.py:736-744) or 'fp32'."""
    from baseline import reference_arm as RA
    model = reference_model(args, True, precision, args.batch)
    batch = reference_batch(args, args.batch, device="cuda")
    ms = RA.time_reference(model, batch, steps, warmup, cuda=True)
    del model
    torch.cuda.empty_cache()
    return ms


def run_reference_cudnn(args):
    """Context rows (not the driver's reference arm): what the reference itself does on a B200."""
    rows = {}
    for prec in ("bf16", "amp", "fp32"):
        ms = time_reference_cudnn(args, prec, max(args.steps, 50) if prec != "fp32" else 10,
                                  max(args.warmup, 20) if prec != "fp32" else 5)
        rows[prec] = {"ms_per_step": ms, "images_per_sec": args.batch / (ms / 1e3)}
    ms = rows["bf16"]["ms_per_step"]
    ips = args.batch / (ms / 1e3)
    print(json.dumps({"impl": "reference-cudnn", "metric": "hr_pixels_per_sec", "value": ips * args.hr ** 2,
                      "unit": "HR-px/s", "images_per_sec": ips, "ms_per_step": ms, "n_gpus": 1,
                      "steps": max(args.steps, 50), "warmup": max(args.warmup, 20), "dtype": "bf16 autocast",
                      "data": "synthetic", "rows": rows,
                      "config": {"workload": "unmodified reference SRModel via PyTorch/cuDNN, nb=%d batch %d HR %d^2" %
                                 (args.nb, args.batch, args.hr)}}))


def ncu_traffic_per_launch(tag):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from this round's committed
    `ncu --set full --cache-control none` capture (profiles/r02_ncu_full_<kernel>.txt, written by
    tools/summarize_ncu.py from tools/collect_ncu.sh's .ncu-rep); None when no capture of that kernel is committed."""
    import re
    path = os.path.join(ROOT, "profiles", "r02_ncu_full_%s.txt" % tag)
    if not os.path.exists(path):
        return None, None
    vals = [float(a) + float(b) for a, b in re.findall(r"DRAM read ([0-9.]+) MB write ([0-9.]+) MB", open(path).read())]
    if not vals:
        return None, None
    return sum(vals) / len(vals) * 1e6, "profiles/r02_ncu_full_%s.txt (mean of %d captured launches)" % (tag, len(vals))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_cpu(args)
    if args.impl == "reference-cudnn":
        return run_reference_cudnn(args)

    from trainner_b200 import _lib
    from trainner_b200.models.sr_model import create_model
    from trainner_b200.parallel import init_distributed
    import torch.distributed as dist

    world = init_distributed()
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    vgg_path = vgg_checkpoint() if rank == 0 or world == 1 else None
    if world > 1:
        dist.barrier()
        vgg_path = vgg_checkpoint()
    # seeded after vgg_checkpoint(), which draws from the global generator only when its cached file is missing:
    # the initial weights are the same whether or not an earlier run left that file behind
    torch.manual_seed(0)
    model = create_model(make_opt(args, vgg_path), device="cuda")
    gen = torch.Generator().manual_seed(1234 + rank)
    host = {"LR": torch.rand(args.batch, 3, args.hr // 4, args.hr // 4, generator=gen).pin_memory(),
            "HR": torch.rand(args.batch, 3, args.hr, args.hr, generator=gen).pin_memory()}
    dev = {k: v.cuda() for k, v in host.items()}
    counter = {"n": 0}

    def step_resident():
        counter["n"] += 1
        model.feed_data(dev)
        model.optimize_parameters(counter["n"])

    sink = {}

    def step_e2e():
        counter["n"] += 1
        model.feed_data(host)                     # pinned host -> device inside the timed region
        model.optimize_parameters(counter["n"])
        sink["log"] = model.get_current_log()     # device -> host read of the step's losses

    # every static plan is captured into a CUDA graph on its third run (runtime.Plan.run): at least 4 untimed steps keep
    # all captures out of the timed region
    args.warmup = max(args.warmup, 4)
    sampler = ClockSampler(local) if rank == 0 else None
    ms = timed_steps(step_resident, args.steps, args.warmup, world)
    if args.dump_outputs and rank == 0:
        dump_outputs(model, args.dump_outputs)
    ms_e2e = timed_steps(step_e2e, args.steps, max(1, args.warmup // 2), world)
    clocks = sampler.stop() if sampler else None

    gb = args.batch * world
    px = args.hr * args.hr
    ips, ips_e2e = gb / (ms / 1e3), gb / (ms_e2e / 1e3)
    pk = peaks()

    # ---- roofline leg: one instrumented step, CUDA events around every kernel launch of the plans
    roof = None
    cpu_base = None
    vs_cudnn = None
    if True:  # every rank runs the instrumented step (it contains the gradient all-reduce); rank 0 reports
        from trainner_b200 import runtime
        rows = []
        orig_run = runtime.Plan.run

        def timed_run(self):
            rows.extend(self.run_timed())

        runtime.Plan.run = timed_run
        detail = [] if os.environ.get("B200_BENCH_DETAIL") else None
        runtime.Plan.detail_sink = detail
        l0 = _lib.launch_count()
        try:
            step_resident()
        finally:
            runtime.Plan.run = orig_run
            runtime.Plan.detail_sink = None
        # kernels of libtrainner_b200.so per step, counted at the C entry points during this eagerly executed
        # step (the timed steps replay the same launches from CUDA graphs, which bypass the host-side counter)
        launches = (_lib.launch_count() - l0) * args.steps
        if detail is not None and rank == 0:
            grp = {}
            for tag, info, t_ms, fl in detail:
                a = grp.setdefault((tag, info), [0, 0.0, 0.0])
                a[0] += 1; a[1] += t_ms; a[2] += fl
            with open(os.environ["B200_BENCH_DETAIL"], "w") as fh:
                for (tag, info), (c, t, fl) in sorted(grp.items(), key=lambda kv: -kv[1][1]):
                    fh.write("%-26s %-44s n=%4d  %8.3f ms  %7.1f TF/s\n" % (tag, info, c, t, fl / (t * 1e-3) / 1e12 if t > 0 else 0))
        torch.cuda.synchronize()
        agg = {}
        for tag, t_ms, fl in rows:
            a = agg.setdefault(tag, [0, 0.0, 0.0])
            a[0] += 1
            a[1] += t_ms
            a[2] += fl
        total_ms = sum(a[1] for a in agg.values())
        dom = max(agg.items(), key=lambda kv: kv[1][1])
        tag, (cnt, t_ms, fl) = dom
        achieved = fl / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
        peak = pk["bf16_tflops_sustained"]
        traffic, traffic_src = ncu_traffic_per_launch(tag)
        roof = {"bound": "tensor", "kernel": tag, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu --set full, warm caches)",
                "traffic_source": traffic_src, "launches_per_step": cnt,
                "avg_launch_ms": t_ms / cnt, "share_of_kernel_time": t_ms / total_ms if total_ms else None,
                "peak_source": pk["source"] + ", sustained figure (kernel timed inside a long step)",
                "per_kernel": {k: {"launches": v[0], "ms": round(v[1], 3),
                                   "tflops": round(v[2] / (v[1] * 1e-3) / 1e12, 1) if v[1] > 0 and v[2] > 0 else None}
                               for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])},
                # algorithmic FLOPs of the reference's step (SURVEY.md 8d); the D-step re-uses the D(fake) / D(real) forwards
                # of the G-step (value-identical), so 2 x 9.123 GMAC per image are not executed
                "step_algorithmic_tflops": GFLOP_PER_IMAGE_STEP * 1e-3 * args.batch,
                "step_frac_of_peak": (GFLOP_PER_IMAGE_STEP * 1e9 * (args.batch / (ms / 1e3))) / (peak * 1e12),
                "step_executed_tflops": (GFLOP_PER_IMAGE_STEP - 2 * 2 * 9.123) * 1e-3 * args.batch,
                "step_frac_of_peak_executed": ((GFLOP_PER_IMAGE_STEP - 2 * 2 * 9.123) * 1e9 * (args.batch / (ms / 1e3))) / (peak * 1e12)}
        from baseline import reference_arm as RA
        # the reference rows run the unmodified reference, which is not part of this repository: only where a
        # reference tree has been staged (tools/stage_reference.py)
        have_ref = RA.reference_available()
        if not have_ref and world == 1 and rank == 0 and not (args.no_cpu_baseline and args.no_cudnn_ref):
            print("bench: no reference tree staged; cpu_baseline and vs_cudnn are not measured", file=sys.stderr)
        if have_ref and not args.no_cpu_baseline and world == 1 and rank == 0:
            c_ips, c_dt, threads = cpu_reference_steps(args, 6, 1)
            cpu_base = {"value": c_ips * px, "unit": "HR-px/s", "images_per_sec": c_ips, "cores": threads,
                        "kind": "reference",
                        "sample": "unmodified reference SRModel on CPU, 6 timed steps after 1 warm-up at 1 image per step "
                                  "(bounded sample of the %d-image step; nb=%d, HR %d^2), fp32" % (args.batch, args.nb, args.hr)}
        if have_ref and not args.no_cudnn_ref and world == 1 and rank == 0:
            # the reference's own GPU path on THIS B200, same config: the >= 6x target of BASELINE.json is
            # images/s of this repo over these rows (>= 20 warm-ups, >= 50 timed iterations each)
            vs_cudnn = {}
            for prec, label in (("bf16", "bf16_autocast"), ("amp", "fp16_amp_gradscaler")):
                r_ms = time_reference_cudnn(args, prec, 50, 20)
                vs_cudnn[label] = {"reference_ms_per_step": r_ms, "reference_images_per_sec": args.batch / (r_ms / 1e3),
                                   "ratio": r_ms / ms, "ratio_e2e": r_ms / ms_e2e}
            vs_cudnn["what"] = ("unmodified reference SRModel (baseline/_ref) on this GPU via PyTorch/cuDNN, "
                                "cudnn.benchmark, 20 warm-ups + 50 timed steps; ratio = reference ms / this repo's ms")
    if world > 1:
        dist.barrier()
    if rank == 0:
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        line = {"metric": "hr_pixels_per_sec", "value": ips * px, "unit": "HR-px/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "images_per_sec": ips,
                "config": {"workload": "ESRGAN 4x G/D step: RRDBNet nb=%d nf=64 + VGG19 conv5_4 L1 + Discriminator_VGG(%d) "
                                       "RaGAN, L1 pixel; LR %d^2 -> HR %d^2" % (args.nb, args.hr, args.hr // 4, args.hr),
                           "global_batch": gb, "per_gpu_batch": args.batch, "parallelism": "dp%d" % world,
                           "l2": "per-step working set (>2 GB of activations) exceeds the 126 MB L2; no explicit flush"},
                "e2e": {"value": ips_e2e * px, "unit": "HR-px/s", "images_per_sec": ips_e2e, "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * len(sink.get("log", {}))},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu_base,
                "vs_cudnn": vs_cudnn}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    # stdout carries exactly ONE JSON line: everything else that writes to file descriptor 1 while the bench runs
    # (NCCL's version banner, the reference's option dumps, library chatter from C code) goes to stderr; the
    # descriptor is restored when the process is done with everything but the JSON line, which print() buffered.
    sys.stdout.flush()
    _saved_fd = os.dup(1)
    os.dup2(2, 1)
    _buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(_buf):
            main()
    finally:
        sys.stdout.flush()
        os.dup2(_saved_fd, 1)
        os.close(_saved_fd)
    lines = [l for l in _buf.getvalue().splitlines() if l.strip()]
    for l in lines[:-1]:
        print(l, file=sys.stderr)
    if lines:
        print(lines[-1], flush=True)
