"""SURVEY.md T10(i) on hardware (needs >= 2 B200s: `python -m pytest tests/test_multi_gpu.py -m gpu` on a machine with two).

Two ranks, one process per GPU, NCCL.  Each rank runs two ESRGAN G/D steps on its own shard of the batch:
  * the gradients a rank holds BEFORE the exchange, and its log_dict, are bit-identical to a single-process run of
    the same shard (same weights, no process group) -- the kernels are deterministic, so "equal" means equal;
  * the exchanged gradient equals the mean of the two ranks' local gradients (fp32 rounding of one add + scale);
  * after the steps both ranks hold identical parameters, and they differ from the single-shard run's.
The single-process path itself is pinned to the unmodified reference by tests/test_reference_parity_gpu.py."""
import os
import socket
from collections import OrderedDict

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _opt(vgg_path):
    return {"model": "sr", "scale": 4, "is_train": True, "datasets": {"train": {"crop_size": 64}},
            "network_G": {"type": "esrgan", "nb": 2, "nf": 64, "gaussian": False, "init_scale": 0.3},
            "network_D": {"type": "discriminator_vgg"},
            "train": {"pixel_weight": 1e-2, "feature_weight": 1.0, "gan_weight": 5e-3, "gan_type": "vanilla",
                      "lr_G": 1e-4, "lr_D": 1e-4, "perceptual_opt": {"pretrained_path": vgg_path}}}


def _shard(rank, step):
    g = torch.Generator().manual_seed(1000 * rank + step)
    return {"LR": torch.rand(4, 3, 16, 16, generator=g), "HR": torch.rand(4, 3, 64, 64, generator=g)}


def _run(model, rank, steps, spy):
    logs = []
    for s in range(1, steps + 1):
        model.feed_data(_shard(rank, s))
        model.optimize_parameters(s)
        logs.append(model.get_current_log())
    model.synchronize()
    torch.cuda.synchronize()
    return logs


def _spy_local_grads(model, store):
    """record each network's flat gradient buffer right before the exchange touches it"""
    from trainner_b200.parallel import flat_buffers_of
    orig = model.exchange.all_reduce_grads

    def wrapped(net):
        key = "G" if net is model.netG else "D"
        store.setdefault(key + "_local", []).append([b.detach().clone() for b in flat_buffers_of(net)])
        orig(net)
        store.setdefault(key + "_reduced", []).append([b.detach().clone() for b in flat_buffers_of(net)])
    model.exchange.all_reduce_grads = wrapped


def _worker(rank, world, port, vgg_path, init_path, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    from trainner_b200.models.sr_model import create_model
    init = torch.load(init_path)
    # ---- (a) single-process run of this rank's shard (no process group yet)
    torch.manual_seed(0)
    solo = create_model(_opt(vgg_path), device="cuda:%d" % rank)
    solo.netG.load_state_dict(init["G"])
    solo.netD.load_state_dict(init["D"])
    solo_store = {}
    _spy_local_grads(solo, solo_store)          # world == 1: the wrapped exchange is a no-op, the spy still records
    orig_step = solo.exchange.step_async

    def step_spy(key, net, fn):                 # world == 1 never calls all_reduce_grads: call the spy explicitly
        solo.exchange.all_reduce_grads(net)
        fn()
    solo.exchange.step_async = step_spy
    solo_logs = _run(solo, rank, 2, solo_store)
    # ---- (b) the same shard inside the 2-rank job
    dist.init_process_group("nccl", rank=rank, world_size=world)
    torch.manual_seed(0)
    model = create_model(_opt(vgg_path), device="cuda:%d" % rank)
    model.netG.load_state_dict(init["G"])
    model.netD.load_state_dict(init["D"])
    store = {}
    _spy_local_grads(model, store)
    logs = _run(model, rank, 2, store)
    res = {"logs": logs, "solo_logs": solo_logs,
           "local": {k: [[t.cpu() for t in bufs] for bufs in v] for k, v in store.items()},
           "solo_local": {k: [[t.cpu() for t in bufs] for bufs in v] for k, v in solo_store.items()},
           "params": OrderedDict((k, v.detach().cpu()) for k, v in list(model.netG.state_dict().items()) +
                                 [("D." + k, v) for k, v in model.netD.state_dict().items() if v.is_floating_point()
                                  and "running" not in k]),
           "solo_params": OrderedDict((k, v.detach().cpu()) for k, v in solo.netG.state_dict().items())}
    torch.save(res, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_step_matches_single_shard_runs_and_mean_of_shards(tmp_path):
    import torch.multiprocessing as mp
    import torchvision
    from trainner_b200.models.sr_model import create_model
    vgg_path = str(tmp_path / "vgg.pth")
    torch.manual_seed(1)
    torch.save(torchvision.models.vgg19(weights=None).state_dict(), vgg_path)
    torch.manual_seed(0)
    m0 = create_model(_opt(vgg_path), device="cuda:0")
    init_path = str(tmp_path / "init.pt")
    torch.save({"G": OrderedDict((k, v.cpu()) for k, v in m0.netG.state_dict().items()),
                "D": OrderedDict((k, v.cpu()) for k, v in m0.netD.state_dict().items())}, init_path)
    del m0
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, vgg_path, init_path, str(tmp_path))) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0
    r = [torch.load(str(tmp_path / ("rank%d.pt" % i))) for i in range(2)]
    for i in range(2):
        # step 1: weights are still the common initial ones -> local gradients and losses == the single-shard run
        assert r[i]["logs"][0] == r[i]["solo_logs"][0], (r[i]["logs"][0], r[i]["solo_logs"][0])
        for key in ("G_local", "D_local"):
            for a, b in zip(r[i]["local"][key][0], r[i]["solo_local"][key][0]):
                assert torch.equal(a, b), "rank %d %s: local gradient differs from the single-shard run" % (i, key)
    for key in ("G", "D"):
        for step in range(2):
            for l0, l1, red0, red1 in zip(r[0]["local"][key + "_local"][step], r[1]["local"][key + "_local"][step],
                                          r[0]["local"][key + "_reduced"][step], r[1]["local"][key + "_reduced"][step]):
                assert torch.equal(red0, red1), "ranks disagree on the exchanged gradient"
                mean = (l0.double() + l1.double()) / 2
                err = float((red0.double() - mean).abs().max() / (mean.abs().max() + 1e-30))
                assert err < 1e-6, (key, step, err)
    for k, v in r[0]["params"].items():
        assert torch.equal(v, r[1]["params"][k]), "parameters diverged between ranks: %s" % k
    moved = sum(float((r[0]["params"][k] - r[0]["solo_params"][k]).abs().sum()) for k in r[0]["solo_params"])
    assert moved > 0, "the exchange had no effect"
