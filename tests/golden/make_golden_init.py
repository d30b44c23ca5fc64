"""SURVEY.md 9.2 T2: the reference's init_weights (networks.py:71-100, kaiming x 0.1) on the reference's own
RRDBNet / Discriminator_VGG under a fixed torch seed -> per-tensor checksums (tests/golden/init.pt).

The B200 modules must consume the RNG in exactly the same order (module iteration order, class-name
matching on 'Conv'/'Linear'/'BatchNorm2d', tensor shapes), so the same seed must give bit-identical tensors.
Run in the build container only (needs /root/reference):  python tests/golden/make_golden_init.py
"""
import math
import os
import sys
from collections import OrderedDict

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import ref_harness as R  # noqa: E402

R._install_shims("/tmp/_golden_torch_home")
import torch  # noqa: E402


def checksums(sd):
    """exactly rounded sums (math.fsum): independent of how a reduction is split across threads or vector lanes"""
    return OrderedDict((k, (math.fsum(v.double().flatten().tolist()), math.fsum(v.double().abs().flatten().tolist())))
                       for k, v in sd.items())


def main():
    from models import networks
    from models.modules.architectures import RRDBNet_arch, discriminators
    fx = OrderedDict()
    for mode in ("upconv", "pixelshuffle"):
        torch.manual_seed(1234)
        g = RRDBNet_arch.RRDBNet(3, 3, 64, 2, upsample_mode=mode, gaussian_noise=False)
        networks.init_weights(g, init_type="kaiming", scale=0.1)
        fx["G_%s" % mode] = checksums(g.state_dict())
    torch.manual_seed(4321)
    d = discriminators.Discriminator_VGG(64, 3, 64)
    networks.init_weights(d, init_type="kaiming", scale=1)
    fx["D_64"] = checksums(d.state_dict())
    torch.save(fx, os.path.join(HERE, "init.pt"))
    print({k: len(v) for k, v in fx.items()})


if __name__ == "__main__":
    main()
