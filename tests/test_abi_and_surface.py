"""CPU: the C-ABI library loads and exports every symbol include/trainner_b200.h declares; the
nn.Module surface (state_dict keys/shapes, init) matches the reference's as recorded in the golden
fixtures; the product path refuses to run without a GPU (no CPU fallback)."""
import ctypes
import math
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_library_exports_every_declared_symbol():
    from trainner_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "trainner_b200.h")).read()
    declared = set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"b200_conv_desc", "b200_wgrad_desc", "b200_pack_entry", "b200_stream_t"}
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), "missing export %s" % name
    assert set(_lib.EXPORTED_SYMBOLS) == declared
    assert lib.b200_version() >= 100


def test_ctypes_signatures_have_the_declared_arity():
    """Every entry point's ctypes argtypes list (trainner_b200/_lib.py) has as many arguments as its declaration in
    include/trainner_b200.h, pointers where the header has pointers and 64-bit integers where it has int64_t."""
    from trainner_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "trainner_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)
    checked = 0
    for name, params in re.findall(r"\bint(?:64_t)?\s+(b200_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", hdr):
        sig = _lib._SIGNATURES.get(name)
        if sig is None:
            continue
        plist = [q.strip() for q in params.split(",") if q.strip() and q.strip() != "void"]
        assert len(plist) == len(sig), "%s: header has %d parameters, ctypes %d" % (name, len(plist), len(sig))
        for q, ct in zip(plist, sig):
            is_ptr = "*" in q or q.startswith("b200_stream_t")
            if is_ptr:
                assert ct is ctypes.c_void_p or isinstance(ct, type(ctypes.POINTER(ctypes.c_int))), (name, q, ct)
            elif q.startswith("int64_t"):
                assert ct is ctypes.c_int64, (name, q, ct)
            elif q.startswith("float"):
                assert ct is ctypes.c_float, (name, q, ct)
            elif q.startswith("int32_t") or q.startswith("int "):
                assert ct is ctypes.c_int32 or ct is ctypes.c_int, (name, q, ct)
        checked += 1
    assert checked >= 25


def test_struct_layouts_match_header(tmp_path):
    """sizeof/offsetof as the C compiler sees include/trainner_b200.h == the ctypes mirrors."""
    import subprocess
    from trainner_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('''#include <stdio.h>
#include <stddef.h>
#include "trainner_b200.h"
int main(void) {
  printf("%zu %zu ", sizeof(b200_bn_finalize_entry), offsetof(b200_bn_finalize_entry, momentum));
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(b200_conv_desc), offsetof(b200_conv_desc, tap_dy),
         offsetof(b200_conv_desc, mask_slope), sizeof(b200_wgrad_desc), sizeof(b200_pack_entry),
         offsetof(b200_pack_entry, cout), sizeof(b200_chain_stage), offsetof(b200_chain_stage, out_c),
         offsetof(b200_chain_stage, act), sizeof(b200_chain_desc));
  return 0;
}''')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    want = [ctypes.sizeof(_lib.BnFinalizeEntry), _lib.BnFinalizeEntry.momentum.offset,
            ctypes.sizeof(_lib.ConvDesc), _lib.ConvDesc.tap_dy.offset, _lib.ConvDesc.mask_slope.offset,
            ctypes.sizeof(_lib.WgradDesc), ctypes.sizeof(_lib.PackEntry), _lib.PackEntry.cout.offset,
            ctypes.sizeof(_lib.ChainStage), _lib.ChainStage.out_c.offset, _lib.ChainStage.act.offset,
            ctypes.sizeof(_lib.ChainDesc)]
    assert got == want


def test_state_dict_surface_matches_reference():
    from trainner_b200.architectures import RRDBNet_arch, discriminators
    fx = torch.load(os.path.join(GOLD, "modules.pt"))
    for mode in ("upconv", "pixelshuffle"):
        net = RRDBNet_arch.RRDBNet(3, 3, 64, 2, upsample_mode=mode)
        got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
        assert list(got.items()) == [(k, tuple(v)) for k, v in fx["rrdb_%s" % mode]["shapes"].items()]
    for size in (32, 64):
        net = discriminators.Discriminator_VGG(size, 3, 64)
        got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
        assert list(got.items()) == [(k, tuple(v)) for k, v in fx["disc_%d" % size]["shapes"].items()]
    c1 = torch.load(os.path.join(GOLD, "config1.pt"))
    net = RRDBNet_arch.RRDBNet(3, 3, 64, 1)
    assert [k for k in net.state_dict()] == list(c1["g_shapes"].keys())
    full = RRDBNet_arch.RRDBNet(3, 3, 64, 23)
    assert sum(p.numel() for p in full.parameters()) == 16697987       # SURVEY.md 8a a3
    d256 = discriminators.Discriminator_VGG(256, 3, 64)
    assert sum(p.numel() for p in d256.parameters()) == 21058953      # SURVEY.md 8a a4
    assert len(d256.state_dict()) == 83


def test_init_weights_class_name_contract():
    """networks.py:41-54 matches on class names containing 'Conv'/'Linear'; scale 0.1, bias 0."""
    from trainner_b200 import networks
    torch.manual_seed(0)
    net = networks.define_G({"type": "esrgan", "nb": 1, "nf": 64, "gaussian": False})
    w = net.state_dict()["model.1.sub.0.RDB1.conv1.0.weight"]
    fan_in = 64 * 9
    assert abs(float(w.std()) - 0.1 * (2.0 / fan_in) ** 0.5) < 0.1 * 0.1 * (2.0 / fan_in) ** 0.5
    assert float(net.state_dict()["model.0.bias"].abs().max()) == 0.0
    d = networks.define_D({"type": "discriminator_vgg"}, size=32)
    assert float(d.state_dict()["features.3.weight"].min()) == 1.0


def test_init_weights_bit_identical_to_reference():
    """SURVEY.md 9.2 T2: same torch seed -> the tensors of the reference's init_weights (networks.py:71-100) on the
    reference's own modules (tests/golden/make_golden_init.py), bit for bit: the module iteration order, the
    class-name matching and every parameter shape are the reference's."""
    from trainner_b200 import networks
    from trainner_b200.architectures import RRDBNet_arch, discriminators
    fx = torch.load(os.path.join(GOLD, "init.pt"))

    def checks(sd):
        # exactly rounded sums (as make_golden_init.py records them): a float64 torch.sum splits its reduction by
        # thread count, which moves the last bit from one machine to the next
        return [(k, (math.fsum(v.double().flatten().tolist()), math.fsum(v.double().abs().flatten().tolist())))
                for k, v in sd.items()]

    for mode in ("upconv", "pixelshuffle"):
        torch.manual_seed(1234)
        g = RRDBNet_arch.RRDBNet(3, 3, 64, 2, upsample_mode=mode, gaussian_noise=False)
        networks.init_weights(g, "kaiming", 0.1)
        assert checks(g.state_dict()) == list(fx["G_%s" % mode].items()), mode
    torch.manual_seed(4321)
    d = discriminators.Discriminator_VGG(64, 3, 64)
    networks.init_weights(d, "kaiming", 1)
    assert checks(d.state_dict()) == list(fx["D_64"].items())


def test_no_cpu_fallback():
    from trainner_b200.architectures import RRDBNet_arch
    from trainner_b200 import ops
    net = RRDBNet_arch.RRDBNet(3, 3, 64, 1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(torch.rand(1, 3, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.maxpool2x2(torch.zeros(1, 4, 4, 8, dtype=torch.bfloat16))


def test_product_code_never_imports_oracle():
    pkg = os.path.join(ROOT, "trainner_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py") or f.endswith(".cu") or f.endswith(".cuh"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
