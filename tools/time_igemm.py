"""Per-layer timing of the implicit-GEMM conv (csrc/conv_igemm.cu) at config-2 shapes.
    python tools/time_igemm.py            # B200_IGEMM_DEBUG=1 is honoured by the library
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from trainner_b200 import ops

SHAPES = [  # (n, h, w, cin, cout)
    (16, 256, 256, 64, 64), (16, 128, 128, 64, 128), (16, 128, 128, 128, 128), (16, 64, 64, 128, 256),
    (16, 64, 64, 256, 256), (16, 32, 32, 256, 512), (16, 32, 32, 512, 512), (16, 16, 16, 512, 512),
]
if len(sys.argv) > 1:
    SHAPES = [SHAPES[int(a)] for a in sys.argv[1:]]
torch.manual_seed(0)
for n, h, w, cin, cout in SHAPES:
    x = (torch.randn(n, h, w, cin, device="cuda") * 0.5).to(torch.bfloat16)
    wt = torch.randn(cout, cin, 3, 3, device="cuda") * 0.05
    b = torch.randn(cout, device="cuda") * 0.1
    y = ops.conv2d(x, wt, b)
    import ctypes as C
    from trainner_b200 import _lib
    from trainner_b200.runtime import make_conv_desc, taps_conv, stream_ptr
    wp = ops.pack_weight(wt, 0)
    d = make_conv_desc(n, h, w, cin, 0, cin, h, w, h, w, cout, 0, cout, taps_conv(3, 1), 9, wp.shape[1], wp.shape[2])
    P = lambda t: C.c_void_p(t.data_ptr())
    run = lambda: _lib.lib.b200_conv_igemm(C.byref(d), P(x), P(wp), P(b), None, None, None, P(y), stream_ptr())
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), wt.to(torch.bfloat16).float(), b, padding=1)
    err = float((y.float().permute(0, 3, 1, 2) - ref).norm() / ref.norm())
    # L2 flush between timed calls is pointless here: the activations (>= 33 MB in + out) stream anyway
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    fl = 2.0 * n * h * w * cin * cout * 9
    print("conv3x3 %3d -> %3d @ %dx%dx%d : %.1f us  %.0f TF/s  rel-L2 vs fp32 conv %.2e" % (cin, cout, n, h, w, ms * 1e3, fl / ms / 1e9, err))
