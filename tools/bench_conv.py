"""Micro-benchmark of fod_conv2d_nhwc against cuDNN fp32 (TF32 off) on the layer shapes of the detector (development tool)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F
from faster_orefsdet_b200 import ops
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.benchmark = True
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
dev = "cuda"
shapes = [  # name, H, W, Cin, Cout, k (a name ending in "_s2": stride 2)
    ("stem3_s2", 320, 320, 64, 128, 3), ("stem2", 320, 320, 64, 64, 3), ("osa2_0", 160, 160, 128, 64, 3), ("osa2_1", 160, 160, 64, 64, 3),
    ("osa2_cat", 160, 160, 320, 112, 1), ("osa3_0", 80, 80, 112, 80, 3), ("osa3_1", 80, 80, 80, 80, 3),
    ("osa3_cat", 80, 80, 352, 256, 1), ("osa4_0", 40, 40, 256, 96, 3), ("osa4_1", 40, 40, 96, 96, 3),
    ("osa4_cat", 40, 40, 544, 384, 1), ("osa5_0", 20, 20, 384, 112, 3), ("osa5_cat", 20, 20, 720, 512, 1),
    ("fpn_out3", 80, 80, 128, 128, 3), ("fpn_lat3", 80, 80, 256, 128, 1), ("tower4", 40, 40, 128, 128, 3),
]
only = sys.argv[2].split(",") if len(sys.argv) > 2 else None
# the 3x3 layers whose input the model hands over pre-split (split hand-off): also timed with such an input, which the
# shared-memory A kernel serves (OSA5, N = 112, stays on the tensor-memory path)
PRESPLIT = {"stem3_s2", "stem2", "osa2_0", "osa2_1", "osa3_0", "osa3_1", "osa4_0", "osa4_1", "osa5_0"}


def presplit(x, amax):
    """fp32 NHWC view -> [16 x fp16 hi | 16 x fp16 lo] of x * 2^e per 16 channels (2^e from amax), as an fp32 NHWC view"""
    n, c, h, w = x.shape
    _, ex = torch.frexp(amax.reshape(-1)[:1])
    xs = x.permute(0, 2, 3, 1) * ((141 - ex.to(torch.int32)) << 23).view(torch.float32)
    hi = xs.half()
    lo = (xs - hi.float()).half()
    packed = torch.cat([hi.reshape(n, h, w, c // 16, 16), lo.reshape(n, h, w, c // 16, 16)], dim=-1)
    return packed.contiguous().view(torch.float32).reshape(n, h, w, c).permute(0, 3, 1, 2)


def timeit(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


tot_a = tot_b = 0.0
for name, H, W, cin, cout, k in shapes:
    if only and name not in only:
        continue
    x = torch.randn(B, H, W, cin, device=dev).permute(0, 3, 1, 2)
    w = torch.randn(cout, cin, k, k, device=dev) / (cin * k * k) ** 0.5
    wc = w.contiguous(memory_format=torch.channels_last)
    b = torch.randn(cout, device=dev)
    packed = ops.conv2d_pack(w)
    ax = ops.absmax(x)
    st = 2 if name.endswith("_s2") else 1
    y = ops.conv2d_nhwc(x, packed, b, cout, k, True, x_amax=ax, stride=st)
    ref = F.relu(F.conv2d(x, wc, b, padding=k // 2, stride=st))
    err = float((y - ref).abs().max()) / float(ref.abs().max())
    t_a = timeit(lambda: ops.conv2d_nhwc(x, packed, b, cout, k, True, out=y, x_amax=ax, stride=st))
    fl = 2.0 * B * (H // st) * (W // st) * cin * cout * k * k
    t_b = timeit(lambda: F.relu_(F.conv2d(x, wc, b, padding=k // 2, stride=st)))
    split = ""
    if name in PRESPLIT:
        xp = presplit(x, ax)
        if st == 1:
            fn = lambda: ops.conv2d_nhwc(xp, packed, b, cout, k, True, out=y, x_amax=ax, x_presplit=True)
        else:
            fn = lambda: ops.conv2d_nhwc_split(xp, packed, b, cout, k, y, ax, x_presplit_from=0, slice_ch=[0], stride=2)
        t_s = timeit(fn)
        same = torch.equal(fn(), ops.conv2d_nhwc(x, packed, b, cout, k, True, x_amax=ax, stride=st))
        split = f"   pre-split {t_s:7.3f} ms ({fl/t_s/1e9:6.1f}){'' if same else '  DIFFERS from the fp32 input'}"
        del xp
    tot_a += t_a
    tot_b += t_b
    print(f"{name:9s} {H}x{W} {cin}->{cout} k{k}: tc {t_a:7.3f} ms ({fl/t_a/1e9:6.1f} TFLOP/s fp32-equiv)   cudnn {t_b:7.3f} ms "
          f"({fl/t_b/1e9:5.1f})   rel err {err:.1e}{split}", flush=True)
    del x, y, ref
print(f"total: tc {tot_a:.2f} ms, cudnn {tot_b:.2f} ms")
