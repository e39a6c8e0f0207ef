"""Developer tool: time the implicit-GEMM convolution alone on the backbone's main shapes."""
import ctypes as C, sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rethinking-flow-and-diffusion-bridge-models-for-speech-enhancement_b200"))
import torch
from fdbm_b200 import _lib
lib = _lib.load(); h16 = _lib.operand_dtype()
st = lambda: torch.cuda.current_stream().cuda_stream
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
shapes = [  # T, F, C1, k, C2, Cout, residual, f32 out, sums
    (256, 256, 128, 3, 0, 128, False, False, True),    # Conv_0 level 0 (h16 out + stats)
    (256, 256, 128, 3, 0, 128, True, True, True),      # Conv_1 level 0 (residual, fp32 out + stats)
    (256, 256, 256, 3, 0, 128, False, False, True),    # up-path Conv_0 level 0
    (256, 256, 128, 3, 256, 128, False, True, True),   # up-path Conv_1 + Conv_2
    (128, 128, 128, 3, 0, 128, True, True, True),
    (64, 64, 256, 3, 0, 256, True, True, True),
    (64, 64, 512, 3, 0, 256, False, False, True),
    (32, 32, 256, 3, 0, 256, True, True, True),
    (16, 16, 256, 3, 0, 256, True, True, True),
]
shapes.append((256, 256, 64, 1, 0, 128, False, False, True))      # first conv (im2col K-block): the epilogue alone
if os.environ.get("CB_ONLY"):
    shapes = [shapes[int(i)] for i in os.environ["CB_ONLY"].split(",")]
for (T, F, C1, k, C2, Cout, res, f32o, sm) in shapes:
    x1 = torch.randn(B, T, F, C1).to(h16).cuda()
    x2 = torch.randn(B, T, F, C2).to(h16).cuda() if C2 else None
    nb = C.c_int64(); lib.fdbm_pack_conv_weights(None, C1, k, None, C2, Cout, None, C.byref(nb), None)
    wp = (torch.randn(nb.value // 2) * 0.02).to(h16).cuda()
    bias = torch.randn(Cout).cuda()
    resid = torch.randn(B, T, F, Cout).cuda() if res else None
    out = torch.empty(B, T, F, Cout, device="cuda") if f32o else None
    o16 = None if f32o else torch.empty(B, T, F, Cout, dtype=h16, device="cuda")
    sums = torch.empty(B, Cout, 2, dtype=torch.float64, device="cuda") if sm else None
    gn = len(sys.argv) > 3 and sys.argv[3] == "gn" and C2 == 0
    if gn:
        s1 = torch.stack([x1.double().sum((1, 2)), x1.double().pow(2).sum((1, 2))], -1).contiguous()
        gam = torch.ones(C1, device="cuda"); bet = torch.zeros(C1, device="cuda"); tab = torch.empty(B * C1 * 2, device="cuda")
        d = _lib.ConvDesc(n_seg=1, wpack=wp.data_ptr(), bias=bias.data_ptr(), residual=resid.data_ptr() if res else None,
                          scale=0.7071, B=B, T=T, F=F, Cout=Cout, out_f32=out.data_ptr() if f32o else None,
                          out_h16=o16.data_ptr() if o16 is not None else None, sums=sums.data_ptr() if sm else None)
        d.seg[0] = _lib.ConvSeg(in_=x1.data_ptr(), C=C1, taps=k * k, norm_tab=tab.data_ptr(), tab_stride=C1, act=1)
    def run():
        if gn:
            rc = lib.fdbm_gn_table(s1.data_ptr(), C1, None, 0, gam.data_ptr(), bet.data_ptr(), 0, B, T * F, tab.data_ptr(), None, st())
            assert rc == 0, lib.fdbm_last_error()
            rc = lib.fdbm_conv_igemm_ex(C.byref(d), st())
            assert rc == 0, lib.fdbm_last_error()
            return
        rc = lib.fdbm_conv_igemm(x1.data_ptr(), C1, k, x2.data_ptr() if C2 else None, C2, wp.data_ptr(), bias.data_ptr(), None,
                                 resid.data_ptr() if res else None, 0.7071, B, T, F, Cout, out.data_ptr() if f32o else None,
                                 o16.data_ptr() if o16 is not None else None, sums.data_ptr() if sm else None, st())
        assert rc == 0, lib.fdbm_last_error()
    for _ in range(3): run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(reps): run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    fl = 2.0 * B * T * F * Cout * (k * k * C1 + C2)
    print(("gn " if gn else "   ") + f"B={B} T={T} F={F} C1={C1} k={k} C2={C2} Cout={Cout} res={int(res)} f32={int(f32o)}: {ms*1e3:8.1f} us  {fl/ms/1e9:7.1f} TFLOP/s")
