"""Times the wide-path kernels alone (wide_tc.cu) at the BASELINE config-5 layer shape: one layer as a one-layer
chain_tc_kernel launch, and dw_tc_kernel with the reduction of its partials."""
import ctypes, sys
sys.path.insert(0, ".")
import torch
from loma_nerf_b200 import api
ctx = api.Context(0); ctx.set_stream(torch.cuda.current_stream()); lib = ctx.lib
P = ctypes.c_void_p
lib.lnb_test_wide_gemm_bf16.argtypes = [P] * 3 + [ctypes.c_longlong, ctypes.c_int, ctypes.c_int] + [P] * 4
lib.lnb_test_wide_dw.argtypes = [P, P, ctypes.c_int, P, ctypes.c_int, ctypes.c_longlong, P, P]
for (M, N, K) in [(786432, 256, 256), (786432, 256, 64), (113664, 256, 256)]:
    A = torch.randn(M, K, device="cuda").to(torch.bfloat16); B = torch.randn(N, K, device="cuda").to(torch.bfloat16)
    bias = torch.randn(N, device="cuda")
    bits = torch.randint(-2**31, 2**31 - 1, (M, N // 32), dtype=torch.int32, device="cuda")
    bout = torch.empty_like(bits)
    C = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    for masked in (False, True):
        f = lambda: lib.lnb_test_wide_gemm_bf16(ctx.h, A.data_ptr(), B.data_ptr(), M, N, K, None if masked else bias.data_ptr(),
                                                bits.data_ptr() if masked else None, None if masked else bout.data_ptr(), C.data_ptr())
        for _ in range(3): f()
        pr = ctx.profile_dominant(lambda: [f() for _ in range(10)])
        us = pr["ms_per_launch"] * 1e3
        gb = (M * K * 2 + M * N * 2 + M * N / 8) / 1e9
        print(f"gemm bf16 masked={masked} M={M} N={N} K={K}: {us:.1f} us  {2*M*N*K/us/1e6:.1f} TFLOP/s  {gb/us*1e6:.0f} GB/s", flush=True)
    if M > 500000:
        Z = torch.randn(M, N, device="cuda").to(torch.bfloat16)
        dW = torch.empty(K, N, device="cuda"); db = torch.empty(N, device="cuda")
        f = lambda: lib.lnb_test_wide_dw(ctx.h, A.data_ptr(), K, Z.data_ptr(), N, M, dW.data_ptr(), db.data_ptr())
        for _ in range(3): f()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(10): f()
        t1.record(); torch.cuda.synchronize()
        print(f"dW + colsum + reduce rows={M} in={K} out={N}: {t0.elapsed_time(t1)*100:.1f} us per call", flush=True)
