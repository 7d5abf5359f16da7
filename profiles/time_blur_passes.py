"""Time the two passes of the direct Gaussian blur (pnp_gaussian_blur) with the library's in-situ profiler: 35 background-like
binary maps per call (the per-batch background blur of configs[1]), sigma = 0.05 * max(H, W).  The 35 maps (16-43 MB) stay
in L2 between calls.  Usage:
    python profiles/time_blur_passes.py [path/to/libpnp_ovss_b200.so] [iters]
Loads the given library build (default: the package's), so two builds can be compared in alternating processes."""
import ctypes
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "pnp_ovss_b200", "libpnp_ovss_b200.so")
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 200
lib = ctypes.CDLL(path)
lib.pnp_gaussian_blur_workspace_bytes.restype = ctypes.c_size_t
lib.pnp_gaussian_blur_workspace_bytes.argtypes = [ctypes.c_int] * 3 + [ctypes.c_double]
lib.pnp_gaussian_blur.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_size_t] + [ctypes.c_int] * 3 + [ctypes.c_double, ctypes.c_int,
                                                                                                  ctypes.c_void_p]
lib.pnp_profile_kernel_name.restype = ctypes.c_char_p
V, HZ = 7, 8     # kBlurVertical, kBlurHorizontal
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)
st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
print(torch.cuda.get_device_name(0), os.path.basename(os.path.dirname(path)) or path)
for H, W in ((336, 336), (480, 640)):
    B = 35
    x = (torch.rand((B, H, W), generator=g, device=dev) > 0.7).float()
    out = torch.empty_like(x)
    mm = torch.empty((B, 2), device=dev)
    s = 0.05 * max(H, W)
    n = lib.pnp_gaussian_blur_workspace_bytes(B, H, W, s)
    ws = torch.empty(n, dtype=torch.uint8, device=dev)

    def call():
        rc = lib.pnp_gaussian_blur(x.data_ptr(), out.data_ptr(), mm.data_ptr(), ws.data_ptr(), n, B, H, W, s, 0, st)
        assert rc == 0, rc

    for _ in range(20):
        call()
    torch.cuda.synchronize()
    tot = (ctypes.c_float * 32)()
    cnt = (ctypes.c_int * 32)()
    lib.pnp_profile_start(ctypes.c_uint((1 << V) | (1 << HZ)))
    for _ in range(iters):
        call()
    torch.cuda.synchronize()
    lib.pnp_profile_stop(tot, cnt, 32)
    print("%dx%d x%d  %s %.2f us  %s %.2f us  (per call, mean of %d)" % (
        H, W, B, lib.pnp_profile_kernel_name(V).decode(), 1e3 * tot[V] / cnt[V], lib.pnp_profile_kernel_name(HZ).decode(),
        1e3 * tot[HZ] / cnt[HZ], cnt[V]))
