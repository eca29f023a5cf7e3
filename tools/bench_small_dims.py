"""Timing of the small and non-power-of-two lengths the reference's drivers use (SURVEY.md 8(f) item 4):
python tools/bench_small_dims.py"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "clifford-vae_b200")]
import torch
from clifford_b200 import _lib
dev = torch.device("cuda:0"); _lib.ensure_device(dev); _raw = _lib.load(); st = torch.cuda.current_stream().cuda_stream


class _Checked:
    """every C-ABI call's status is checked: a refused launch must not read as a fast one"""
    def __getattr__(self, name):
        fn = getattr(_raw, name)
        def call(*a):
            _lib.check(fn(*a), name)
        return call


lib = _Checked()
PEAK = 6548.8


def timeit(fn, reps=10):
    for _ in range(3): fn()
    torch.cuda.synchronize(); a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize(); return a.elapsed_time(b) / reps


# power-of-two small d (per-token latents of cnn/cliffordar_model.py: D = 16 ..): the register/shared-memory FFT path
for d in (16, 32, 64, 128, 256):
    B = (1 << 28) // (12 * d)
    loc = torch.randn(B, d, device=dev); kap = torch.rand(B, device=dev) * 9 + 0.1; z = torch.empty(B, 2 * d, device=dev); kl = torch.empty(B, device=dev)
    ms = timeit(lambda: lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0, z.data_ptr(), None, None, kl.data_ptr(), None, B, d, st))
    gb = B * (12 * d + 8) / ms / 1e6
    print(f"clifford fwd rng      d={d:5d} B={B:8d} {ms:8.3f} ms {B/ms*1e3:.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
    del loc, z
# the reference's default MNIST dims (mnist/mnist_clifpws.py:713-719): n = 2d is not a power of two -> direct-DFT kernels
for d in (2, 5, 10, 20, 40, 64, 100, 200, 300):
    B = 1 << 16
    loc = torch.randn(B, d, device=dev); kap = torch.rand(B, device=dev) * 9 + 0.1; z = torch.empty(B, 2 * d, device=dev); kl = torch.empty(B, device=dev)
    ms = timeit(lambda: lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0, z.data_ptr(), None, None, kl.data_ptr(), None, B, d, st))
    gb = B * (12 * d + 8) / ms / 1e6
    print(f"clifford fwd rng      d={d:5d} B={B:8d} {ms:8.3f} ms {B/ms*1e3:.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%  (direct DFT, n={2*d}, {"row tiles" if 2 * d <= 512 else "one CTA per row"})")
    if d <= 256:
        # backward and log_prob of the same rows
        gz = torch.randn(B, 2 * d, device=dev); tps = torch.rand(B, d, device=dev) * 0.98 + 0.01; dl = torch.empty(B, d, device=dev); dk = torch.empty(B, device=dev)
        ms = timeit(lambda: lib.cvb_clifford_ps_rsample_backward(gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, tps.data_ptr(), dl.data_ptr(), dk.data_ptr(), B, d, st))
        gb = B * (20 * d + 8) / ms / 1e6
        print(f"clifford bwd          d={d:5d} B={B:8d} {ms:8.3f} ms {B/ms*1e3:.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
        lp = torch.empty(B, device=dev)
        ms = timeit(lambda: lib.cvb_clifford_ps_log_prob(z.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, lp.data_ptr(), None, None, None, B, d, st))
        gb = B * (12 * d + 8) / ms / 1e6
        print(f"clifford log_prob     d={d:5d} B={B:8d} {ms:8.3f} ms {B/ms*1e3:.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
        del gz, tps, dl
    del loc, z
for d in (32, 64, 128, 256, 512):
    N = (1 << 28) // (12 * d)
    a = torch.randn(N, d, device=dev); b = torch.randn(N, d, device=dev); o = torch.empty(N, d, device=dev)
    ms = timeit(lambda: lib.cvb_vsa_bind(a.data_ptr(), b.data_ptr(), o.data_ptr(), N, N, N, d, 0, st))
    gb = N * 12 * d / ms / 1e6
    print(f"bind                  d={d:5d} N={N:8d} {ms:8.3f} ms {N/ms*1e3:.3e} vec/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
    del a, b, o
# non-power-of-two VSA lengths: heat-map dims 144 / 484 (scripts/binding_depth_heatmap.py:101), d+1 latents 41 / 129 / 513
# (mnist/mnist_clifpws.py:235-236), odd sizes
for d in (4, 10, 21, 41, 80, 100, 129, 144, 484, 513, 1000, 3000):
    N = max(4096, (1 << 26) // (12 * d))
    a = torch.randn(N, d, device=dev); b = torch.randn(N, d, device=dev); o = torch.empty(N, d, device=dev)
    for name, mode in (("bind", 0), ("unbind inv", 1), ("unbind deconv", 2)):
        ms = timeit(lambda: lib.cvb_vsa_bind(a.data_ptr(), b.data_ptr(), o.data_ptr(), N, N, N, d, mode, st), reps=5)
        gb = N * 12 * d / ms / 1e6
        print(f"{name:14s} d={d:5d} N={N:8d} {ms:8.3f} ms {N/ms*1e3:.3e} vec/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
    del a, b, o
