"""Per-op timing helper (CUDA events, ~1 GiB of traffic per launch): python tools/bench_ops.py [bind|clifford|all]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "clifford-vae_b200")]
import torch
from clifford_b200 import _lib

dev = torch.device("cuda:0")
_lib.ensure_device(dev)
lib = _lib.load()
st = torch.cuda.current_stream().cuda_stream
PEAK = 6548.8


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


what = sys.argv[1] if len(sys.argv) > 1 else "all"
if what in ("bind", "all"):
    for dd in (1024, 2048, 4096, 8192, 16384):
        N = (1 << 30) // (12 * dd)
        a = torch.randn(N, dd, device=dev); b = torch.randn(N, dd, device=dev); o = torch.empty(N, dd, device=dev)
        ms = timeit(lambda: lib.cvb_vsa_bind(a.data_ptr(), b.data_ptr(), o.data_ptr(), N, N, N, dd, 0, st))
        gb = N * 12 * dd / (ms * 1e-3) / 1e9
        print(f"bind d={dd:6d} N={N:7d} {ms:8.3f} ms {N/(ms*1e-3):.3e} vec/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
        del a, b, o
if what in ("clifford", "all"):
    for B, d in ((4096, 2048), (65536, 2048), (262144, 512), (131072, 1024)):
        loc = torch.randn(B, d, device=dev); kap = torch.rand(B, device=dev) * 9.87 + 0.13
        z = torch.empty(B, 2 * d, device=dev); kl = torch.empty(B, device=dev)
        tps = torch.empty(B, d, device=dev)
        ms = timeit(lambda: lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0,
                                                        z.data_ptr(), None, None, kl.data_ptr(), None, B, d, st))
        gb = B * (12 * d + 8) / (ms * 1e-3) / 1e9
        print(f"clifford fwd rng   B={B:7d} d={d:5d} {ms:8.3f} ms {B/(ms*1e-3):.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
        tp = torch.rand(B, d, device=dev).clamp(1e-6, 1 - 1e-6); g = torch.randn(B, d, device=dev)
        ms = timeit(lambda: lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, tp.data_ptr(), g.data_ptr(), 0, 0,
                                                        z.data_ptr(), None, None, kl.data_ptr(), None, B, d, st))
        gb = B * (20 * d + 8) / (ms * 1e-3) / 1e9
        print(f"clifford fwd inject B={B:7d} d={d:5d} {ms:8.3f} ms {B/(ms*1e-3):.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}% (20d+8 B/row)")
        gz = torch.randn(B, 2 * d, device=dev); dloc = torch.empty(B, d, device=dev); dk = torch.empty(B, device=dev)
        lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0, z.data_ptr(), tps.data_ptr(), None, None, None, B, d, st)
        ms = timeit(lambda: lib.cvb_clifford_ps_rsample_backward(gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None,
                                                                 tps.data_ptr(), dloc.data_ptr(), dk.data_ptr(), B, d, st))
        gb = B * (20 * d + 8) / (ms * 1e-3) / 1e9
        print(f"clifford bwd rng   B={B:7d} d={d:5d} {ms:8.3f} ms {B/(ms*1e-3):.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}% (20d+8 B/row)")
        lp = torch.empty(B, device=dev)
        ms = timeit(lambda: lib.cvb_clifford_ps_log_prob(z.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, lp.data_ptr(), None, None, None, B, d, st))
        gb = B * (12 * d + 8) / (ms * 1e-3) / 1e9
        print(f"clifford log_prob  B={B:7d} d={d:5d} {ms:8.3f} ms {B/(ms*1e-3):.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
        del loc, z, tp, g, gz, dloc, tps
if what in ("fused", "all"):
    for B, d in ((4096, 2048), (65536, 2048), (262144, 512)):
        n = 2 * d
        loc = torch.randn(B, d, device=dev); kap = torch.rand(B, device=dev) * 9.87 + 0.13
        roles = torch.randn(B, n, device=dev) / n ** 0.5
        z = torch.empty(B, n, device=dev); out = torch.empty(B, n, device=dev); kl = torch.empty(B, device=dev)
        def sep():
            lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0, z.data_ptr(), None, None, kl.data_ptr(), None, B, d, st)
            lib.cvb_vsa_bind(z.data_ptr(), roles.data_ptr(), out.data_ptr(), B, B, B, n, 0, st)
        def fused(zp):
            return lambda: lib.cvb_clifford_ps_rsample_bind(loc.data_ptr(), kap.data_ptr(), B, None, None, 7, 0, roles.data_ptr(), B,
                                                            zp, out.data_ptr(), None, kl.data_ptr(), None, B, d, st)
        for name, fn, byts in (("separate rsample+KL, bind", sep, 36 * d + 8 + 8 * d), ("fused rsample+KL+bind (z written)", fused(z.data_ptr()), 28 * d + 12),
                               ("fused rsample+KL+bind (z skipped)", fused(None), 20 * d + 12)):
            ms = timeit(fn)
            gb = B * byts / (ms * 1e-3) / 1e9
            print(f"{name:36s} B={B:7d} d={d:5d} {ms:8.3f} ms {B/(ms*1e-3):.3e} samples/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
        del loc, roles, z, out
if what in ("sphere", "all"):
    for fam in ("ps", "vmf"):
        B, D = 1 << 18, 513
        loc = torch.nn.functional.normalize(torch.randn(B, D, device=dev), dim=-1); kap = torch.rand(B, device=dev) * 9.2 + 0.8
        z = torch.empty(B, D, device=dev); save = torch.empty(B, 2, device=dev)
        if fam == "ps":
            f = lambda: lib.cvb_powerspherical_rsample(loc.data_ptr(), kap.data_ptr(), B, None, None, 3, 0, z.data_ptr(), save.data_ptr(), B, D, st)
        else:
            f = lambda: lib.cvb_vmf_rsample(loc.data_ptr(), kap.data_ptr(), B, None, None, 0, None, 3, 0, z.data_ptr(), save.data_ptr(), B, D, st)
        ms = timeit(f)
        gb = B * (8 * D + 8) / (ms * 1e-3) / 1e9
        print(f"{fam} rsample B={B} D={D} {ms:8.3f} ms {B/(ms*1e-3):.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
if what in ("iwae", "all"):
    # IWAE latent terms (mnist/mlp_vae.py:161,181): S samples per posterior + log q(z|x) of each
    for B, d, S in ((4096, 2048, 1), (1024, 512, 10), (4096, 512, 10), (8192, 2048, 10)):
        rows = B * S
        loc = torch.randn(B, d, device=dev); kap = torch.rand(B, device=dev) * 9.87 + 0.13
        z = torch.empty(rows, 2 * d, device=dev); lp = torch.empty(rows, device=dev)
        def sep():
            lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0, z.data_ptr(), None, None, None, None, rows, d, st)
            lib.cvb_clifford_ps_log_prob(z.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, lp.data_ptr(), None, None, None, rows, d, st)
        def fused():
            lib.cvb_clifford_ps_rsample_log_prob(loc.data_ptr(), kap.data_ptr(), B, None, None, 7, 0, z.data_ptr(), lp.data_ptr(), None, None, rows, d, st)
        def plain():
            lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0, z.data_ptr(), None, None, None, None, rows, d, st)
        for name, fn in (("rsample only", plain), ("separate rsample, log_prob", sep), ("fused rsample+log_prob", fused)):
            ms = timeit(fn)
            print(f"iwae {name:28s} B={B:6d} S={S:3d} d={d:5d} {ms:8.3f} ms {rows/(ms*1e-3):.3e} samples/s")
        del loc, z, lp
if what in ("sphere_bwd", "all"):
    for fam in ("ps", "vmf"):
        B, D = 1 << 18, 513
        loc = torch.nn.functional.normalize(torch.randn(B, D, device=dev), dim=-1); kap = torch.rand(B, device=dev) * 9.2 + 0.8
        z = torch.empty(B, D, device=dev); save = torch.empty(B, 2, device=dev)
        gz = torch.randn(B, D, device=dev); dloc = torch.empty(B, D, device=dev); dk = torch.empty(B, device=dev)
        if fam == "ps":
            lib.cvb_powerspherical_rsample(loc.data_ptr(), kap.data_ptr(), B, None, None, 3, 0, z.data_ptr(), save.data_ptr(), B, D, st)
            f = lambda: lib.cvb_powerspherical_rsample_backward(gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), B, None, None, save.data_ptr(), 3, 0,
                                                                dloc.data_ptr(), dk.data_ptr(), B, D, st)
        else:
            lib.cvb_vmf_rsample(loc.data_ptr(), kap.data_ptr(), B, None, None, 0, None, 3, 0, z.data_ptr(), save.data_ptr(), B, D, st)
            f = lambda: lib.cvb_vmf_rsample_backward(gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), B, None, save.data_ptr(), 3, 0,
                                                     dloc.data_ptr(), dk.data_ptr(), B, D, st)
        ms = timeit(f)
        gb = B * (12 * D + 12) / (ms * 1e-3) / 1e9
        print(f"{fam} rsample bwd B={B} D={D} {ms:8.3f} ms {B/(ms*1e-3):.3e} rows/s {gb:7.1f} GB/s {100*gb/PEAK:5.1f}% (12D+12 B/row)")
if what in ("vsa_small", "all"):
    for dd in (1024, 4096):
        N = (1 << 30) // (8 * dd)
        a = torch.randn(N, dd, device=dev); b = torch.randn(N, dd, device=dev); o = torch.empty(N, dd, device=dev); r = torch.empty(N, device=dev)
        ws_bytes = lib.cvb_vsa_bundle_workspace_bytes(N, dd)
        ws = torch.empty(max(int(ws_bytes), 4) // 4 + 1, device=dev); od = torch.empty(dd, device=dev)
        perm = torch.randperm(dd, device=dev)
        for name, fn, byts in (
                ("cosine", lambda: lib.cvb_vsa_cosine(a.data_ptr(), b.data_ptr(), r.data_ptr(), N, N, N, dd, st), N * (8 * dd + 4)),
                ("normalize", lambda: lib.cvb_vsa_normalize(a.data_ptr(), o.data_ptr(), N, dd, st), N * 8 * dd),
                ("invert", lambda: lib.cvb_vsa_invert(a.data_ptr(), o.data_ptr(), N, dd, st), N * 8 * dd),
                ("permute", lambda: lib.cvb_vsa_permute(a.data_ptr(), perm.data_ptr(), o.data_ptr(), N, dd, 0, st), N * 8 * dd),
                ("bundle", lambda: lib.cvb_vsa_bundle(a.data_ptr(), od.data_ptr(), N, dd, 1.0, ws.data_ptr(), st), N * 4 * dd)):
            ms = timeit(fn)
            gb = byts / (ms * 1e-3) / 1e9
            print(f"{name:10s} d={dd:5d} N={N:7d} {ms:8.3f} ms {gb:7.1f} GB/s {100*gb/PEAK:5.1f}%")
        del a, b, o
