"""Per-op timing of the von Mises torus latent (CUDA events): forward with the offsets saved, backward, log_prob.
python tools/bench_vm_torus.py.  % of the HBM roofline on algorithmic bytes per row: forward with phi saved 16d+8
(loc read, z + phi written, entropy), backward 20d+8 (grad_z, loc, phi read, dloc written, dkappa), log_prob 12d+8."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "clifford-vae_b200")]
import torch
from clifford_b200 import _lib

dev = torch.device("cuda:0")
_lib.ensure_device(dev)
lib = _lib.load()
st = torch.cuda.current_stream().cuda_stream
PEAK = 7700.0      # GB/s, HBM3e of one B200 (data sheet)


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


print(torch.cuda.get_device_name(0))
for B, d in ((4096, 2048), (65536, 2048), (65536, 512)):
    torch.manual_seed(0)
    loc = torch.randn(B, d, device=dev)
    kap = torch.rand(B, device=dev) * 9.87 + 0.13
    z = torch.empty(B, 2 * d, device=dev); phi = torch.empty(B, d, device=dev)
    ent, dent = torch.empty(B, device=dev), torch.empty(B, device=dev)

    def fwd():
        lib.cvb_clifford_vm_rsample_kl(loc.data_ptr(), kap.data_ptr(), 1, 0, B, 7, 0, z.data_ptr(), phi.data_ptr(),
                                       ent.data_ptr(), None, dent.data_ptr(), B, d, st)
    def fwd_plain():
        lib.cvb_clifford_vm_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, 7, 0, z.data_ptr(), B, d, st)
    gz = torch.randn(B, 2 * d, device=dev); dloc = torch.empty(B, d, device=dev); dk = torch.empty(B, device=dev)
    def bwd():
        lib.cvb_clifford_vm_rsample_backward(gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, phi.data_ptr(),
                                             dloc.data_ptr(), dk.data_ptr(), B, d, st)
    lp = torch.empty(B, device=dev)
    def logp():
        lib.cvb_clifford_vm_log_prob(z.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, lp.data_ptr(), None, None, None,
                                     B, d, st)
    for name, fn, nbytes in (("vm fwd (phi saved, entropy)", fwd, 16 * d + 8), ("vm fwd (plain, old entry)", fwd_plain, 8 * d + 8),
                             ("vm backward", bwd, 20 * d + 8), ("vm log_prob", logp, 12 * d + 8)):
        ms = timeit(fn)
        gb = B * nbytes / (ms * 1e-3) / 1e9
        print(f"{name:30s} B={B:6d} d={d:5d} {ms:8.3f} ms {gb:7.1f} GB/s {100 * gb / PEAK:5.1f}% of 7.7 TB/s")
