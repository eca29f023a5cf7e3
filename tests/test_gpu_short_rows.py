"""GPU: the row-tile kernels for short rows (csrc/clifford_small.cuh, bind_small_kernel) on awkward shapes -- lengths from
1 circle / 1 element up to the limit of that path, odd lengths, row counts that do not fill a tile -- called through the
C ABI into guarded buffers (sentinel rows before and after the output: compute-sanitizer is not available on this GPU pool),
and compared with the oracle (Clifford: injected draws) or an fp64 torch.fft reference (bind / unbind)."""
import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _guarded(rows, cols):
    buf = torch.full((rows + 2, cols), float("nan"), device=DEV)
    return buf, buf[1:-1]


def _guards_intact(buf):
    return bool(torch.isnan(buf[0]).all()) and bool(torch.isnan(buf[-1]).all())


# Row counts for the larger tiles: with rows = 2 SMs RT + 3, ceil(rows / RT) >= 2 SMs > ceil(rows / 2RT), so
# small_rows_per_tile picks RT unless the tile's shared memory passes 48 KB.  On 148 SMs that gives, for the forward /
# backward / log_prob kernels: RT everywhere for d <= 65; at d = 100 the backward and log_prob run RT = 16 for "rt32";
# at d = 255 and 256 the forward runs RT = 16 for "rt32" and the backward and log_prob RT = 4 throughout.  bind_small_kernel
# (every length for the quotient modes 2 and 3, d <= 48 for the others) runs RT up to d = 100 and RT = 8 at d = 255, 256.
SM_ROWS = ["rt8", "rt16", "rt32"]


def _rows(rows):
    """an int, or "rtN": 2 SMs N + 3"""
    if isinstance(rows, int):
        return rows
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * int(rows[2:]) + 3


@pytest.mark.parametrize("d", [1, 2, 3, 7, 33, 65, 100, 255, 256])
@pytest.mark.parametrize("rows", [1, 3, 37] + SM_ROWS)
def test_clifford_short_rows_forward_backward_logprob(d, rows):
    from clifford_b200 import _lib
    from oracle import latent_oracle as O
    if d >= 16 and (d & (d - 1)) == 0:
        pytest.skip("power-of-two d >= 16 runs on the FFT engine")
    rows = _rows(rows)
    lib = _lib.load()
    _lib.ensure_device(torch.device(DEV))
    st = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator().manual_seed(1000 * d + rows)
    loc = torch.randn(rows, d, generator=gen) * 2
    kap = torch.rand(rows, 1, generator=gen) * 9 + 0.05
    tp = torch.distributions.Beta(0.5 + kap.expand(rows, d) + 1e-7, torch.tensor(0.5)).sample().clamp(1e-6, 1 - 1e-6)
    g = torch.randn(rows, d, generator=gen)
    gz = torch.randn(rows, 2 * d, generator=gen)
    lo, ka = loc.clone().requires_grad_(), kap.clone().requires_grad_()
    zo = O.clifford_ps_rsample(lo, ka, tp, g)
    dlo, dka = torch.autograd.grad((zo * gz).sum(), [lo, ka])
    locd, kapd, tpd, gd, gzd = (t.to(DEV).contiguous() for t in (loc, kap.reshape(-1), tp, g, gz))
    zbuf, z = _guarded(rows, 2 * d)
    klbuf, kl = _guarded(rows, 1)
    _lib.check(lib.cvb_clifford_ps_rsample(locd.data_ptr(), kapd.data_ptr(), 1, 0, rows, tpd.data_ptr(), gd.data_ptr(), 0, 0,
                                           z.data_ptr(), None, None, kl.data_ptr(), None, rows, d, st), "fwd")
    torch.cuda.synchronize()
    assert _guards_intact(zbuf) and _guards_intact(klbuf)
    assert rel_err(z.cpu(), zo.detach()) < 1e-5
    dlbuf, dl = _guarded(rows, d)
    dkbuf, dk = _guarded(rows, 1)
    _lib.check(lib.cvb_clifford_ps_rsample_backward(gzd.data_ptr(), locd.data_ptr(), kapd.data_ptr(), 1, 0, rows, tpd.data_ptr(),
                                                    gd.data_ptr(), None, dl.data_ptr(), dk.data_ptr(), rows, d, st), "bwd")
    torch.cuda.synchronize()
    assert _guards_intact(dlbuf) and _guards_intact(dkbuf)
    if d > 1:
        assert rel_err(dl.cpu()[:, 1:], dlo[:, 1:]) < 5e-5
        assert rel_err(dk.cpu(), dka) < 5e-4
    assert float(dl[:, 0].abs().max()) == 0.0
    lpbuf, lp = _guarded(rows, 1)
    _lib.check(lib.cvb_clifford_ps_log_prob(z.data_ptr(), locd.data_ptr(), kapd.data_ptr(), 1, 0, rows, lp.data_ptr(), None, None,
                                            None, rows, d, st), "log_prob")
    torch.cuda.synchronize()
    assert _guards_intact(lpbuf)
    lpo = O.clifford_ps_log_prob(zo.detach(), loc, kap.expand(rows, d)).reshape(-1).double()
    # conditioning of log1p(cos(loc - angle)): a bin almost opposite its mean direction amplifies fp32 angle noise (~4e-7)
    # by 1 / (1 + dot) -- the same bound the golden-vector log_prob test uses
    ang = torch.angle(torch.fft.fft(zo.detach().double(), dim=-1)[..., :d])
    one_p_dot = (1 + torch.cos(loc.double() - ang)).clamp_min(1e-7)
    bound = (kap.double().expand(rows, d) * 4e-7 / one_p_dot).sum(-1)
    err = (lp.cpu().reshape(-1).double() - lpo).abs()
    assert bool((err <= 2e-5 * lpo.abs() + bound + 1e-6).all()), (err, bound)


@pytest.mark.parametrize("d", [1, 2, 3, 5, 17, 31, 48, 49, 100, 255, 256])
@pytest.mark.parametrize("rows", [1, 3, 37] + SM_ROWS)
def test_bind_short_vectors_all_modes(d, rows):
    from clifford_b200 import _lib
    rows = _rows(rows)
    lib = _lib.load()
    _lib.ensure_device(torch.device(DEV))
    st = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator().manual_seed(77 * d + rows)
    a = torch.randn(rows, d, generator=gen, dtype=torch.float64) / np.sqrt(d)
    b = torch.randn(rows, d, generator=gen, dtype=torch.float64) / np.sqrt(d)
    well = rows > 37
    if well:
        # thousands of random rows hold some near-zero bin: for the quotient modes take b with spectrum magnitudes in
        # [0.5, 2] (random phases) so that every mode holds 1e-5
        h = d // 2 + 1
        mag = 0.5 * 4.0 ** torch.rand(rows, h, generator=gen, dtype=torch.float64)
        Bh = torch.polar(mag, 2 * np.pi * torch.rand(rows, h, generator=gen, dtype=torch.float64))
        Bh[:, 0] = mag[:, 0]
        if d % 2 == 0:
            Bh[:, -1] = mag[:, -1]
        b = torch.fft.irfft(Bh, n=d).float().double()
    A, Bf = torch.fft.fft(a), torch.fft.fft(b)
    want = {0: torch.fft.ifft(A * Bf).real, 1: torch.fft.ifft(A * Bf.conj()).real, 2: torch.fft.ifft(A / (Bf + 1e-12)).real,
            3: torch.fft.ifft(A / (Bf + 1e-12).conj()).real, 4: -torch.fft.ifft(A * Bf.conj()).real}
    ad, bd = a.float().to(DEV).contiguous(), b.float().to(DEV).contiguous()
    for mode, ref in want.items():
        obuf, o = _guarded(rows, d)
        _lib.check(lib.cvb_vsa_bind(ad.data_ptr(), bd.data_ptr(), o.data_ptr(), rows, rows, rows, d, mode, st), f"bind mode {mode}")
        torch.cuda.synchronize()
        assert _guards_intact(obuf), (d, rows, mode)
        tol = 5e-3 if mode in (2, 3) and not well else 1e-5  # the quotient is as ill-conditioned as min |B_k| makes it
        assert rel_err(o.cpu(), ref) < tol, (d, rows, mode)
    # broadcasting: one b row for every a row
    obuf, o = _guarded(rows, d)
    _lib.check(lib.cvb_vsa_bind(ad.data_ptr(), bd.data_ptr(), o.data_ptr(), rows, rows, 1, d, 0, st), "bind broadcast")
    torch.cuda.synchronize()
    assert _guards_intact(obuf)
    assert rel_err(o.cpu(), torch.fft.ifft(A * Bf[:1]).real) < 1e-5
