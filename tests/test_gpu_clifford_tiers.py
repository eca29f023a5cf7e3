"""GPU: the power-spherical Clifford kernels on every tier of their size dispatch (csrc/clifford_launch.cuh) against the
oracle evaluated in float64 on the CPU from the same draws.

The tiers: the FFT engine (power-of-two d in [16, 8192] with 8-byte aligned output / gradient / value rows), the
row-tile kernels (n = 2d <= 512) and the direct-DFT kernels (everything else, up to their shared-memory limit).  Each
call goes through the C ABI into NaN-guarded buffers: a store outside the rows, or a slot left unwritten, shows.

Tolerances are the suite's (max-norm relative unless stated): z 1e-5 (2e-5 for device-RNG samples, which use the fast
sincos); dloc 5e-5; dkappa 5e-4 (2e-3 on table-sampled rows, whose gradient is the table map's own); log_prob 2e-5 plus
the conditioning bound of log1p(cos(loc - angle)); log_prob gradients 1e-4 on well-conditioned bins; value gradient 2e-4.

Length limits of the direct-DFT tier, from its shared-memory formulas against kGenericSmemLimit (200 KB): the forward
takes d <= 8533, the backward and log_prob d <= 8528.  So d in [8529, 8533] can be sampled but not differentiated."""
import math

import numpy as np
import pytest
import torch

from conftest import rel_err

DEV = "cuda"
ROW_TILE = [2, 8, 40, 200]
FFT = [16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]
DIRECT = [257, 300, 1000, 4097]
S = 3                                   # samples per loc row in the broadcast cases: rows = S * loc_rows
GUARD = 64                              # NaN floats before and after every output
HEAD = (0.03, 10.0)                     # (floor, kmax) of the folded concentration head


# ---- float64 references on the CPU ----------------------------------------------------------------------------------
def _kappa_el(kap, rows, d):
    """per-element concentrations (rows, d) of a row-scalar (loc_rows,) or per-element (loc_rows, d) kappa"""
    k = kap.reshape(kap.shape[0], -1).expand(kap.shape[0], d)
    return k.repeat(rows // kap.shape[0], 1)


def ref_rsample(loc, kap, tp, sgn, gz):
    """z, dloc, dkappa (per row, or per element) of z = O.clifford_ps_rsample in float64 by autograd; loc (L, d), kap (L,)
    or (L, d), draws / grad_z per row (rows = S * L).  The sign draw enters as g = sgn (s = g / (|g| + 1e-7))."""
    from oracle import latent_oracle as O
    rows, d = tp.shape
    lo = loc.double().repeat(rows // loc.shape[0], 1).requires_grad_()
    rowk = kap.dim() == 1
    ka = (kap.double().repeat(rows // kap.shape[0])[:, None] if rowk else _kappa_el(kap.double(), rows, d)).requires_grad_()
    z = O.clifford_ps_rsample(lo, ka, tp.double(), sgn.double())
    dlo, dka = torch.autograd.grad((z * gz.double()).sum(), [lo, ka])
    return z.detach(), dlo, (dka.reshape(-1) if rowk else dka)


def ref_entropy(kap_el):
    """entropy, kl, per-element dH/dkappa of rows of per-element concentrations (float64)"""
    from oracle import latent_oracle as O
    k = kap_el.double()
    return O.clifford_ps_entropy(k), O.clifford_ps_kl(k), O.clifford_ps_entropy_backward(k)


def lp_of_spectrum(F, loc, kap_el):
    """O.clifford_ps_log_prob with the spectrum F = fft(value)[..., :d] as the argument (for d log_prob / d F)"""
    from oracle import latent_oracle as O
    ang = torch.angle(F)
    dot = torch.clamp(torch.cos(loc) * torch.cos(ang) + torch.sin(loc) * torch.sin(ang), min=-1.0 + O.EPS, max=1.0 - O.EPS)
    return (O.ps_log_normalizer(kap_el, 2) + kap_el * torch.log1p(dot)).sum(-1)


def ref_log_prob(value, loc, kap):
    """log_prob, dlp/dloc, dlp/dkappa (per row or per element), dlp/dF (rows, d, 2) and 1 + dot per bin, all float64"""
    rows, n = value.shape
    d = n // 2
    rowk = kap.dim() == 1
    F = torch.fft.fft(value.double(), dim=-1)[:, :d].detach().requires_grad_()
    lo = loc.double().repeat(rows // loc.shape[0], 1).requires_grad_()
    ka = (kap.double().repeat(rows // kap.shape[0])[:, None] if rowk else _kappa_el(kap.double(), rows, d)).requires_grad_()
    lp = lp_of_spectrum(F, lo, ka.expand(rows, d))
    dF, dlo, dka = torch.autograd.grad(lp.sum(), [F, lo, ka])
    one_p_dot = (1 + torch.cos(lo.detach() - torch.angle(F.detach()))).clamp_min(1e-7)
    return lp.detach(), dlo, (dka.reshape(-1) if rowk else dka), torch.view_as_real(dF), one_p_dot, ka.detach().expand(rows, d)


def assert_log_prob(got, ref):
    """kernel (lp, dl, dk, dF) against ref_log_prob: conditioning-aware, as the golden-vector log_prob test"""
    lp, dl, dk, dF = got
    rlp, rdl, rdk, rdF, one_p_dot, kap_el = ref
    cond = 4e-7 / one_p_dot                     # fp32 angle noise amplified by 1 / (1 + dot), per bin
    err = (lp.double() - rlp).abs()
    assert bool((err <= 2e-5 * rlp.abs() + (kap_el * cond).sum(-1) + 1e-6).all()), float(err.max())
    well = one_p_dot > 1e-2
    if dl is not None:
        assert rel_err(dl.numpy()[well.numpy()], rdl.numpy()[well.numpy()]) < 1e-4
        dk_bound = cond.sum(-1) if dk.dim() == 1 else cond
        assert bool(((dk.double() - rdk).abs() <= 2e-5 * float(rdk.abs().max()) + dk_bound).all())
    if dF is not None:
        w = well.numpy()
        assert rel_err(dF.numpy()[w], rdF.numpy()[w]) < 2e-4


def tprime_and_sign(saved, kap, d, table):
    """(t', sign) of the draws a device-RNG forward saved: copysign(t', s), or on table-sampled rows the signed table
    coordinate, mapped to t' by the numpy restatement of the table (test_gpu_clifford._tprime_from_table_coordinate)"""
    saved = saved.clone()
    saved[:, 0] = 0.5                           # circle 0 is never drawn (its slot is left unwritten)
    sgn = torch.where(torch.signbit(saved), -1.0, 1.0)
    if table:
        from test_gpu_clifford import _tprime_from_table_coordinate
        k = kap.reshape(-1, 1).repeat(saved.shape[0] // kap.shape[0], 1)
        return _tprime_from_table_coordinate(saved.abs().numpy(), k.numpy()), sgn
    return saved.abs(), sgn


def make_inputs(d, rowk, loc_rows, rows, seed, clamp=1e-6):
    """loc (L, d), kappa (L,) | (L, d) in (0.03, 10), injected draws t' ~ Beta(1/2 + kappa + 1e-7, 1/2), normal g and an
    upstream gradient, all (rows, d) / (rows, 2d) float32 on the CPU"""
    torch.manual_seed(seed)                     # the Beta draws come from the global generator
    gen = torch.Generator().manual_seed(seed)
    loc = torch.randn(loc_rows, d, generator=gen) * 2
    kap = torch.rand((loc_rows,) if rowk else (loc_rows, d), generator=gen) * 9.97 + 0.03
    alpha = 0.5 + _kappa_el(kap, rows, d) + 1e-7
    tp = torch.distributions.Beta(alpha, torch.full_like(alpha, 0.5)).sample().clamp(clamp, 1 - clamp)
    g = torch.randn(rows, d, generator=gen)
    gz = torch.randn(rows, 2 * d, generator=gen)
    return loc, kap, tp, g, gz


def value_near(z, seed):
    """a sample plus small noise, as test_log_prob_gradient_wrt_value_vs_oracle_autograd"""
    gen = torch.Generator().manual_seed(seed)
    return (z + 0.02 * torch.randn(z.shape, generator=gen, dtype=z.dtype) / z.shape[1] ** 0.5).float()


def test_references_run_on_cpu():
    """the float64 references at a toy size: the spectrum form of log_prob is the oracle's, and the autograd gradient of
    the sample is the oracle's closed form"""
    from oracle import latent_oracle as O
    for rowk in (True, False):
        loc, kap, tp, g, gz = make_inputs(5, rowk, 2, 6, seed=1)
        z, dlo, dka = ref_rsample(loc, kap, tp, torch.sign(g), gz)
        k_el = _kappa_el(kap.double(), 6, 5)
        cl, ck = O.clifford_ps_rsample_backward(loc.double().repeat(3, 1), k_el, tp.double(), torch.sign(g).double(), gz.double())
        assert rel_err(dlo, cl) < 1e-10 and rel_err(dka, ck.sum(-1) if rowk else ck) < 1e-10
        v = value_near(z, 2)
        lp, _, _, dF, _, _ = ref_log_prob(v, loc, kap)
        assert rel_err(lp, O.clifford_ps_log_prob(v.double(), loc.double().repeat(3, 1), k_el)) < 1e-12
        assert dF.shape == (6, 5, 2)
        ent, kl, dent = ref_entropy(k_el)
        assert ent.shape == kl.shape == (6,) and dent.shape == (6, 5) and float(dent[:, 0].abs().max()) == 0


# ---- the C ABI into guarded buffers ---------------------------------------------------------------------------------
def _lib():
    from clifford_b200 import _lib as L
    L.ensure_device(torch.device(DEV))
    return L, L.load()


def call(name, *args):
    """the status code of one C-ABI call on the current stream"""
    _, lib = _lib()
    return getattr(lib, name)(*args, torch.cuda.current_stream().cuda_stream)


def ok(name, *args):
    L, _ = _lib()
    L.check(call(name, *args), name)


class Out:
    """a NaN-filled output of `shape` inside NaN guards, starting `shift` bytes past a 256-byte boundary"""

    def __init__(self, *shape, shift=0):
        self.n = math.prod(shape)
        self.lo = GUARD + shift // 4
        self.buf = torch.full((self.n + 2 * GUARD,), float("nan"), device=DEV)
        self.t = self.buf[self.lo:self.lo + self.n].view(shape)
        assert self.t.data_ptr() % 256 == shift

    @property
    def p(self):
        return self.t.data_ptr()

    def guards_intact(self):
        return bool(torch.isnan(self.buf[:self.lo]).all()) and bool(torch.isnan(self.buf[self.lo + self.n:]).all())

    def untouched(self):
        return bool(torch.isnan(self.buf).all())

    def cpu(self):
        torch.cuda.synchronize()
        assert self.guards_intact()
        return self.t.cpu()


def dev(t, shift=0):
    """a device copy of t, `shift` bytes past a 256-byte boundary (NaN around it)"""
    if shift == 0:
        return t.to(DEV).contiguous()
    o = Out(*t.shape, shift=shift)
    o.t.copy_(t.to(DEV))
    return o.t


def k_strides(kap, d):
    return (1, 0) if kap.dim() == 1 else (d, 1)


def run_rsample(loc, kap, tp, g, d, rows, z_shift=0, save=False, entropy=False, seed=11, offset=5):
    """cvb_clifford_ps_rsample; tp / g None draws on the device.  Returns (rc, z, tp_signed, entropy, kl, dentropy) Outs"""
    krs, kes = k_strides(kap, d)
    z = Out(rows, 2 * d, shift=z_shift)
    tps = Out(rows, d) if save else None
    e = [Out(rows) for _ in range(3)] if entropy else [None] * 3
    pp = (lambda o: None if o is None else o.p)
    rc = call("cvb_clifford_ps_rsample", loc.data_ptr(), kap.data_ptr(), krs, kes, loc.shape[0],
              None if tp is None else tp.data_ptr(), None if g is None else g.data_ptr(), seed, offset, z.p, pp(tps),
              pp(e[0]), pp(e[1]), pp(e[2]), rows, d)
    return rc, z, tps, e[0], e[1], e[2]


def run_backward(gz, loc, kap, tp, g, tps, d, rows):
    krs, kes = k_strides(kap, d)
    dl = Out(rows, d)
    dk = Out(rows) if kes == 0 else Out(rows, d)
    rc = call("cvb_clifford_ps_rsample_backward", gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), krs, kes, loc.shape[0],
              None if tp is None else tp.data_ptr(), None if g is None else g.data_ptr(),
              None if tps is None else tps.data_ptr(), dl.p, dk.p, rows, d)
    return rc, dl, dk


def run_log_prob(value, loc, kap, d, rows, grads=True, entry="cvb_clifford_ps_log_prob"):
    krs, kes = k_strides(kap, d)
    lp = Out(rows)
    dl = Out(rows, d) if grads else None
    dk = (Out(rows) if kes == 0 else Out(rows, d)) if grads else None
    dF = Out(rows, d, 2) if grads else None
    pp = (lambda o: None if o is None else o.p)
    rc = call(entry, value.data_ptr(), loc.data_ptr(), kap.data_ptr(), krs, kes, loc.shape[0], lp.p, pp(dl), pp(dk), pp(dF),
              rows, d)
    return rc, lp, dl, dk, dF


def _cpu(*outs):
    return tuple(None if o is None else o.cpu() for o in outs)


# ---- the tier matrix ------------------------------------------------------------------------------------------------
def _loc_rows(d):
    return 2 if d >= 4097 else (3 if d >= 512 else 5)


@pytest.mark.gpu
@pytest.mark.parametrize("broadcast", [False, True], ids=["rows=B", "rows=SxB"])
@pytest.mark.parametrize("rowk", [True, False], ids=["rowk", "elk"])
@pytest.mark.parametrize("d", ROW_TILE + FFT + DIRECT)
def test_tier_matrix(d, rowk, broadcast):
    L = _loc_rows(d)
    rows = S * L if broadcast else L
    loc, kap, tp, g, gz = make_inputs(d, rowk, L, rows, seed=7 * d + 2 * rowk + broadcast)
    locd, kapd, tpd, gd, gzd = (dev(t) for t in (loc, kap, tp, g, gz))
    z_ref, dl_ref, dk_ref = ref_rsample(loc, kap, tp, g, gz)
    rc, z, _, ent, kl, dent = run_rsample(locd, kapd, tpd, gd, d, rows, entropy=rowk)
    assert rc == 0
    assert rel_err(z.cpu(), z_ref) < 1e-5
    if rowk:
        e_ref, kl_ref, de_ref = ref_entropy(_kappa_el(kap, rows, d))
        assert rel_err(ent.cpu(), e_ref) < 1e-5
        assert float((kl.cpu().double() - kl_ref).abs().max()) < 1e-5 * max(d - 1, 1) * math.log(2 * math.pi)
        assert rel_err(dent.cpu(), de_ref.sum(-1)) < 2e-5

    # backward from the injected draws
    rc, dl, dk = run_backward(gzd, locd, kapd, tpd, gd, None, d, rows)
    assert rc == 0
    assert rel_err(dl.cpu(), dl_ref) < 5e-5
    assert rel_err(dk.cpu(), dk_ref) < 5e-4

    # device RNG with the draws saved, then the backward from them
    rc, z, tps, _, _, _ = run_rsample(locd, kapd, None, None, d, rows, save=True)
    assert rc == 0
    table = rowk and 512 <= d <= 8192 and (d & (d - 1)) == 0       # table-sampled rows (all kappa here are <= 32)
    tp_rng, sgn = tprime_and_sign(tps.cpu(), kap, d, table)
    z_rng = z.cpu()
    z_ref, dl_ref, dk_ref = ref_rsample(loc, kap, tp_rng, sgn, gz)
    assert rel_err(z_rng, z_ref) < 2e-5
    rc, dl, dk = run_backward(gzd, locd, kapd, None, None, tps.t, d, rows)
    assert rc == 0
    # table rows: the oracle is driven through t' = cos^2(phi / 2) in fp32 (see test_rng_mode_invariants_...)
    assert rel_err(dl.cpu(), dl_ref) < (3e-4 if table else 5e-5)
    assert rel_err(dk.cpu(), dk_ref) < (2e-3 if table else 5e-4)

    # log_prob with every derivative output, at a value near a sample of well-conditioned draws
    _, _, tpc, gc, _ = make_inputs(d, rowk, L, rows, seed=7 * d + 2 * rowk + broadcast, clamp=1e-3)
    value = value_near(ref_rsample(loc, kap, tpc, gc, gz)[0], seed=d)
    rc, lp, dl, dk, dF = run_log_prob(dev(value), locd, kapd, d, rows)
    assert rc == 0
    assert_log_prob(_cpu(lp, dl, dk, dF), ref_log_prob(value, loc, kap))
    # and the evaluation variant (no derivative outputs)
    rc, lp, _, _, _ = run_log_prob(dev(value), locd, kapd, d, rows, grads=False)
    assert rc == 0
    assert_log_prob((lp.cpu(), None, None, None), ref_log_prob(value, loc, kap))


@pytest.mark.gpu
@pytest.mark.parametrize("d", ROW_TILE + FFT + DIRECT)
def test_spectrum_adjoint_and_phases_to_vector(d):
    """cvb_clifford_spectrum_adjoint against float64 autograd of fft(value)[..., :d]; cvb_clifford_phases_to_vector
    against O.clifford_uniform_rsample"""
    from oracle import latent_oracle as O
    rows = 2 if d >= 4097 else 7
    gen = torch.Generator().manual_seed(d)
    H = torch.randn(rows, d, 2, generator=gen)
    v = torch.zeros(rows, 2 * d, dtype=torch.float64, requires_grad=True)
    F = torch.fft.fft(v, dim=-1)[:, :d]
    (want,) = torch.autograd.grad((F.real * H[..., 0].double() + F.imag * H[..., 1].double()).sum(), [v])
    out = Out(rows, 2 * d)
    ok("cvb_clifford_spectrum_adjoint", dev(H).data_ptr(), out.p, rows, d)
    assert rel_err(out.cpu(), want) < 1e-5
    u = torch.rand(rows, d, generator=gen)
    out = Out(rows, 2 * d)
    ok("cvb_clifford_phases_to_vector", dev(u).data_ptr(), 2 * math.pi, 0, 0, out.p, rows, d)
    assert rel_err(out.cpu(), O.clifford_uniform_rsample(u.double())) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("rowk", [True, False], ids=["rowk", "elk"])
@pytest.mark.parametrize("d", [2, 40, 257, 2048, 8192])
def test_entropy_kl(d, rowk):
    """cvb_ps_entropy_kl(torus=1): entropy and KL per row, dH/dkappa per row or per element"""
    rows = 9
    gen = torch.Generator().manual_seed(d + rowk)
    kap = torch.rand((rows,) if rowk else (rows, d), generator=gen) * 9.97 + 0.03
    krs, kes = k_strides(kap, d)
    ent, kl = Out(rows), Out(rows)
    dent = Out(rows) if rowk else Out(rows, d)
    ok("cvb_ps_entropy_kl", dev(kap).data_ptr(), krs, kes, rows, d, 0.5, 1, 0.0, ent.p, kl.p, dent.p)
    e_ref, kl_ref, de_ref = ref_entropy(_kappa_el(kap, rows, d))
    assert rel_err(ent.cpu(), e_ref) < 1e-5
    assert float((kl.cpu().double() - kl_ref).abs().max()) < 1e-5 * max(d - 1, 1) * math.log(2 * math.pi)
    assert rel_err(dent.cpu(), de_ref.sum(-1) if rowk else de_ref) < 2e-5


def _softplus64(raw):
    return torch.nn.functional.softplus(raw.double())


@pytest.mark.gpu
@pytest.mark.parametrize("d", [40, 2048, 300])
def test_head_pair(d):
    """cvb_clifford_ps_rsample_head / _backward_head (kappa = min(softplus(raw) + floor, kmax) in the kernel): injected
    draws against the float64 oracle, with every kappa-derivative carrying d kappa / d raw = sigmoid(raw)"""
    L, rows = 3, 9
    loc, _, _, g, gz = make_inputs(d, True, L, rows, seed=d)
    raw = torch.tensor([-3.0, 0.2, 2.0])                 # kappa from 0.08 to 2.2: the clamp at kmax is not active
    kap64 = _softplus64(raw) + HEAD[0]
    torch.manual_seed(d)
    alpha = 0.5 + _kappa_el(kap64.float(), rows, d) + 1e-7
    tp = torch.distributions.Beta(alpha, torch.full_like(alpha, 0.5)).sample().clamp(1e-6, 1 - 1e-6)
    z_ref, dl_ref, dk_ref = ref_rsample(loc, kap64, tp, g, gz)
    chain = torch.sigmoid(raw.double()).repeat(S)
    locd, rawd, tpd, gd, gzd = (dev(t) for t in (loc, raw, tp, g, gz))
    z = Out(rows, 2 * d)
    ent, kl, dent = Out(rows), Out(rows), Out(rows)
    ok("cvb_clifford_ps_rsample_head", locd.data_ptr(), rawd.data_ptr(), L, *HEAD, tpd.data_ptr(), gd.data_ptr(), 0, 0,
       z.p, None, ent.p, kl.p, dent.p, rows, d)
    assert rel_err(z.cpu(), z_ref) < 1e-5
    e_ref, _, de_ref = ref_entropy(_kappa_el(kap64, rows, d))
    assert rel_err(ent.cpu(), e_ref) < 1e-5
    assert rel_err(dent.cpu(), de_ref.sum(-1) * chain) < 2e-5
    dl, dk = Out(rows, d), Out(rows)
    ok("cvb_clifford_ps_rsample_backward_head", gzd.data_ptr(), locd.data_ptr(), rawd.data_ptr(), L, *HEAD, tpd.data_ptr(),
       gd.data_ptr(), None, dl.p, dk.p, rows, d)
    assert rel_err(dl.cpu(), dl_ref) < 5e-5
    assert rel_err(dk.cpu(), dk_ref * chain) < 5e-4


# ---- output alignment -----------------------------------------------------------------------------------------------
# A z / grad_z / value 4 bytes past an 8-byte boundary moves the call off the FFT engine: to the row tiles at d = 16
# and 256, to the direct DFT at d = 512 and 2048.
SHIFT_DIMS = [16, 256, 512, 2048]


@pytest.mark.gpu
@pytest.mark.parametrize("d", SHIFT_DIMS)
def test_shifted_outputs_injected_draws(d):
    rows = 6
    loc, kap, tp, g, gz = make_inputs(d, True, 3, rows, seed=d)
    locd, kapd, tpd, gd, gzd = (dev(t) for t in (loc, kap, tp, g, gz))
    _, z0, _, _, _, _ = run_rsample(locd, kapd, tpd, gd, d, rows)
    rc, z1, _, _, _, _ = run_rsample(locd, kapd, tpd, gd, d, rows, z_shift=4)
    assert rc == 0 and rel_err(z1.cpu(), z0.cpu()) < 1e-5
    _, dl0, dk0 = run_backward(gzd, locd, kapd, tpd, gd, None, d, rows)
    rc, dl1, dk1 = run_backward(dev(gz, 4), locd, kapd, tpd, gd, None, d, rows)
    assert rc == 0
    assert rel_err(dl1.cpu(), dl0.cpu()) < 5e-5 and rel_err(dk1.cpu(), dk0.cpu()) < 5e-4
    _, _, tpc, gc, _ = make_inputs(d, True, 3, rows, seed=d, clamp=1e-3)
    value = value_near(ref_rsample(loc, kap, tpc, gc, gz)[0], seed=d)
    ref = ref_log_prob(value, loc, kap)
    for shift in (0, 4):
        rc, lp, dl, dk, dF = run_log_prob(dev(value, shift), locd, kapd, d, rows)
        assert rc == 0
        assert_log_prob(_cpu(lp, dl, dk, dF), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [512, 2048])
def test_shifted_outputs_with_saved_device_draws_are_refused(d):
    """At power-of-two d >= 512 with one concentration per row the FFT engine saves table coordinates, the other tiers
    t': a forward with z, or a backward with grad_z, off the 8-byte grid would mix the two formats.  Both are refused
    before anything is launched or written; per-element concentrations (t' on every tier) are accepted."""
    L_, _ = _lib()
    rows = 6
    loc, kap, _, _, gz = make_inputs(d, True, 3, rows, seed=d)
    locd, kapd = dev(loc), dev(kap)
    raw = dev(torch.tensor([-1.0, 0.0, 1.0]))
    n0 = L_.launch_count()
    rc, z, tps, _, _, _ = run_rsample(locd, kapd, None, None, d, rows, z_shift=4, save=True)
    assert rc == 2 and "aligned" in L_.load().cvb_last_error_string().decode()
    z2, tps2 = Out(rows, 2 * d, shift=4), Out(rows, d)
    assert call("cvb_clifford_ps_rsample_head", locd.data_ptr(), raw.data_ptr(), 3, *HEAD, None, None, 1, 2, z2.p, tps2.p,
                None, None, None, rows, d) == 2
    torch.cuda.synchronize()
    assert all(o.untouched() for o in (z, tps, z2, tps2))
    assert L_.launch_count() == n0
    # the saved draws of an aligned forward, read by a backward whose gradient rows are off the grid
    _, _, saved, _, _, _ = run_rsample(locd, kapd, None, None, d, rows, save=True)
    n0 = L_.launch_count()
    rc, dl, dk = run_backward(dev(gz, 4), locd, kapd, None, None, saved.t, d, rows)
    assert rc == 2 and "aligned" in L_.load().cvb_last_error_string().decode()
    dl2, dk2 = Out(rows, d), Out(rows)
    assert call("cvb_clifford_ps_rsample_backward_head", dev(gz, 4).data_ptr(), locd.data_ptr(), raw.data_ptr(), 3, *HEAD,
                None, None, saved.t.data_ptr(), dl2.p, dk2.p, rows, d) == 2
    torch.cuda.synchronize()
    assert all(o.untouched() for o in (dl, dk, dl2, dk2))
    assert L_.launch_count() == n0
    # per-element concentrations save t' on every tier: accepted in every pairing of shifted and aligned calls
    _, kel, _, _, _ = make_inputs(d, False, 3, rows, seed=d)
    check_saved_draws_across_tiers(loc, kel, gz, d, rows)


def check_saved_draws_across_tiers(loc, kap, gz, d, rows):
    """device-RNG forwards with z aligned and 4 bytes off, each followed by backwards with grad_z aligned and 4 bytes
    off (the tiers draw differently, so each is checked against the oracle on its own saved draws)"""
    locd, kapd = dev(loc), dev(kap)
    for z_shift in (0, 4):
        rc, z, tps, _, _, _ = run_rsample(locd, kapd, None, None, d, rows, z_shift=z_shift, save=True)
        assert rc == 0
        tp, sgn = tprime_and_sign(tps.cpu(), kap, d, False)
        z_ref, dl_ref, dk_ref = ref_rsample(loc, kap, tp, sgn, gz)
        assert rel_err(z.cpu(), z_ref) < 2e-5, z_shift
        for g_shift in (0, 4):
            rc, dl, dk = run_backward(dev(gz, g_shift), locd, kapd, None, None, tps.t, d, rows)
            assert rc == 0
            assert rel_err(dl.cpu(), dl_ref) < 5e-5 and rel_err(dk.cpu(), dk_ref) < 5e-4, (z_shift, g_shift)


@pytest.mark.gpu
def test_shifted_outputs_with_saved_device_draws_at_256():
    """d = 256 never saves table coordinates: a shifted z (row tiles) or grad_z is accepted in every pairing with the
    FFT engine.  (The tiers' device samplers make different draws for the same seed: what must hold is that every
    backward reads the draws its forward saved.)"""
    d, rows = 256, 6
    loc, kap, _, _, gz = make_inputs(d, True, 3, rows, seed=d)
    check_saved_draws_across_tiers(loc, kap, gz, d, rows)


@pytest.mark.gpu
def test_autograd_gradient_at_an_odd_offset():
    """A loss that packs z behind one float hands CliffordPSRsample.backward a contiguous gradient 4 bytes past an 8-byte
    boundary.  With saved device draws at d = 2048 (table-sampled rows) dloc and dkappa must not depend on that."""
    from clifford_b200 import ops
    B, d = 64, 2048
    gen = torch.Generator().manual_seed(3)
    loc = (torch.randn(B, d, generator=gen) * 2).to(DEV).requires_grad_()
    kap = (torch.rand(B, 1, generator=gen) * 9.97 + 0.03).to(DEV).requires_grad_()
    w = torch.randn(B, 2 * d, generator=gen).to(DEV)
    s = torch.zeros((), device=DEV)

    def grads(packed):
        torch.manual_seed(99)                                      # the same device draws on both calls
        z, _, _ = ops.CliffordPSRsample.apply(loc, kap, 1, None, False)
        seen = []
        z.register_hook(lambda g: seen.append(g.data_ptr() % 8))
        if packed:
            flat = torch.cat([s.view(1), z.flatten()])
            loss = (flat[1:] * w.flatten()).sum() + flat[0]
        else:
            loss = (z * w).sum()
        out = torch.autograd.grad(loss, [loc, kap])
        return out, seen

    (dl0, dk0), seen0 = grads(False)
    (dl1, dk1), seen1 = grads(True)
    assert seen0 == [0] and seen1 == [4]
    assert torch.equal(dl1, dl0) and torch.equal(dk1, dk0)


# ---- length limits of the direct-DFT tier ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_longest_differentiable_length():
    """d = 8528, the longest length the direct-DFT backward and log_prob take: all three against float64 on 2 rows"""
    d, rows = 8528, 2
    loc, kap, tp, g, gz = make_inputs(d, True, rows, rows, seed=d)
    locd, kapd, tpd, gd, gzd = (dev(t) for t in (loc, kap, tp, g, gz))
    z_ref, dl_ref, dk_ref = ref_rsample(loc, kap, tp, g, gz)
    rc, z, _, _, _, _ = run_rsample(locd, kapd, tpd, gd, d, rows)
    assert rc == 0 and rel_err(z.cpu(), z_ref) < 1e-5
    rc, dl, dk = run_backward(gzd, locd, kapd, tpd, gd, None, d, rows)
    assert rc == 0 and rel_err(dl.cpu(), dl_ref) < 5e-5 and rel_err(dk.cpu(), dk_ref) < 5e-4
    _, _, tpc, gc, _ = make_inputs(d, True, rows, rows, seed=d, clamp=1e-3)
    value = value_near(ref_rsample(loc, kap, tpc, gc, gz)[0], seed=d)
    rc, lp, dl, dk, dF = run_log_prob(dev(value), locd, kapd, d, rows)
    assert rc == 0
    assert_log_prob(_cpu(lp, dl, dk, dF), ref_log_prob(value, loc, kap))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [8529, 8534, 16384])
def test_lengths_past_the_limits_are_refused(d):
    """d = 8529 .. 8533 can be sampled but not differentiated; from d = 8534 (and at every longer power of two) every
    entry point refuses, before launching or writing anything"""
    L_, _ = _lib()
    rows = 2
    loc, kap, tp, g, gz = make_inputs(d, True, rows, rows, seed=d)
    locd, kapd, tpd, gd, gzd = (dev(t) for t in (loc, kap, tp, g, gz))
    n0 = L_.launch_count()
    outs = []
    rc, dl, dk = run_backward(gzd, locd, kapd, tpd, gd, None, d, rows)
    assert rc == 2
    rc, lp, dl2, dk2, dF = run_log_prob(gzd, locd, kapd, d, rows)
    assert rc == 2
    rc, lp2, _, _, _ = run_log_prob(gzd, locd, kapd, d, rows, grads=False, entry="cvb_clifford_vm_log_prob")
    assert rc == 2
    outs += [dl, dk, lp, dl2, dk2, dF, lp2]
    if d <= 8533:
        rc, z, _, _, _, _ = run_rsample(locd, kapd, tpd, gd, d, rows)
        assert rc == 0
        z_ref, _, _ = ref_rsample(loc, kap, tp, g, gz)
        assert rel_err(z.cpu(), z_ref) < 1e-5
        torch.cuda.synchronize()
        assert L_.launch_count() == n0 + 1
    else:
        for args in ((tpd, gd, False), (None, None, True)):
            rc, z, tps, _, _, _ = run_rsample(locd, kapd, args[0], args[1], d, rows, save=args[2])
            assert rc == 2
            outs += [z] + ([tps] if tps is not None else [])
        z = Out(rows, 2 * d)
        assert call("cvb_clifford_spectrum_adjoint", gzd.data_ptr(), z.p, rows, d) == 2
        z2 = Out(rows, 2 * d)
        assert call("cvb_clifford_phases_to_vector", tpd.data_ptr(), 1.0, 0, 0, z2.p, rows, d) == 2
        z3 = Out(rows, 2 * d)
        assert call("cvb_clifford_vm_rsample", locd.data_ptr(), kapd.data_ptr(), 1, 0, rows, 1, 2, z3.p, rows, d) == 2
        outs += [z, z2, z3]
        torch.cuda.synchronize()
        assert L_.launch_count() == n0
    assert all(o.untouched() for o in outs)


# ---- the log_prob row-constant cache and its fallback ---------------------------------------------------------------
@pytest.mark.gpu
def test_log_prob_past_the_row_constant_cache():
    """clifford_log_prob_kernel precomputes the row constants of its first kLpConstCache = 256 rows per group and
    recomputes them past that.  A group's stride is at most SMs * 2048 / T rows (T = d / 16 threads per FFT), so
    256 * SMs * 2048 / T + 37 rows reach the recomputing branch whatever the occupancy.  value, loc and kappa are
    periodic in the row (period P = loc_rows): every row must equal row r mod P, and the first P rows the float64
    reference.  Evaluation variant, gradient variant and the von Mises log_prob."""
    from test_gpu_clifford_vm import _lp_ref
    d, P = 2048, 997
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rows = 256 * sms * 2048 // (d // 16) + 37
    loc, kap, tp, g, gz = make_inputs(d, True, P, P, seed=5, clamp=1e-3)
    value = value_near(ref_rsample(loc, kap, tp, g, gz)[0], seed=6)
    ref = ref_log_prob(value, loc, kap)
    locd, kapd = dev(loc), dev(kap)
    torch.cuda.reset_peak_memory_stats()
    idx = torch.arange(rows, device=DEV) % P

    def periodic(t):
        """every row of t (rows, ...) equals row r mod P to 1e-6 relative (checked in chunks)"""
        for i in range(0, rows, 64 * P):
            got, want = t[i:i + 64 * P], t[:P][idx[i:i + 64 * P]]
            assert bool(((got - want).abs() <= 1e-6 * want.abs()).all()), i

    def log_prob(entry, grads):
        vd = dev(value).repeat((rows + P - 1) // P, 1)[:rows]
        out = run_log_prob(vd, locd, kapd, d, rows, grads=grads, entry=entry)
        assert out[0] == 0
        torch.cuda.synchronize()
        del vd
        return out[1:]

    lp, dl, dk, _ = log_prob("cvb_clifford_ps_log_prob", False)
    periodic(lp.t)
    assert_log_prob((lp.t[:P].cpu(), None, None, None), ref)
    del lp
    lp, dl, dk, dF = log_prob("cvb_clifford_ps_log_prob", True)
    for t in (lp.t, dl.t, dk.t):
        periodic(t)
    assert_log_prob((lp.t[:P].cpu(), dl.t[:P].cpu(), dk.t[:P].cpu(), dF.t[:P].cpu()), ref)
    del lp, dl, dk, dF
    torch.cuda.empty_cache()
    lp, _, _, _ = log_prob("cvb_clifford_vm_log_prob", False)
    periodic(lp.t)
    want = _lp_ref(value.double(), loc.double(), kap.double()[:, None])
    assert float((lp.t[:P].cpu().double() - want).abs().max()) <= 1e-5 * (float(want.abs().max()) + 1.0)
    print(f"rows={rows} on {sms} SMs; peak GPU memory {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")
