"""GPU: the reparameterised von Mises torus latent (CliffordTorusDistribution): draws unchanged by the new forward entry,
the implicit pathwise gradient against SciPy's CDF, the log density against an fp64 torch restatement, the fused
entropy / KL, robustness over concentrations, and one VAE training step.  Every row length path: the FFT engine
(power-of-two d in [16, 8192]), the short-row tiles (2d <= 512) and the direct DFT (any other d)."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"
DS = [1, 2, 5, 20, 40, 300, 16, 512, 2048, 8192]


def _rows(d):
    return 6 if d >= 2048 else 24


def _entry(name, *args):
    from clifford_b200 import _lib
    from clifford_b200.ops import _launch
    _launch(name, torch.device(DEV), *args)


def _kappa_rows(rows):
    """concentrations from 1e-3 to 1e3, log-spaced over the rows"""
    return torch.logspace(-3, 3, rows, device=DEV)


def _draw(loc, kap, rowk, seed=123, off=7, with_phi=True):
    """(z, phi) from cvb_clifford_vm_rsample_kl; kap (B,) for row-scalar, (B, d) otherwise"""
    from clifford_b200._lib import ptr
    B, d = loc.shape
    z = torch.empty(B, 2 * d, device=DEV)
    phi = torch.zeros(B, d, device=DEV) if with_phi else None
    krs, kes = (1, 0) if rowk else (d, 1)
    _entry("cvb_clifford_vm_rsample_kl", ptr(loc), ptr(kap), krs, kes, B, seed, off, ptr(z), ptr(phi), None, None, None, B, d)
    return z, phi


def _oracle_dphi(phi, k):
    """-d_kappa F / f in fp64 by Richardson-extrapolated central differences of scipy's CDF (lower tail; J is odd)"""
    from scipy.stats import vonmises
    a = -np.abs(phi)
    h = 1e-4 * np.maximum(k, 1e-2)
    d1 = (vonmises.cdf(a, k + h) - vonmises.cdf(a, k - h)) / (2 * h)
    d2 = (vonmises.cdf(a, k + h / 2) - vonmises.cdf(a, k - h / 2)) / h
    J = -((4 * d2 - d1) / 3) / vonmises.pdf(a, k)
    return np.where(phi >= 0, -J, J)


@pytest.mark.parametrize("d", DS)
def test_new_forward_entry_draws_the_same_z(d):
    from clifford_b200._lib import ptr
    torch.manual_seed(d)
    B = _rows(d)
    loc = torch.randn(B, d, device=DEV)
    for rowk in (True, False):
        kap = _kappa_rows(B) if rowk else torch.rand(B, d, device=DEV) * 20
        z_old = torch.empty(B, 2 * d, device=DEV)
        krs, kes = (1, 0) if rowk else (d, 1)
        _entry("cvb_clifford_vm_rsample", ptr(loc), ptr(kap), krs, kes, B, 123, 7, ptr(z_old), B, d)
        z_new, phi = _draw(loc, kap, rowk)
        assert torch.equal(z_old, z_new), (d, rowk)
        if d > 1:
            # the saved offsets are the drawn phases: theta = loc + phi reproduces the spectrum's angles
            F = torch.fft.rfft(z_new.double(), dim=-1)[:, 1:d]
            dth = torch.angle(F) - (loc.double() + phi.double())[:, 1:]
            assert float(torch.remainder(dth + math.pi, 2 * math.pi).sub(math.pi).abs().max()) < 1e-4
    # the distribution: the same z with and without a graph, one generator step per call
    from dists.clifford import CliffordTorusDistribution
    kap = torch.rand(B, 1, device=DEV) * 5 + 0.1
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    zs = []
    for grad in (False, True):
        torch.manual_seed(5)
        l, k = loc.clone().requires_grad_(grad), kap.clone().requires_grad_(grad)
        o0 = gen.get_offset()
        zs.append(CliffordTorusDistribution(l, k).rsample(torch.Size([3])))
        assert gen.get_offset() == o0 + 4
    assert zs[0].grad_fn is None and zs[1].grad_fn is not None
    assert torch.equal(zs[0], zs[1].detach())


@pytest.mark.parametrize("d", DS)
def test_backward_dkappa_and_dloc_against_fp64(d):
    """dkappa against sum_k dL/dtheta_k * d phi_k / d kappa (SciPy CDF oracle); dloc against fp64 autograd of irfft."""
    from clifford_b200._lib import ptr
    torch.manual_seed(100 + d)
    B = _rows(d)
    S = 3
    loc = torch.randn(B, d, device=DEV)
    for rowk in (True, False):
        kap = _kappa_rows(B) if rowk else torch.logspace(-3, 3, B * d, device=DEV)[torch.randperm(B * d, device=DEV)].view(B, d)
        rows = S * B
        z = torch.empty(rows, 2 * d, device=DEV)
        phi = torch.zeros(rows, d, device=DEV)
        krs, kes = (1, 0) if rowk else (d, 1)
        _entry("cvb_clifford_vm_rsample_kl", ptr(loc), ptr(kap), krs, kes, B, 9, 1, ptr(z), ptr(phi), None, None, None, rows, d)
        gz = torch.randn(rows, 2 * d, device=DEV)
        dloc = torch.empty(rows, d, device=DEV)
        dk = torch.empty((rows,) if rowk else (rows, d), device=DEV)
        _entry("cvb_clifford_vm_rsample_backward", ptr(gz), ptr(loc), ptr(kap), krs, kes, B, ptr(phi), ptr(dloc), ptr(dk), rows, d)
        # fp64 reference: theta = loc + phi (phi held fixed), z = irfft of the unit Hermitian spectrum
        loc64 = loc.double().repeat(S, 1)
        th = (loc64 + phi.double()).requires_grad_()
        X = torch.polar(torch.ones_like(th), th)
        X = torch.cat([X, torch.ones(rows, 1, dtype=X.dtype, device=DEV)], dim=1)
        mask = torch.ones(d + 1, dtype=torch.float64, device=DEV)
        mask[0] = 0.0
        X = torch.where(mask.bool(), X, torch.ones_like(X))
        zr = torch.fft.irfft(X, n=2 * d, dim=-1)
        (zr * gz.double()).sum().backward()
        dth = th.grad.clone()
        dth[:, 0] = 0.0
        assert float((dloc.double() - dth).abs().max()) <= 1e-5 * max(1.0, float(dth.abs().max())), (d, rowk)
        k_el = (kap[:, None].expand(B, d) if rowk else kap).double().repeat(S, 1).cpu().numpy()
        J = torch.from_numpy(_oracle_dphi(phi.double().cpu().numpy(), k_el)).to(DEV)
        J[:, 0] = 0.0
        contrib = dth * J
        ref = contrib.sum(-1) if rowk else contrib
        tol = 2e-5 * torch.clamp(ref.abs(), min=1.0)
        assert bool(torch.isfinite(dk).all())
        assert bool(((dk.double() - ref).abs() <= tol).all()), (d, rowk, float((dk.double() - ref).abs().max()))


@pytest.mark.parametrize("k", [0.1, 2.0, 10.0, 50.0])
def test_pathwise_gradient_is_unbiased(k):
    """L(z) = sum_{k>=1} Re(rfft(z)_k e^{-i loc_k}) has E[L] = (d-1) A(kappa): the mean pathwise dL/dkappa over 2^16 rows
    equals (d-1)(1 - A/kappa - A^2) within 4 standard errors."""
    from scipy import special
    from dists.clifford import CliffordTorusDistribution
    torch.manual_seed(int(k * 10) + 1)
    B, d = 1 << 16, 512
    loc = torch.rand(B, d, device=DEV) * 6 - 3
    kap = torch.full((B, 1), k, device=DEV, requires_grad=True)
    z = CliffordTorusDistribution(loc, kap).rsample()
    F = torch.fft.rfft(z, dim=-1)[:, 1:d]
    L = (F * torch.polar(torch.ones_like(loc[:, 1:]), -loc[:, 1:])).real.sum(-1)
    g, = torch.autograd.grad(L.sum(), kap)
    g = g.double().reshape(-1)
    A = special.i1e(k) / special.i0e(k)
    expect = (d - 1) * (1 - A / k - A * A)
    se = float(g.std()) / math.sqrt(B)
    assert abs(float(g.mean()) - expect) < 4 * se + 1e-6 * abs(expect), (k, float(g.mean()), expect, se)


def _lp_ref(value, loc, kap):
    """fp64 torch restatement: a_k = angle(rfft(value)_k), sum_{k>=1} kappa cos(a - loc) - ln(2 pi I0(kappa))"""
    d = loc.shape[-1]
    a = torch.angle(torch.fft.rfft(value, dim=-1)[..., :d])
    kk = kap.expand_as(loc)
    t = kk * torch.cos(a - loc) - (math.log(2 * math.pi) + torch.log(torch.special.i0e(kk)) + kk)
    return t[..., 1:].sum(-1)


@pytest.mark.parametrize("d", DS)
def test_log_prob_value_and_gradients(d):
    from dists.clifford import CliffordTorusDistribution
    torch.manual_seed(200 + d)
    B, S = _rows(d), 3
    for rowk in (True, False):
        loc = torch.randn(B, d, device=DEV, requires_grad=True)
        kap = ((torch.rand(B, 1, device=DEV) * 20 + 0.05) if rowk else (torch.rand(B, d, device=DEV) * 20 + 0.05)).requires_grad_()
        q = CliffordTorusDistribution(loc, kap)
        with torch.no_grad():
            v = q.rsample(torch.Size([S])) + (0.01 / math.sqrt(2 * d)) * torch.randn(S, B, 2 * d, device=DEV)
        v.requires_grad_()
        lp = q.log_prob(v)
        assert lp.shape == (S, B)
        w = torch.randn(S, B, device=DEV)
        gv, gl, gk = torch.autograd.grad((lp * w).sum(), (v, loc, kap))
        v64, l64, k64 = (t.detach().double().requires_grad_() for t in (v, loc, kap))
        ref = _lp_ref(v64, l64, k64)
        rv, rl, rk = torch.autograd.grad((ref * w.double()).sum(), (v64, l64, k64))
        scale = float(ref.detach().abs().max()) + 1.0
        assert float((lp.double() - ref).abs().max()) <= 1e-5 * scale, (d, rowk)
        for got, want in ((gv, rv), (gl, rl), (gk, rk)):
            assert float((got.double() - want).abs().max()) <= 1e-5 * (float(want.abs().max()) + 1.0), (d, rowk)
        if d == 1:
            assert float(lp.abs().max()) == 0.0 and float(gv.abs().max()) == 0.0 and float(gk.abs().max()) == 0.0


@pytest.mark.parametrize("d", [16, 20, 300])
def test_log_prob_of_own_samples_estimates_the_entropy(d):
    from dists.clifford import CliffordTorusDistribution
    torch.manual_seed(d)
    B, S = 8, 4096
    q = CliffordTorusDistribution(torch.randn(B, d, device=DEV), torch.rand(B, 1, device=DEV) * 8 + 0.2)
    lp = q.log_prob(q.rsample(torch.Size([S])))
    assert lp.shape == (S, B)
    mc = -lp.double().mean(0)
    se = lp.double().std(0) / math.sqrt(S)
    assert bool(((mc - q.entropy().double()).abs() < 5 * se + 1e-3).all())


@pytest.mark.parametrize("d", DS)
def test_fused_entropy_and_kl(d):
    from clifford_b200._lib import ptr
    from dists.clifford import CliffordTorusDistribution, CliffordTorusUniform
    torch.manual_seed(300 + d)
    B = _rows(d)
    loc = torch.randn(B, d, device=DEV)
    kap = _kappa_rows(B)
    z = torch.empty(B, 2 * d, device=DEV)
    ent, kl, dent = (torch.empty(B, device=DEV) for _ in range(3))
    _entry("cvb_clifford_vm_rsample_kl", ptr(loc), ptr(kap), 1, 0, B, 1, 2, ptr(z), None, ptr(ent), ptr(kl), ptr(dent), B, d)
    ent_ref, dent_ref = torch.empty(B, device=DEV), torch.empty(B, device=DEV)
    _entry("cvb_clifford_vm_entropy", ptr(kap), 1, 0, B, d, ptr(ent_ref), ptr(dent_ref))
    assert torch.equal(ent, ent_ref) and torch.equal(dent, dent_ref)
    assert float((kl.double() - ((d - 1) * math.log(2 * math.pi) - ent_ref.double())).abs().max()) <= 1e-6 * (d + 1)
    # through the distribution: the cached entropy carries d/dkappa, KL to the uniform prior gets a gradient
    k1 = kap[:, None].clone().requires_grad_()
    q = CliffordTorusDistribution(loc, k1)
    q.rsample()
    kl_t = torch.distributions.kl.kl_divergence(q, CliffordTorusUniform(d, device=DEV))
    g, = torch.autograd.grad(kl_t.sum(), k1)
    # kl_divergence forms -H + (d-1) ln 2 pi in fp32: one rounding of the O(d) terms
    assert torch.allclose(kl_t.detach(), kl, rtol=1e-6, atol=4e-7 * (d + 1) * 1.84)
    assert torch.allclose(g.reshape(-1), -dent_ref, rtol=1e-6, atol=1e-6)
    if d > 1:
        assert float(g.abs().max()) > 0


@pytest.mark.parametrize("d", DS)
def test_robust_over_concentrations(d):
    from dists.clifford import CliffordTorusDistribution
    torch.manual_seed(400 + d)
    B = _rows(d)
    loc = torch.randn(B, d, device=DEV, requires_grad=True)
    kap = torch.logspace(-6, 4, B, device=DEV)[:, None].requires_grad_()
    q = CliffordTorusDistribution(loc, kap)
    z = q.rsample(torch.Size([3]))
    lp = q.log_prob(z)
    gl, gk, = torch.autograd.grad((z * torch.randn_like(z)).sum() + lp.sum() + q.entropy().sum(), (loc, kap))
    for t in (z, lp, gl, gk):
        assert bool(torch.isfinite(t).all()), d
    if d == 1:
        assert float(lp.abs().max()) == 0.0
    # per-element concentrations over the same range
    kap_e = torch.logspace(-6, 4, B * d, device=DEV).view(B, d).requires_grad_()
    q = CliffordTorusDistribution(loc, kap_e)
    z = q.rsample()
    gl, gk = torch.autograd.grad((z * torch.randn_like(z)).sum() + q.log_prob(z).sum(), (loc, kap_e))
    assert bool(torch.isfinite(gl).all() and torch.isfinite(gk).all()), d


def test_empty_batches_launch_nothing():
    from clifford_b200 import _lib
    from dists.clifford import CliffordTorusDistribution
    loc = torch.zeros(0, 16, device=DEV, requires_grad=True)
    kap = torch.ones(0, 1, device=DEV, requires_grad=True)
    q = CliffordTorusDistribution(loc, kap)
    _lib.ensure_device(torch.device(DEV))
    n0 = _lib.launch_count()
    z = q.rsample(torch.Size([2]))
    lp = q.log_prob(z)
    (z.sum() + lp.sum()).backward()
    assert z.shape == (2, 0, 32) and lp.shape == (2, 0)
    assert _lib.launch_count() == n0


def test_vae_training_step_reaches_both_encoder_heads():
    from dists.clifford import CliffordTorusDistribution, CliffordTorusUniform
    torch.manual_seed(0)
    B, D, d = 64, 784, 20
    enc = torch.nn.Sequential(torch.nn.Linear(D, 256), torch.nn.ReLU()).to(DEV)
    fc_loc, fc_k = torch.nn.Linear(256, d).to(DEV), torch.nn.Linear(256, 1).to(DEV)
    dec = torch.nn.Sequential(torch.nn.Linear(2 * d, 256), torch.nn.ReLU(), torch.nn.Linear(256, D)).to(DEV)
    x = torch.rand(B, D, device=DEV)
    h = enc(x)
    q = CliffordTorusDistribution(fc_loc(h), torch.nn.functional.softplus(fc_k(h)) + 0.03)
    z = q.rsample()
    rec = torch.nn.functional.binary_cross_entropy_with_logits(dec(z), x, reduction="none").sum(-1)
    kl = torch.distributions.kl.kl_divergence(q, CliffordTorusUniform(d, device=DEV))
    (rec + kl).mean().backward()
    for p in (fc_loc.weight, fc_k.weight, enc[0].weight):
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()) and float(p.grad.abs().max()) > 0
    # the reconstruction term alone reaches both heads (through the sample, not only through the KL)
    for p in (fc_loc, fc_k, enc, dec):
        p.zero_grad()
    h = enc(x)
    q = CliffordTorusDistribution(fc_loc(h), torch.nn.functional.softplus(fc_k(h)) + 0.03)
    torch.nn.functional.binary_cross_entropy_with_logits(dec(q.rsample()), x).backward()
    assert float(fc_loc.weight.grad.abs().max()) > 0 and float(fc_k.weight.grad.abs().max()) > 0
