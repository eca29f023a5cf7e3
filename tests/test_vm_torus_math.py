"""CPU checks of the von Mises torus reparameterisation math (no GPU): the closed-form implicit gradient d phi / d kappa
that csrc/clifford_kernels.cuh (vm_dphi_dkappa) integrates, against SciPy's von Mises CDF; a float32 restatement of
the kernel's quadrature against the same oracle; and the C-ABI table entries of the new entry points."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KAPPAS = [1e-3, 0.05, 1.0, 4.0, 10.0, 32.0, 100.0, 1e3]


def _A(k):
    from scipy import special
    return special.i1e(k) / special.i0e(k)


def _closed_form(phi, k):
    """-int_0^phi (cos t - A) e^{k (cos t - cos phi)} dt, integrated from the side without cancellation."""
    from scipy import integrate
    A, a = _A(k), abs(phi)
    f = lambda t: (np.cos(t) - A) * np.exp(k * (np.cos(t) - np.cos(a)))
    if np.cos(a) >= A:
        v = -integrate.quad(f, 0.0, a, epsabs=0.0, epsrel=1e-13, limit=200)[0]
    else:
        v = integrate.quad(f, a, np.pi, epsabs=0.0, epsrel=1e-13, limit=200)[0]
    return v if phi >= 0 else -v


def _oracle(phi, k):
    """-d_kappa F / f by central differences of scipy's CDF, on the lower tail (J is odd in phi)."""
    from scipy.stats import vonmises
    a = -abs(phi)
    h = 1e-4 * max(k, 1e-2)
    d1 = (vonmises.cdf(a, k + h) - vonmises.cdf(a, k - h)) / (2 * h)
    d2 = (vonmises.cdf(a, k + h / 2) - vonmises.cdf(a, k - h / 2)) / h
    dF = (4 * d2 - d1) / 3                              # Richardson: O(h^4)
    J = -dF / vonmises.pdf(a, k)                         # J(-|phi|)
    return -J if phi >= 0 else J


def _phis(k, xmax=32.0):
    """a grid over the bulk and the tails of VonMises(0, k), up to ~8 standard deviations: draws whose density is down
    to e^-xmax of the mode's"""
    sd = 1.0 / np.sqrt(k) if k > 1 else 1.5
    grid = [0.01, 0.2, 0.9, 2.0, 2.9, 3.1] + list(np.linspace(0.1, 8.0, 12) * sd)
    return [p for p in grid if p < np.pi and k * (1 - np.cos(p)) < xmax]


@pytest.mark.parametrize("k", KAPPAS)
def test_closed_form_matches_scipy_cdf_oracle(k):
    # tail draws to density e^-14 of the mode (beyond it the CDF differences lose the digits, not the closed form: the
    # deeper tails are checked against adaptive quadrature of the closed form below)
    # scipy's CDF switches to a normal approximation for kappa >= 50: its own error on J reaches 1.4e-6 there (tails)
    tol = 1e-7 if k < 50 else 5e-6
    for p in _phis(k, 14.0):
        for phi in (p, -p):
            ref = _oracle(phi, k)
            got = _closed_form(phi, k)
            assert abs(got - ref) <= tol * max(1.0, abs(ref)), (k, phi, got, ref)


def _kernel_quadrature_f32(phi, k):
    """float32 restatement of vm_dphi_dkappa (12-point Gauss-Legendre panels; see its comment)."""
    F = np.float32
    x01, w = np.polynomial.legendre.leggauss(12)
    u, w = ((x01 + 1) / 2).astype(F), (w / 2).astype(F)
    k = F(k)
    a = F(abs(phi))
    b = F(-np.expm1(np.log(_A(float(k))))) if k > 0 else F(1)
    S, C = np.sin(a / F(2), dtype=F), np.cos(a / F(2), dtype=F)
    x = F(2) * k * S * S
    if x <= 3:
        t = a * u
        st = np.sin(t / F(2))
        e = F(2) * k * np.sin((a + t) / F(2)) * np.sin((a - t) / F(2))
        J = -a * np.sum(w * (b - F(2) * st * st) * np.exp(e), dtype=F)
    else:
        cma = b - F(2) * S * S
        r = S / C
        e1 = np.arcsinh(min(F(0.70710678) / r, np.sqrt(F(40) / x)))
        sh = np.sinh(e1 * u)
        sp = r * sh
        J = e1 * np.sum(w * (cma - F(2) * S * S * sh * sh) * np.exp(-x * sh * sh) * F(2) * sp / np.sqrt(F(1) - sp * sp),
                        dtype=F)
        if k * C * C < 40:
            sp = np.sin(F(0.78539816) * (F(1) + u))
            c2s2 = C * C * sp * sp
            J += F(0.78539816) * np.sum(w * (cma - F(2) * c2s2) * np.exp(-F(2) * k * c2s2) * F(2) * C * sp
                                        / np.sqrt(S * S + c2s2), dtype=F)
    return float(J if phi >= 0 else -J)


@pytest.mark.parametrize("k", KAPPAS + [1e-6, 1.5, 19.5, 1e4])
def test_kernel_quadrature_meets_the_accuracy_bar(k):
    """The fp32 quadrature of the backward kernel within 2e-6 max(1, |J|) of the closed form (the GPU backward test
    allows 2e-5 on row sums)."""
    for p in _phis(k) + [np.pi - 1e-3]:
        ref = _closed_form(p, k)
        got = _kernel_quadrature_f32(p, k)
        assert np.isfinite(got) and abs(got - ref) <= 2e-6 * max(1.0, abs(ref)), (k, p, got, ref)
    assert _kernel_quadrature_f32(0.0, k) == 0.0


def test_small_concentration_limit():
    for p in (0.3, 1.7, 3.0):
        assert abs(_closed_form(p, 1e-9) + np.sin(p)) < 1e-8


def test_new_entry_points_in_header_and_ctypes_table():
    from clifford_b200 import _lib
    src = open(os.path.join(ROOT, "include", "clifford_b200.h")).read()
    arity = {"cvb_clifford_vm_rsample_kl": 15, "cvb_clifford_vm_rsample_backward": 12, "cvb_clifford_vm_log_prob": 13}
    for name, n in arity.items():
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", src, re.S)
        assert m, name
        assert m.group(1).count(",") + 1 == n, name
        assert len(_lib._SIGNATURES[name][0]) == n and name in _lib.EXPORTED_SYMBOLS
    # the forward-only entry keeps its signature
    assert len(_lib._SIGNATURES["cvb_clifford_vm_rsample"][0]) == 11
