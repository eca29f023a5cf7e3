"""GPU: the FFT-engine Clifford kernels at all ten lengths (d = 16 .. 8192) with enough rows that every group of threads
loops over rows, against float64 references.

The kernels are persistent: once the rows outnumber the groups a grid holds, each group takes further rows (from a
dynamic-schedule slot where its FFT has >= 32 threads) and carries state from one row to the next -- the inverse-CDF
cells of table-sampled rows, the prefetched next row's kappa and staged inputs, a table row's phasors in registers, the
bind spectrum.  An SM holds at most 2048 threads and a group is T = d / E threads (E = 4 points per thread below d = 64,
8 at 64 and 128, 16 from 256), so rows = 3 * SMs * 2048 / T + 37 make every group take several rows whatever the grid.

Deterministic calls get inputs periodic in the row with a prime period P: the first P rows are compared with the
float64 oracle on the CPU, every other row must be bitwise equal to row r mod P.  The log_prob kernels are held to 1e-6
relative there instead, because clifford_log_prob_kernel takes a row's constants from a per-group cache or recomputes
them depending on the row's position (test_gpu_clifford_tiers.test_log_prob_past_the_row_constant_cache).  Device-RNG
calls are compared with the oracle on their own saved draws on 64 rows: the first 16, the last 16 (taken in a group's
final iterations) and 32 seeded random ones.  Every case runs with loc / kappa materialised to all rows and with
loc_rows = P (the kernels' row % loc_rows).  Outputs start NaN-filled inside NaN guards: a row no group claimed, or a
store past the end, fails.  Tolerances are the suite's (test_gpu_clifford_tiers' docstring)."""
import math

import pytest
import torch

from conftest import rel_err
from test_gpu_clifford_tiers import (DEV, Out, _kappa_el, assert_log_prob, call, dev, make_inputs, ref_entropy,
                                     ref_log_prob, ref_rsample, run_backward, run_log_prob, run_rsample, tprime_and_sign,
                                     value_near)
from test_gpu_clifford_vm import _lp_ref, _oracle_dphi

FFT = [16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]
LOC_ROWS = ["loc_rows=rows", "loc_rows=P"]
# row concentrations on both sides of 1/pi and of 32 (the inverse-CDF table's range: table-sampled vs exact rows)
KAPPAS = [0.03, 0.1, 0.25, 0.3, 0.35, 0.5, 1.0, 2.0, 4.0, 8.0, 16.0, 31.9, 32.5, 40.0, 64.0, 100.0]
SEED, OFFSET = 11, 5                    # run_rsample's device-RNG key


@pytest.fixture(scope="module")
def keyed_draws():
    """device draws keyed by (seed, offset) alone: no launch counter left registered by an earlier graph capture"""
    from clifford_b200 import _lib
    _lib.ensure_device(torch.device(DEV))
    _lib.check(_lib.load().cvb_set_rng_device_counter(None), "cvb_set_rng_device_counter")


def gpu(f):
    return pytest.mark.gpu(pytest.mark.usefixtures("keyed_draws")(f))


def period(d):
    return 13 if d >= 4096 else 61


def n_rows(d):
    """3 * SMs * 2048 / T + 37: more than three times the groups any grid of this length can hold"""
    e = 4 if d < 64 else (8 if d < 256 else 16)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return 3 * sms * 2048 // (d // e) + 37


def tile(t, rows):
    """a device copy of t (P, ...) repeated to `rows` rows: row r is row r mod P"""
    P = t.shape[0]
    return t.to(DEV).repeat((rows + P - 1) // P, *([1] * (t.dim() - 1)))[:rows].contiguous()


def params(loc, kap, rows, lr):
    """loc / kappa on the device: materialised to `rows` rows, or P rows read through row % loc_rows"""
    return (tile(loc, rows), tile(kap, rows)) if lr == LOC_ROWS[0] else (dev(loc), dev(kap))


def guarded(o):
    torch.cuda.synchronize()
    assert o.guards_intact()
    return o.t


def periodic(t, P, rel=0.0):
    """every row of t equals row r mod P: bitwise, or to `rel` relative (checked on the GPU in chunks)"""
    rows = t.shape[0]
    step = P * max(1, (1 << 22) // (P * max(1, t[0].numel())))
    for i in range(0, rows, step):
        got = t[i:i + step]
        want = t[:P][torch.arange(i, i + got.shape[0], device=DEV) % P]
        same = torch.equal(got, want) if rel == 0 else bool(((got - want).abs() <= rel * want.abs()).all())
        assert same, f"rows {i}..{i + got.shape[0]} differ from their period"


def gpu_rel(x, ref):
    """max-norm relative error on the GPU (NaN fails)"""
    err = float((x.double() - ref.double()).abs().max())
    return err / max(float(ref.double().abs().max()), 1e-30) if err == err else math.inf


def per_row(t, P, rows):
    """the float64 row values of P distinct rows, expanded on the GPU to all rows"""
    return t.double().to(DEV)[torch.arange(rows, device=DEV) % P]


def sampled_rows(rows, n=64, seed=0):
    """the first n/4 rows, the last n/4 and n/2 seeded random rows in between"""
    q = n // 4
    gen = torch.Generator().manual_seed(seed)
    mid = torch.randperm(rows - 2 * q, generator=gen)[:n - 2 * q].sort().values + q
    return torch.cat([torch.arange(q), mid, torch.arange(rows - q, rows)])


def cycling_kappa(P):
    return torch.tensor([KAPPAS[(3 * p) % len(KAPPAS)] for p in range(P)])


def draws_of(saved, kap, d):
    """(t', sign) of a device-RNG forward's saved draws, row by row: table coordinates on table-sampled rows (one
    concentration <= 32 per row at d >= 512), copysign(t', s) elsewhere"""
    tp, sgn = tprime_and_sign(saved, kap, d, False)
    if kap.dim() == 1 and d >= 512:
        tab = kap + 1e-7 <= 32.0
        if bool(tab.any()):
            tp[tab] = tprime_and_sign(saved[tab], kap[tab], d, True)[0]
    return tp, sgn


def bind64(a, b):
    """the float64 bind (circular convolution) of rows of a and b, on a's device"""
    from oracle import latent_oracle as O
    return O.bind(a.double(), b.double().to(a.device))


def vm_z_from_theta(theta):
    """the von Mises torus sample of phases theta (rows, d): irfft of the unit Hermitian spectrum with bins 0 and d
    equal to 1, in float64 (theta[:, 0] ignored)"""
    rows, d = theta.shape
    X = torch.polar(torch.ones_like(theta[:, 1:]), theta[:, 1:])
    one = torch.ones(rows, 1, dtype=X.dtype, device=X.device)
    return torch.fft.irfft(torch.cat([one, X, one], dim=1), n=2 * d, dim=-1)


def test_new_references_run_on_cpu():
    """bind64 is the circular convolution; vm_z_from_theta is the oracle's phases -> vector map"""
    from oracle import latent_oracle as O
    gen = torch.Generator().manual_seed(3)
    a, b = (torch.randn(3, 10, generator=gen, dtype=torch.float64) for _ in range(2))
    conv = torch.stack([sum(a[:, j] * b[:, (i - j) % 10] for j in range(10)) for i in range(10)], dim=1)
    assert rel_err(bind64(a, b), conv) < 1e-12
    assert rel_err(bind64(a, b[:1]), bind64(a, b[:1].expand(3, 10))) < 1e-12
    u = torch.rand(4, 9, generator=gen, dtype=torch.float64)
    assert rel_err(vm_z_from_theta(2 * math.pi * u), O.clifford_uniform_rsample(u)) < 1e-12
    th = u.clone().requires_grad_()
    (vm_z_from_theta(th) * torch.randn(4, 18, generator=gen, dtype=torch.float64)).sum().backward()
    assert float(th.grad[:, 0].abs().max()) == 0.0


def check_entropies(ent, kl, dent, kap, d, P, rows):
    """row entropy / KL / dH/dkappa of every row against float64 of the P distinct concentrations"""
    e_ref, kl_ref, de_ref = ref_entropy(_kappa_el(kap, P, d))
    assert gpu_rel(guarded(ent), per_row(e_ref, P, rows)) < 1e-5
    assert float((guarded(kl).double() - per_row(kl_ref, P, rows)).abs().max()) < 1e-5 * (d - 1) * math.log(2 * math.pi)
    assert gpu_rel(guarded(dent), per_row(de_ref.sum(-1), P, rows)) < 2e-5


# ---- 1. injected draws: rsample, backward, log_prob -----------------------------------------------------------------
@gpu
@pytest.mark.parametrize("lr", LOC_ROWS)
@pytest.mark.parametrize("rowk", [True, False], ids=["rowk", "elk"])
@pytest.mark.parametrize("d", FFT)
def test_injected_draws(d, rowk, lr):
    P, rows = period(d), n_rows(d)
    loc, kap, tp, g, gz = make_inputs(d, rowk, P, P, seed=3 * d + rowk)
    locd, kapd = params(loc, kap, rows, lr)
    tpd, gd, gzd = tile(tp, rows), tile(g, rows), tile(gz, rows)
    z_ref, dl_ref, dk_ref = ref_rsample(loc, kap, tp, g, gz)
    rc, z, _, ent, kl, dent = run_rsample(locd, kapd, tpd, gd, d, rows, entropy=rowk)
    assert rc == 0
    assert rel_err(guarded(z)[:P].cpu(), z_ref) < 1e-5
    periodic(z.t, P)
    if rowk:
        check_entropies(ent, kl, dent, kap, d, P, rows)
        for o in (ent, kl, dent):
            periodic(o.t, P)
    del z, ent, kl, dent

    rc, dl, dk = run_backward(gzd, locd, kapd, tpd, gd, None, d, rows)
    assert rc == 0
    assert rel_err(guarded(dl)[:P].cpu(), dl_ref) < 5e-5
    assert rel_err(guarded(dk)[:P].cpu(), dk_ref) < 5e-4
    periodic(dl.t, P)
    periodic(dk.t, P)
    del dl, dk, tpd, gd, gzd

    _, _, tpc, gc, _ = make_inputs(d, rowk, P, P, seed=3 * d + rowk, clamp=1e-3)
    value = value_near(ref_rsample(loc, kap, tpc, gc, gz)[0], seed=d)
    ref = ref_log_prob(value, loc, kap)
    vd = tile(value, rows)
    rc, lp, dl, dk, dF = run_log_prob(vd, locd, kapd, d, rows)
    assert rc == 0
    assert_log_prob(tuple(guarded(o)[:P].cpu() for o in (lp, dl, dk, dF)), ref)
    for o in (lp, dl, dk, dF):
        periodic(o.t, P, rel=1e-6)         # clifford_log_prob_kernel: cached or recomputed row constants
    del lp, dl, dk, dF
    rc, lp, _, _, _ = run_log_prob(vd, locd, kapd, d, rows, grads=False)
    assert rc == 0
    assert_log_prob((guarded(lp)[:P].cpu(), None, None, None), ref)
    periodic(lp.t, P, rel=1e-6)


# ---- 2 + 3. device RNG with saved draws, the training-path backward, and the lean sampler ---------------------------
def check_rng_rows(z, tps, dl, dk, rows_s, loc, kap, gz, d):
    """sample, dloc and dkappa of one-concentration-per-row device-RNG rows `rows_s` against the oracle on the draws the
    forward saved (test_rng_mode_invariants_and_backward_vs_oracle, test_mixed_table_and_exact_rows_backward_vs_oracle)"""
    P = loc.shape[0]
    pr = rows_s % P
    loc_s, kap_s, gz_s = loc[pr], kap[pr], gz[pr]
    saved = tps[rows_s].cpu()
    assert not bool(torch.isnan(saved[:, 1:]).any())
    tp, sgn = draws_of(saved, kap_s, d)
    z_ref, dl_ref, dk_ref = ref_rsample(loc_s, kap_s, tp, sgn, gz_s)
    assert rel_err(z[rows_s].cpu(), z_ref) < 2e-5
    got_dl, got_dk = dl[rows_s].cpu(), dk[rows_s].cpu()
    # table rows: the oracle is driven through t' = cos^2(phi / 2) in fp32 (see test_rng_mode_invariants_...)
    assert rel_err(got_dl[:, 1:], dl_ref[:, 1:]) < (3e-4 if d >= 512 else 5e-5)
    table = (kap_s + 1e-7 <= 32.0) & (d >= 512)
    exact_low = (kap_s + 1e-7 <= 32.0) & (d < 512)
    if bool(table.any()):
        assert rel_err(got_dk[table], dk_ref[table]) < 2e-3
    if bool(exact_low.any()):
        assert rel_err(got_dk[exact_low], dk_ref[exact_low]) < 5e-4
    for r in torch.nonzero(kap_s + 1e-7 > 32.0).reshape(-1).tolist():
        # row by row: the high-concentration rows have small gradients that a max-norm over the batch would hide
        assert abs(float(got_dk[r]) - float(dk_ref[r])) < 3e-3 * max(abs(float(dk_ref[r])), 1e-3), (int(rows_s[r]), float(kap_s[r]))


def lean_matches_full(locd, kapd, d, rows, z, ent, kl, dent):
    """the lean sampler (no saved draws: the headline call) against the full one of the same (seed, offset): z at 1e-5;
    entropy / KL / dH/dkappa from the same fp64 prologue to 1e-6 (returns whether they are bitwise equal)"""
    rc, zl, _, el, kll, dl = run_rsample(locd, kapd, None, None, d, rows, entropy=True)
    assert rc == 0
    assert gpu_rel(guarded(zl), z) < 1e-5
    bitwise = True
    for a, b in ((el, ent), (kll, kl), (dl, dent)):
        a = guarded(a)
        assert bool(((a - b).abs() <= 1e-6 * b.abs()).all())
        bitwise &= torch.equal(a, b)
    return zl, bitwise


@gpu
@pytest.mark.parametrize("lr", LOC_ROWS)
@pytest.mark.parametrize("d", FFT)
def test_device_rng_row_kappa_and_lean_sampler(d, lr):
    P, rows = period(d), n_rows(d)
    gen = torch.Generator().manual_seed(d)
    loc = torch.randn(P, d, generator=gen) * 2
    kap = cycling_kappa(P)
    gz = torch.randn(P, 2 * d, generator=gen)
    locd, kapd = params(loc, kap, rows, lr)
    rc, z, tps, ent, kl, dent = run_rsample(locd, kapd, None, None, d, rows, save=True, entropy=True)
    assert rc == 0
    rc, dl, dk = run_backward(tile(gz, rows), locd, kapd, None, None, guarded(tps), d, rows)
    assert rc == 0
    check_rng_rows(guarded(z), tps.t, guarded(dl), guarded(dk), sampled_rows(rows, seed=d), loc, kap, gz, d)
    check_entropies(ent, kl, dent, kap, d, P, rows)
    del tps, dl, dk
    _, bitwise = lean_matches_full(locd, kapd, d, rows, z.t, ent.t, kl.t, dent.t)
    print(f"d={d} {lr}: lean entropy / KL / dH bitwise equal to the full sampler's: {bitwise}")

    if d == 2048:
        # the benchmark's shape: B = 4096 rows, one loc row each
        B = 4096
        loc = torch.randn(B, d, generator=gen) * 2
        kap = cycling_kappa(B)
        gz = torch.randn(B, 2 * d, generator=gen)
        locd, kapd = dev(loc), dev(kap)
        rc, z, tps, ent, kl, dent = run_rsample(locd, kapd, None, None, d, B, save=True, entropy=True)
        assert rc == 0
        rc, dl, dk = run_backward(dev(gz), locd, kapd, None, None, guarded(tps), d, B)
        assert rc == 0
        check_rng_rows(guarded(z), tps.t, guarded(dl), guarded(dk), sampled_rows(B, seed=1), loc, kap, gz, d)
        check_entropies(ent, kl, dent, kap, d, B, B)
        _, bitwise = lean_matches_full(locd, kapd, d, B, z.t, ent.t, kl.t, dent.t)
        print(f"d={d} B={B}: lean entropy / KL / dH bitwise equal to the full sampler's: {bitwise}")


@gpu
@pytest.mark.parametrize("lr", LOC_ROWS)
@pytest.mark.parametrize("d", FFT)
def test_device_rng_element_kappa(d, lr):
    """per-element concentrations, log-uniform in [0.03, 100] (no table: copysign(t', s) saved on every row).  Besides
    the oracle on the kernel's own draws: each circle's draws follow that circle's Beta(1/2 + kappa + 1e-7, 1/2) law --
    the summed deviation of t' from its mean, over all rows, within 6 standard deviations for every circle"""
    P, rows = period(d), n_rows(d)
    gen = torch.Generator().manual_seed(d + 1)
    loc = torch.randn(P, d, generator=gen) * 2
    kap = torch.exp(torch.rand(P, d, generator=gen) * math.log(100 / 0.03) + math.log(0.03))
    gz = torch.randn(P, 2 * d, generator=gen)
    locd, kapd = params(loc, kap, rows, lr)
    rc, z, tps, _, _, _ = run_rsample(locd, kapd, None, None, d, rows, save=True)
    assert rc == 0
    rc, dl, dk = run_backward(tile(gz, rows), locd, kapd, None, None, guarded(tps), d, rows)
    assert rc == 0
    rows_s = sampled_rows(rows, seed=d)
    pr = rows_s % P
    tp, sgn = tprime_and_sign(tps.t[rows_s].cpu(), kap, d, False)
    z_ref, dl_ref, dk_ref = ref_rsample(loc[pr], kap[pr], tp, sgn, gz[pr])
    assert rel_err(guarded(z)[rows_s].cpu(), z_ref) < 2e-5
    assert rel_err(guarded(dl)[rows_s].cpu(), dl_ref) < 5e-5
    assert rel_err(guarded(dk)[rows_s].cpu(), dk_ref) < 5e-4
    del z, dl, dk
    a = 0.5 + tile(kap, rows)[:, 1:].double() + 1e-7
    dev_sum = (tps.t[:, 1:].abs().double() - a / (a + 0.5)).sum(0)
    sd = (a * 0.5 / ((a + 0.5) ** 2 * (a + 1.5))).sum(0).sqrt()
    zscore = (dev_sum / sd).abs()
    assert float(zscore.max()) < 6.0, int(zscore.argmax()) + 1


# ---- 4. fused sample + bind ------------------------------------------------------------------------------------------
def run_bind(locd, kapd, tpd, gd, bd, d, rows, with_z):
    z = Out(rows, 2 * d) if with_z else None
    bound = Out(rows, 2 * d)
    e = [Out(rows) for _ in range(3)]
    rc = call("cvb_clifford_ps_rsample_bind", locd.data_ptr(), kapd.data_ptr(), locd.shape[0],
              None if tpd is None else tpd.data_ptr(), None if gd is None else gd.data_ptr(), SEED, OFFSET, bd.data_ptr(),
              bd.shape[0], None if z is None else z.p, bound.p, e[0].p, e[1].p, e[2].p, rows, d)
    return rc, z, bound, e[0], e[1], e[2]


@gpu
@pytest.mark.parametrize("lr", LOC_ROWS)
@pytest.mark.parametrize("d", FFT)
def test_rsample_bind(d, lr):
    P, rows = period(d), n_rows(d)
    loc, kap, tp, g, gz = make_inputs(d, True, P, P, seed=5 * d)
    b = torch.randn(P, 2 * d, generator=torch.Generator().manual_seed(d)) / (2 * d) ** 0.5
    locd, kapd = params(loc, kap, rows, lr)
    tpd, gd = tile(tp, rows), tile(g, rows)
    z_ref = ref_rsample(loc, kap, tp, g, gz)[0]
    for b_rows in (rows, 1):
        bd = tile(b, rows) if b_rows == rows else dev(b[:1])
        want = bind64(z_ref, b if b_rows == rows else b[:1])
        for with_z in (True, False):
            rc, z, bound, ent, kl, dent = run_bind(locd, kapd, tpd, gd, bd, d, rows, with_z)
            assert rc == 0
            if with_z:
                assert rel_err(guarded(z)[:P].cpu(), z_ref) < 1e-5
                periodic(z.t, P)
            assert rel_err(guarded(bound)[:P].cpu(), want) < 2e-5, (b_rows, with_z)
            periodic(bound.t, P)
            check_entropies(ent, kl, dent, kap, d, P, rows)
            for o in (ent, kl, dent):
                periodic(o.t, P)
            del z, bound, ent, kl, dent
    del tpd, gd
    # device RNG: the same key and sampler as cvb_clifford_ps_rsample's, so the lean call's z; bound = bind(z, b)
    bd = tile(b, rows)
    rc, z, bound, _, _, _ = run_bind(locd, kapd, None, None, bd, d, rows, True)
    assert rc == 0
    rc, zl, _, _, _, _ = run_rsample(locd, kapd, None, None, d, rows)
    assert rc == 0
    assert gpu_rel(guarded(z), guarded(zl)) < 1e-5
    del zl
    err = top = 0.0
    got = guarded(bound)
    step = max(1, (1 << 21) // d)
    for i in range(0, rows, step):
        want = bind64(z.t[i:i + step], bd[i:i + step])
        err = max(err, float((got[i:i + step].double() - want).abs().max()))
        top = max(top, float(want.abs().max()))
    assert err < 2e-5 * top, err / top


# ---- 5. fused sample + log q ----------------------------------------------------------------------------------------
def run_rsample_log_prob(locd, kapd, tpd, gd, d, rows):
    z, lp, ent, kl = Out(rows, 2 * d), Out(rows), Out(rows), Out(rows)
    rc = call("cvb_clifford_ps_rsample_log_prob", locd.data_ptr(), kapd.data_ptr(), locd.shape[0],
              None if tpd is None else tpd.data_ptr(), None if gd is None else gd.data_ptr(), SEED, OFFSET, z.p, lp.p,
              ent.p, kl.p, rows, d)
    return rc, z, lp, ent, kl


@gpu
@pytest.mark.parametrize("lr", LOC_ROWS)
@pytest.mark.parametrize("d", FFT)
def test_rsample_log_prob(d, lr):
    P, rows = period(d), n_rows(d)
    loc, kap, tp, g, gz = make_inputs(d, True, P, P, seed=7 * d)
    locd, kapd = params(loc, kap, rows, lr)
    z_ref = ref_rsample(loc, kap, tp, g, gz)[0]
    rc, z, lp, ent, kl = run_rsample_log_prob(locd, kapd, tile(tp, rows), tile(g, rows), d, rows)
    assert rc == 0
    assert rel_err(guarded(z)[:P].cpu(), z_ref) < 1e-5
    # log q is the density at the draw (t', s): the oracle's sample of s = sign(g) (its s = g / (|g| + 1e-7) moves the
    # phase of a circle whose |g| is small, which the sample z follows but log q does not)
    z_draw = ref_rsample(loc, kap, tp, torch.sign(g), gz)[0]
    assert_log_prob((guarded(lp)[:P].cpu(), None, None, None), ref_log_prob(z_draw, loc, kap))
    for o in (z, lp, ent, kl):
        periodic(o.t, P)                  # log_prob: two addends onto zero, order-independent
    e_ref, kl_ref, _ = ref_entropy(_kappa_el(kap, P, d))
    assert rel_err(ent.t[:P].cpu(), e_ref) < 1e-5
    assert float((kl.t[:P].cpu().double() - kl_ref).abs().max()) < 1e-5 * (d - 1) * math.log(2 * math.pi)
    del z, lp, ent, kl
    # device RNG: the full sampler with log q makes the draws it makes with saved draws (z bitwise equal), and the lean
    # sampler's z to 1e-5.  log q(z) against float64 of those saved draws on the sampled rows, with the conditioning of
    # the draws' float32 t' (1 + cos(theta - loc) = 2 t').  (The stand-alone log_prob kernel is no reference here: it
    # reads the float32 z, which does not resolve a t' of 1e-7.)
    rc, z, lp, _, _ = run_rsample_log_prob(locd, kapd, None, None, d, rows)
    assert rc == 0
    rc, zs, tps, _, _, _ = run_rsample(locd, kapd, None, None, d, rows, save=True)
    assert rc == 0
    assert torch.equal(guarded(z), guarded(zs))
    del zs
    rc, zl, _, _, _, _ = run_rsample(locd, kapd, None, None, d, rows)
    assert rc == 0
    assert gpu_rel(z.t, guarded(zl)) < 1e-5
    del zl
    from oracle import latent_oracle as O
    rows_s = sampled_rows(rows, seed=d)
    pr = rows_s % P
    saved = guarded(tps)[rows_s].cpu()
    assert not bool(torch.isnan(saved[:, 1:]).any())
    tp_s = draws_of(saved, kap[pr], d)[0].double()[:, 1:].clamp(5.9604645e-8, 0.99999994)
    k = kap[pr].double()
    c0 = torch.cos(loc[pr, 0].double()).clamp(-1 + 1e-7, 1 - 1e-7)
    want = (d * O.ps_log_normalizer(k[:, None].expand(-1, d), 2)[:, 0] + k * ((d - 1) * math.log(2) + torch.log1p(c0)) +
            k * torch.log(tp_s).sum(-1))
    got = guarded(lp)[rows_s].cpu().double()
    bound = 2e-5 * want.abs() + k * (4e-7 / (2 * tp_s)).sum(-1) + 1e-6
    assert bool(((got - want).abs() <= bound).all()), float((got - want).abs().max())


# ---- 6. the von Mises family ----------------------------------------------------------------------------------------
def vm_kappa(P, d, rowk, gen):
    """concentrations from 1e-3 to 1e3, log-spaced and shuffled: (P,) or (P, d)"""
    n = P if rowk else P * d
    k = torch.logspace(-3, 3, n)[torch.randperm(n, generator=gen)]
    # kept 1 % away from 50, where SciPy's von Mises CDF changes approximation: the oracle's difference quotient must
    # not straddle it
    k = torch.where((k / 50 - 1).abs() < 1e-2, k * 1.03, k)
    return k if rowk else k.view(P, d)


@gpu
@pytest.mark.parametrize("lr", LOC_ROWS)
@pytest.mark.parametrize("rowk", [True, False], ids=["rowk", "elk"])
@pytest.mark.parametrize("d", FFT)
def test_von_mises(d, rowk, lr):
    P, rows = period(d), n_rows(d)
    gen = torch.Generator().manual_seed(d + 2 * rowk)
    loc = torch.randn(P, d, generator=gen)
    kap = vm_kappa(P, d, rowk, gen)
    gz = torch.randn(P, 2 * d, generator=gen)
    locd, kapd = params(loc, kap, rows, lr)
    krs, kes = (1, 0) if rowk else (d, 1)
    L = locd.shape[0]
    z0 = Out(rows, 2 * d)
    assert call("cvb_clifford_vm_rsample", locd.data_ptr(), kapd.data_ptr(), krs, kes, L, 9, 1, z0.p, rows, d) == 0
    z, phi = Out(rows, 2 * d), Out(rows, d)
    e = [Out(rows) for _ in range(3)] if rowk else [None] * 3
    pp = (lambda o: None if o is None else o.p)
    assert call("cvb_clifford_vm_rsample_kl", locd.data_ptr(), kapd.data_ptr(), krs, kes, L, 9, 1, z.p, phi.p, pp(e[0]),
                pp(e[1]), pp(e[2]), rows, d) == 0
    assert torch.equal(guarded(z), guarded(z0))
    del z0
    if rowk:
        kapm = tile(kap, rows)
        ent, dent = Out(rows), Out(rows)
        assert call("cvb_clifford_vm_entropy", kapm.data_ptr(), 1, 0, rows, d, ent.p, dent.p) == 0
        assert torch.equal(guarded(e[0]), guarded(ent)) and torch.equal(guarded(e[2]), guarded(dent))
        kl_want = (d - 1) * math.log(2 * math.pi) - ent.t.double()
        assert float((guarded(e[1]).double() - kl_want).abs().max()) <= 1e-6 * (d + 1)

    # the sample and the backward on sampled rows: z from the saved offsets, dloc by float64 autograd, dkappa by the
    # SciPy CDF oracle
    dlo, dk = Out(rows, d), (Out(rows) if rowk else Out(rows, d))
    assert call("cvb_clifford_vm_rsample_backward", tile(gz, rows).data_ptr(), locd.data_ptr(), kapd.data_ptr(), krs, kes,
                L, guarded(phi).data_ptr(), dlo.p, dk.p, rows, d) == 0
    rows_s = sampled_rows(rows, n=16 if d >= 4096 else 64, seed=d)
    pr = rows_s % P
    phi_s = phi.t[rows_s].cpu().double()
    phi_s[:, 0] = 0.0                                # circle 0 is never drawn (its slot is left unwritten)
    assert not bool(torch.isnan(phi_s).any())
    th = (loc[pr].double() + phi_s).requires_grad_()
    zr = vm_z_from_theta(th)
    assert rel_err(guarded(z)[rows_s].cpu(), zr.detach()) < 1e-5
    (zr * gz[pr].double()).sum().backward()
    dth = th.grad
    dth[:, 0] = 0.0
    got_dl = guarded(dlo)[rows_s].cpu().double()
    assert float((got_dl - dth).abs().max()) <= 1e-5 * max(1.0, float(dth.abs().max()))
    k_el = (kap[pr][:, None].expand(-1, d) if rowk else kap[pr]).double().numpy()
    J = torch.from_numpy(_oracle_dphi(phi_s.numpy(), k_el))
    J[:, 0] = 0.0
    contrib = dth * J
    ref = contrib.sum(-1) if rowk else contrib
    got_dk = guarded(dk)[rows_s].cpu().double()
    assert bool(torch.isfinite(got_dk).all())
    assert bool(((got_dk - ref).abs() <= 2e-5 * ref.abs().clamp_min(1.0)).all()), float((got_dk - ref).abs().max())
    del dlo, dk

    # log_prob with derivatives at a value near the first P samples, periodic in the row
    value = (z.t[:P].cpu().double() + (0.01 / math.sqrt(2 * d)) * torch.randn(P, 2 * d, generator=gen, dtype=torch.float64)).float()
    del z, phi
    rc, lp, dl, dkk, dF = run_log_prob(tile(value, rows), locd, kapd, d, rows, entry="cvb_clifford_vm_log_prob")
    assert rc == 0
    v64, l64 = value.double(), loc.double().requires_grad_()
    k64 = (kap[:, None] if rowk else kap).double().requires_grad_()
    ref = _lp_ref(v64, l64, k64)
    rl, rk = torch.autograd.grad(ref.sum(), (l64, k64))
    assert float((guarded(lp)[:P].cpu().double() - ref.detach()).abs().max()) <= 1e-5 * (float(ref.detach().abs().max()) + 1.0)
    for got, want in ((guarded(dl)[:P], rl), (guarded(dkk)[:P], rk.reshape(-1) if rowk else rk)):
        assert float((got.cpu().double() - want).abs().max()) <= 1e-5 * (float(want.abs().max()) + 1.0)
    for o in (lp, dl, dkk, dF):
        periodic(guarded(o), P, rel=1e-6)   # the row-constant cache, as in the power-spherical log_prob


# ---- 7. back-to-back launches ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("d", FFT)
def test_back_to_back_launches(d):
    """sample (device RNG, draws saved) -> log_prob(z) -> backward from the saved draws, then two injected samples, all
    issued without synchronising: each kernel enters under programmatic dependent launch and each looping launch takes a
    fresh schedule slot.  Bitwise equal to the same chain with a device synchronise after every call."""
    P, rows = period(d), n_rows(d)
    loc, kap, tp, g, gz = make_inputs(d, True, P, P, seed=11 * d)
    locd, kapd = dev(loc), dev(kap)
    tpd, gd, gzd = tile(tp, rows), tile(g, rows), tile(gz, rows)

    def chain(sync):
        o = dict(z=Out(rows, 2 * d), tps=Out(rows, d), ent=Out(rows), lp=Out(rows), dlp=Out(rows, d), dkp=Out(rows),
                 dF=Out(rows, d, 2), dl=Out(rows, d), dk=Out(rows), zi=Out(rows, 2 * d), zj=Out(rows, 2 * d))
        torch.cuda.synchronize()
        step = torch.cuda.synchronize if sync else (lambda: None)
        L = P
        rcs = [call("cvb_clifford_ps_rsample", locd.data_ptr(), kapd.data_ptr(), 1, 0, L, None, None, SEED, OFFSET, o["z"].p,
                    o["tps"].p, o["ent"].p, None, None, rows, d)]
        step()
        rcs.append(call("cvb_clifford_ps_log_prob", o["z"].p, locd.data_ptr(), kapd.data_ptr(), 1, 0, L, o["lp"].p,
                        o["dlp"].p, o["dkp"].p, o["dF"].p, rows, d))
        step()
        rcs.append(call("cvb_clifford_ps_rsample_backward", gzd.data_ptr(), locd.data_ptr(), kapd.data_ptr(), 1, 0, L, None,
                        None, o["tps"].p, o["dl"].p, o["dk"].p, rows, d))
        step()
        for k in ("zi", "zj"):
            rcs.append(call("cvb_clifford_ps_rsample", locd.data_ptr(), kapd.data_ptr(), 1, 0, L, tpd.data_ptr(),
                            gd.data_ptr(), 0, 0, o[k].p, None, None, None, None, rows, d))
        assert rcs == [0] * 5
        return {k: guarded(v) for k, v in o.items()}

    a, b = chain(False), chain(True)
    for k in a:
        x, y = (a[k][:, 1:], b[k][:, 1:]) if k == "tps" else (a[k], b[k])    # circle 0 of the saved draws is unwritten
        assert torch.equal(x, y), k
    assert torch.equal(a["zi"], a["zj"])
    assert rel_err(a["zi"][:P].cpu(), ref_rsample(loc, kap, tp, g, gz)[0]) < 1e-5
    periodic(a["zi"], P)
