"""GPU parity: utils.vsa ops (ctypes -> C ABI) vs golden vectors from the reference and the oracle."""
import math

import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
VSA = ["k5_d64", "k3_d1024", "k4_d37", "k2_d513", "k2_d4096", "k1_d16384", "k3_d144"]


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.mark.parametrize("name", VSA)
def test_vsa_ops_match_reference(golden_vsa, name):
    from utils import vsa
    c = golden_vsa[name]
    a = T(c["a"]).requires_grad_()
    cc = T(c["c"]).requires_grad_()
    b = T(c["b_unitary"])
    ab = vsa.bind(a, cc)
    assert rel_err(ab.detach().cpu(), c["bind_ac"]) < 1e-5
    da, dc = torch.autograd.grad((ab * T(c["grad_out"])).sum(), [a, cc])
    assert rel_err(da.cpu(), c["da"]) < 2e-5
    assert rel_err(dc.cpu(), c["dc"]) < 2e-5
    a_, c_ = a.detach(), cc.detach()
    assert rel_err(vsa.unbind(T(c["bind_ac"]), c_, "inv").cpu(), c["unbind_inv"]) < 1e-5
    assert rel_err(vsa.unbind(T(c["bind_ac"]), c_, "*").cpu(), c["unbind_inv"]) < 1e-5
    # deconvolution divides by |F_c|^2 which can be tiny for an HRR vector: conditioning-limited
    assert rel_err(vsa.unbind(T(c["bind_ac"]), c_, "†").cpu(), c["unbind_deconv"]) < 2e-3
    assert rel_err(vsa.unbind(T(c["bind_ac"]), c_, "deconv").cpu(), c["unbind_deconv"]) < 2e-3
    assert rel_err(vsa.bind(a_, b).cpu(), c["bind_a_unitary"]) < 1e-5
    rec = vsa.unbind(T(c["bind_a_unitary"]), b, "inv")
    assert rel_err(rec.cpu(), c["unbind_unitary"]) < 1e-5
    assert rel_err(rec.cpu(), c["a"]) < 1e-4                       # unitary unbind recovers a
    assert rel_err(vsa.unbind(vsa.bind(a_, b), b, "†").cpu(), c["a"]) < 1e-4
    assert rel_err(vsa.invert(a_).cpu(), c["invert_a"]) == 0
    assert rel_err(vsa.bundle(a_, True).cpu(), c["bundle_norm"]) < 1e-5
    assert rel_err(vsa.bundle(a_, False).cpu(), c["bundle_raw"]) < 1e-5
    assert rel_err(vsa.normalize_vectors(a_).cpu(), c["normalize_a"]) < 1e-6
    assert rel_err(vsa.similarity(a_, c_).cpu(), c["sim_ac"]) < 1e-4
    assert np.max(np.abs(vsa.similarity(a_[0], c_).cpu().numpy() - c["sim_bcast"])) < 1e-6
    perm = T(c["perm"])
    assert rel_err(vsa.permute_vector(a_, perm).cpu(), c["permute_a"]) == 0
    assert rel_err(vsa.unpermute_vector(a_, perm).cpu(), c["unpermute_a"]) == 0
    with pytest.raises(ValueError):
        vsa.unbind(a_, c_, "nope")


@pytest.mark.parametrize("d", [32, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 100, 513])
def test_bind_all_sizes_vs_oracle_and_identities(d):
    from utils import vsa
    from oracle import latent_oracle as O
    torch.manual_seed(d)
    k = 37 if d <= 4096 else 5
    a = torch.randn(k, d) / d ** 0.5
    b = torch.randn(k, d) / d ** 0.5
    ag, bg = a.to(DEV), b.to(DEV)
    out = vsa.bind(ag, bg)
    assert rel_err(out.cpu(), O.bind(a, b)) < 1e-5
    # commutative, associative, invert(invert) = id, broadcasting (1,d) and (d,)
    assert rel_err(vsa.bind(bg, ag).cpu(), out.cpu()) < 1e-6
    c = torch.randn(k, d, device=DEV) / d ** 0.5
    assert rel_err(vsa.bind(vsa.bind(ag, bg), c).cpu(), vsa.bind(ag, vsa.bind(bg, c)).cpu()) < 2e-5
    assert torch.equal(vsa.invert(vsa.invert(ag)), ag)
    assert rel_err(vsa.bind(ag, bg[:1]).cpu(), O.bind(a, b[:1])) < 1e-5
    assert rel_err(vsa.bind(ag, bg[0]).cpu(), O.bind(a, b[0])) < 1e-5
    assert rel_err(vsa.unbind(ag, bg, "inv").cpu(), O.unbind(a, b, "inv")) < 1e-5
    # unbind == bind with the explicit invert
    assert rel_err(vsa.unbind(ag, bg, "inv").cpu(), vsa.bind(ag, vsa.invert(bg)).cpu()) < 1e-5
    # the quotient modes (2: A / (B + 1e-12), 3: A / conj(B + 1e-12)) and the adjoint mode 4 (-A conj B) against float64,
    # with a well-conditioned b (spectrum magnitudes in [0.5, 2], random phases) so that the quotients hold 1e-5 too
    from clifford_b200 import _lib
    h = d // 2 + 1
    mag = 0.5 * 4.0 ** torch.rand(k, h, dtype=torch.float64)
    Bh = torch.polar(mag, 2 * math.pi * torch.rand(k, h, dtype=torch.float64))
    Bh[:, 0] = mag[:, 0]                               # the bins irfft keeps real
    if d % 2 == 0:
        Bh[:, -1] = mag[:, -1]
    bq = torch.fft.irfft(Bh, n=d).float()
    A, Bf = torch.fft.fft(a.double()), torch.fft.fft(bq.double())
    want = {2: A / (Bf + 1e-12), 3: A / (Bf + 1e-12).conj(), 4: -A * Bf.conj()}
    bqd = bq.to(DEV)
    for mode, ref in want.items():
        out = torch.empty(k, d, device=DEV)
        _lib.check(_lib.load().cvb_vsa_bind(ag.data_ptr(), bqd.data_ptr(), out.data_ptr(), k, k, k, d, mode,
                                            torch.cuda.current_stream().cuda_stream), f"bind mode {mode}")
        assert rel_err(out.cpu(), torch.fft.ifft(ref).real) < 1e-5, mode


@pytest.mark.parametrize("d", [64, 1024, 37])
def test_autograd_of_unbind_and_friends_vs_oracle(d):
    from utils import vsa
    from oracle import latent_oracle as O
    torch.manual_seed(3 * d)
    k = 6
    a = torch.randn(k, d) / d ** 0.5
    b = O.unitary_init_from_uniform(torch.rand(k, (d - 1) // 2), torch.rand(k, (d - 1) // 2), d) \
        + 0.05 * torch.randn(k, d) / d ** 0.5
    g = torch.randn(k, d)
    for method in ("inv", "deconv"):
        ac, bc = a.clone().requires_grad_(), b.clone().requires_grad_()
        ag, bg = a.to(DEV).requires_grad_(), b.to(DEV).requires_grad_()
        ro = O.unbind(ac, bc, method)
        rg = vsa.unbind(ag, bg, method)
        assert rel_err(rg.detach().cpu(), ro.detach()) < 2e-5
        dao, dbo = torch.autograd.grad((ro * g).sum(), [ac, bc])
        dag, dbg = torch.autograd.grad((rg * g.to(DEV)).sum(), [ag, bg])
        assert rel_err(dag.cpu(), dao) < 5e-5, method
        assert rel_err(dbg.cpu(), dbo) < 5e-5, method
    # similarity / normalize / bundle / invert / permute backward
    ac, bc = a.clone().requires_grad_(), b.clone().requires_grad_()
    ag, bg = a.to(DEV).requires_grad_(), b.to(DEV).requires_grad_()
    w = torch.randn(k)
    perm = torch.randperm(d)
    fo = (O.similarity(O.normalize_vectors(ac), O.invert(bc)) * w).sum() + \
        (O.bundle(O.permute_vector(ac, perm)) * g[0]).sum() + (O.similarity(ac[0], bc) * w).sum()
    fg = (vsa.similarity(vsa.normalize_vectors(ag), vsa.invert(bg)) * w.to(DEV)).sum() + \
        (vsa.bundle(vsa.permute_vector(ag, perm.to(DEV))) * g[0].to(DEV)).sum() + \
        (vsa.similarity(ag[0], bg) * w.to(DEV)).sum()
    assert abs(float(fo) - float(fg)) < 1e-4 * max(1.0, abs(float(fo)))
    dao, dbo = torch.autograd.grad(fo, [ac, bc])
    dag, dbg = torch.autograd.grad(fg, [ag, bg])
    assert rel_err(dag.cpu(), dao) < 5e-5
    assert rel_err(dbg.cpu(), dbo) < 5e-5


def test_init_generators():
    from utils import vsa
    torch.manual_seed(11)
    for d in (1024, 513, 64, 144):
        u = vsa.unitary_init(50, d, device=DEV)
        F = torch.fft.fft(u.double(), dim=-1)
        assert float((F.abs() - 1).abs().max()) < 5e-5, d           # unit Fourier magnitude
        assert float(F[:, 0].real.min()) > 0.999                    # DC = 1
        ph = torch.angle(F[:, 1:(d + 1) // 2]).abs() / np.pi
        assert float(ph.min()) >= 1e-3 - 1e-4 and float(ph.max()) <= 1 - 1e-3 + 1e-4
        h = vsa.hrr_init(4096, d, device=DEV)
        assert abs(float(h.mean())) < 3e-3 / d ** 0.5 * 10
        assert abs(float(h.var()) * d - 1) < 0.02
    from scipy.stats import kstest
    h = vsa.hrr_init(64, 1024, device=DEV).flatten().cpu().numpy() * 32.0
    assert kstest(h, "norm").pvalue > 1e-3
    # unitary vectors give exact unbinding
    a = vsa.hrr_init(8, 1024, device=DEV)
    b = vsa.unitary_init(8, 1024, device=DEV)
    assert rel_err(vsa.unbind(vsa.bind(a, b), b).cpu(), a.cpu()) < 1e-4


def test_bundle_large_and_full_size_bind_properties():
    """C4-sized pieces: 2^16 x 1024 bind round trip with unitary keys and a 2^16-vector bundle."""
    from utils import vsa
    torch.manual_seed(5)
    N, d = 1 << 16, 1024
    a = vsa.hrr_init(N, d, device=DEV)
    b = vsa.unitary_init(N, d, device=DEV)
    rec = vsa.unbind(vsa.bind(a, b), b)
    assert float((rec - a).abs().max()) < 1e-4 * float(a.abs().max()) * 10
    s = vsa.bundle(a, normalize=True)
    ref = a.double().sum(0) / N ** 0.5
    assert rel_err(s.cpu(), ref.cpu()) < 1e-5
    cs = vsa.similarity(rec, a)
    assert float((cs - 1).abs().max()) < 1e-5


def test_philox_known_answer():
    """Philox4x32-10 known-answer test (Random123 kat_vectors: counter 0, key 0)."""
    import ctypes
    from clifford_b200 import _lib
    _lib.ensure_device(torch.device("cuda:0"))
    lib = _lib.load()
    out = torch.empty(8, dtype=torch.int32, device=DEV)
    rc = lib.cvb_philox_fill(out.data_ptr(), 2, 0, 0, torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    w = [int(x) & 0xFFFFFFFF for x in out.cpu().tolist()]
    assert w[:4] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


def test_sharded_ops_single_rank_use_kernels():
    """clifford_b200.distributed with the real kernels (world size 1 path)."""
    from clifford_b200 import distributed as D
    from utils import vsa
    torch.manual_seed(2)
    items = vsa.normalize_vectors(vsa.hrr_init(300, 256, device=DEV))
    stack = vsa.hrr_init(40, 256, device=DEV)
    got = D.sharded_bundle(stack, 40)
    assert rel_err(got.cpu(), (stack.double().sum(0) / 40 ** 0.5).cpu()) < 1e-5
    q = items[[5, 77, 299]] + 0.01 * torch.randn(3, 256, device=DEV)
    best, idx = D.sharded_cleanup(q, items, 0)
    assert idx.tolist() == [5, 77, 299] and float(best.min()) > 0.9


def test_empty_and_ragged_batches():
    """Edge cases: zero rows, one row, row counts that are not multiples of the CTA group size."""
    from utils import vsa
    from dists.clifford import CliffordPowerSphericalDistribution
    from oracle import latent_oracle as O
    e = torch.empty(0, 64, device=DEV)
    assert vsa.bind(e, e).shape == (0, 64)
    assert vsa.similarity(e, e).shape == (0,)
    assert vsa.normalize_vectors(e).shape == (0, 64)
    q = CliffordPowerSphericalDistribution(torch.empty(0, 32, device=DEV), torch.empty(0, 1, device=DEV))
    assert q.rsample().shape == (0, 64)
    assert q.entropy().shape == (0,)
    torch.manual_seed(1)
    for rows in (1, 3, 5, 129, 1031):
        for d in (64, 256, 1024):
            a, b = torch.randn(rows, d), torch.randn(rows, d)
            assert rel_err(vsa.bind(a.to(DEV), b.to(DEV)).cpu(), O.bind(a, b)) < 1e-5, (rows, d)


def test_c4_full_size_2pow20_vectors():
    """BASELINE config 4 at full size for d = 1024: 2^20 vector pairs (4 GiB per operand) through bind ->
    unbind with unitary keys; size-independent checks: exact recovery (cosine ~ 1), norm preservation,
    linearity of bind in its first argument, and commutativity on a strided subset."""
    from utils import vsa
    torch.manual_seed(8)
    N, d = 1 << 20, 1024
    a = vsa.hrr_init(N, d, device=DEV)
    b = vsa.unitary_init(N, d, device=DEV)
    ab = vsa.bind(a, b)
    # unitary binding preserves the norm (Parseval with |F_b| = 1)
    assert float((ab.norm(dim=-1) / a.norm(dim=-1) - 1).abs().max()) < 1e-4
    rec = vsa.unbind(ab, b)
    cs = vsa.similarity(rec, a)
    assert cs.shape == (N,) and float((cs - 1).abs().max()) < 1e-5
    del rec
    sub = slice(0, N, 4099)
    a2 = vsa.hrr_init(a[sub].shape[0], d, device=DEV)
    lin = vsa.bind(a[sub] + 2.0 * a2, b[sub])
    assert rel_err(lin.cpu(), (ab[sub] + 2.0 * vsa.bind(a2, b[sub])).cpu()) < 2e-5
    assert rel_err(vsa.bind(b[sub], a[sub]).cpu(), ab[sub].cpu()) < 1e-6
    s = vsa.bundle(ab, normalize=True)
    assert s.shape == (d,) and torch.isfinite(s).all()
    assert rel_err(s.cpu(), (ab.double().sum(0) / N ** 0.5).cpu()) < 1e-5


def test_indexing_beyond_2_31_elements():
    """Row offsets are 64-bit: tensors with more than 2^31 elements (C4 sizes: 2^20 vectors at d up to 16384 per GPU)
    round-trip in their LAST rows too.  ~26 GB of device memory."""
    from utils import vsa
    from dists.clifford import CliffordPowerSphericalDistribution
    if torch.cuda.get_device_properties(0).total_memory < 60 * 2 ** 30:
        pytest.skip("needs ~26 GB of device memory")
    torch.manual_seed(8)
    N, d = (1 << 18) + 3, 8192                       # 2.15e9 elements per operand
    a = vsa.hrr_init(N, d, device=DEV)
    key = vsa.unitary_init(1, d, device=DEV)
    assert a.numel() > 2 ** 31 and float(a[-1].abs().max()) > 0 and float(a[N // 2].abs().max()) > 0
    bound = vsa.bind(a, key)
    rec = vsa.unbind(bound, key)
    for sl in (slice(0, 4), slice(N // 2, N // 2 + 4), slice(N - 4, N)):
        assert float((rec[sl] - a[sl]).abs().max()) < 1e-3 * float(a[sl].abs().max())
    cs = vsa.similarity(rec, a)
    assert cs.shape == (N,) and float((cs - 1).abs().max()) < 1e-4
    del bound, rec, cs, a
    torch.cuda.empty_cache()
    B, dl = (1 << 19) + 1, 2048                      # z: 2.15e9 elements
    loc = torch.randn(B, dl, device=DEV)
    kap = torch.rand(B, 1, device=DEV) * 5 + 0.2
    q = CliffordPowerSphericalDistribution(loc, kap, validate_args=False)
    z = q.rsample()
    assert z.numel() > 2 ** 31
    for sl in (slice(0, 8), slice(B - 8, B)):
        F = torch.fft.rfft(z[sl].double(), dim=-1)
        assert float((F.abs() - 1).abs().max()) < 5e-5 and float((z[sl].norm(dim=-1) - 1).abs().max()) < 1e-5
    kl = torch.distributions.kl.kl_divergence(q, __import__("dists.clifford", fromlist=["x"]).CliffordTorusUniform(dl, device=DEV))
    assert kl.shape == (B,) and torch.isfinite(kl).all() and float(kl.min()) > -1e-3


def test_kernels_are_cuda_graph_capturable():
    """The entry points neither allocate nor synchronise, so a chain of them records into a CUDA graph and replays
    with new input contents (INTEGRATION.md: only the device-RNG samplers bake their (seed, offset) into the graph)."""
    from utils import vsa
    from dists.clifford import CliffordPowerSphericalDistribution
    torch.manual_seed(12)
    N, d = 64, 1024
    a = vsa.hrr_init(N, d, device=DEV)
    key = vsa.unitary_init(N, d, device=DEV)
    loc = torch.randn(N, d // 2, device=DEV)
    kap = torch.rand(N, 1, device=DEV) * 4 + 0.3
    q = CliffordPowerSphericalDistribution(loc, kap, validate_args=False)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.no_grad():
        for _ in range(2):                                # warm-up outside capture (lazy init, occupancy cache)
            rec = vsa.unbind(vsa.bind(a, key), key)
            cs = vsa.similarity(rec, a)
            lp = q.log_prob(rec)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(g):
        rec = vsa.unbind(vsa.bind(a, key), key)
        cs = vsa.similarity(rec, a)
        lp = q.log_prob(rec)
    a.copy_(vsa.hrr_init(N, d, device=DEV))               # new contents, same buffers
    g.replay()
    torch.cuda.synchronize()
    assert float((rec - a).abs().max()) < 1e-3 * float(a.abs().max())
    assert float((cs - 1).abs().max()) < 1e-4
    with torch.no_grad():
        assert rel_err(lp.cpu(), q.log_prob(rec.clone()).cpu()) < 1e-6


@pytest.mark.parametrize("d", [4096, 16384])
def test_full_size_c4_streamed_2p20_vectors_vs_fp64_fft(d):
    """BASELINE config 4 at its stated size: 2^20 vector pairs per GPU at d = 4096 and 16384, streamed in chunks
    (d = 16384 would need 192 GiB resident).  Every chunk is compared VALUE BY VALUE with an fp64 evaluation of the
    reference's formula Re ifft(fft a * fft b) (utils/vsa.py:43-46) by cuFFT on the same device, plus the unbind round
    trip on the first chunk."""
    from utils import vsa
    total, chunk, sub = 1 << 20, 1 << 15, 1 << 12
    if d == 4096:
        chunk, sub = 1 << 17, 1 << 14
    gen = torch.Generator(device=DEV)
    worst = 0.0
    for c in range(total // chunk):
        gen.manual_seed(1000 + c)
        a = torch.randn(chunk, d, device=DEV, generator=gen) / d ** 0.5
        b = torch.randn(chunk, d, device=DEV, generator=gen) / d ** 0.5
        out = vsa.bind(a, b)
        for s in range(0, chunk, sub):
            ref = torch.fft.irfft(torch.fft.rfft(a[s:s + sub].double()) * torch.fft.rfft(b[s:s + sub].double()), n=d)
            err = float((out[s:s + sub].double() - ref).abs().max() / ref.abs().max())
            worst = max(worst, err)
            del ref
        if c == 0:
            u = vsa.normalize_vectors(vsa.unitary_init(sub, d, device=DEV))
            rec = vsa.unbind(vsa.bind(a[:sub], u), u)
            assert float((rec - a[:sub]).abs().max() / a[:sub].abs().max()) < 2e-5
        del a, b, out
    assert worst < 1e-5, worst


def test_direct_dft_shared_memory_optin_grows():
    """The direct-DFT kernels size their shared memory at run time: a short length first (< 48 KB, no opt-in) and a long
    one afterwards (> 48 KB) must both launch (the opt-in is tracked per kernel and raised on demand), and so must the
    short one again."""
    from utils import vsa
    torch.manual_seed(3)
    for d in (21, 3000, 21, 6000, 3000):
        a = torch.randn(3, d, device=DEV)
        b = torch.randn(3, d, device=DEV)
        ab = vsa.bind(a, b)
        got = vsa.unbind(ab, b, method="deconv")
        ref = torch.fft.ifft(torch.fft.fft(ab.double()) / (torch.fft.fft(b.double()) + 1e-12)).real
        assert rel_err(got.cpu(), ref.cpu()) < 5e-3, d
