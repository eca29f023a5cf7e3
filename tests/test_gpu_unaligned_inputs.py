"""GPU: the plain-load input paths of the FFT-engine kernels.  Input rows that are 16-byte aligned are staged into shared
memory through TMA (cp.async.bulk); rows that are not are read with plain loads.  Each call here runs on inputs that
start 4 bytes (bind operands, which need 8-byte alignment: 8 bytes) past a 16-byte boundary and is compared with the
same call on aligned copies: bitwise where both calls run the same kernel instantiation, to the op's usual tolerance
where the aligned call runs a specialised one (the lean sampler, the training-path backward, the staged bind)."""
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda"
DIMS = [16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]
ROWS = 4099            # enough rows for the CTAs to loop: dynamic schedule and next-row prefetch


@pytest.fixture(scope="module")
def call():
    from clifford_b200 import _lib
    _lib.ensure_device(torch.device(DEV))
    raw = _lib.load()
    # the device draws keyed by (seed, offset) alone: no launch counter left registered by an earlier graph capture
    _lib.check(raw.cvb_set_rng_device_counter(None), "cvb_set_rng_device_counter")

    def run(name, *args):
        _lib.check(getattr(raw, name)(*args, torch.cuda.current_stream().cuda_stream), name)
    return run


def ptr(t):
    return None if t is None else t.data_ptr()


def shifted(x, offset_bytes):
    """A copy of x that starts offset_bytes past a 16-byte boundary, between NaN guards: a load that strayed outside
    the rows would show in the result."""
    off = offset_bytes // 4
    buf = torch.full((x.numel() + 8,), float("nan"), device=DEV)
    v = buf[off:off + x.numel()].view(x.shape)
    v.copy_(x)
    assert v.data_ptr() % 16 == offset_bytes
    return v


def inputs(d, rows=ROWS):
    g = torch.Generator(device=DEV).manual_seed(1000 + d)
    loc = torch.randn(rows, d, device=DEV, generator=g) * 2
    kap = torch.rand(rows, device=DEV, generator=g) * 9.9 + 0.03
    tprime = torch.rand(rows, d, device=DEV, generator=g) * 0.98 + 0.01
    gnoise = torch.randn(rows, d, device=DEV, generator=g)
    return loc, kap, tprime, gnoise


def rsample(call, loc, kap, tprime=None, gnoise=None, save=False):
    rows, d = loc.shape
    z = torch.zeros(rows, 2 * d, device=DEV)
    kl = torch.zeros(rows, device=DEV)
    tps = torch.zeros(rows, d, device=DEV) if save else None
    call("cvb_clifford_ps_rsample", loc.data_ptr(), kap.data_ptr(), 1, 0, rows, ptr(tprime), ptr(gnoise), 7, 3,
         z.data_ptr(), ptr(tps), None, kl.data_ptr(), None, rows, d)
    return z, kl, tps


# outputs start zeroed: slots a kernel leaves unwritten (circle 0 of the saved draws) compare equal
def assert_equal(got, ref):
    for a, b in zip(got, ref):
        if b is not None:
            assert torch.equal(a, b)


@pytest.mark.parametrize("d", DIMS)
def test_rsample_injected_draws(call, d):
    loc, kap, tp, g = inputs(d)
    ref = rsample(call, loc, kap, tp, g)
    assert_equal(rsample(call, shifted(loc, 4), kap, shifted(tp, 4), shifted(g, 4)), ref)


@pytest.mark.parametrize("d", DIMS)
def test_rsample_device_rng(call, d):
    loc, kap, _, _ = inputs(d)
    # with the draws saved for the backward, both calls run the full sampler
    ref = rsample(call, loc, kap, save=True)
    assert_equal(rsample(call, shifted(loc, 4), kap, save=True), ref)
    # plain sampling: aligned rows take the lean sampler, the others the full one
    z_lean, kl_lean, _ = rsample(call, loc, kap)
    z, kl, _ = rsample(call, shifted(loc, 4), kap)
    assert rel_err(z.cpu(), z_lean.cpu()) < 1e-5
    assert rel_err(kl.cpu(), kl_lean.cpu()) < 1e-5


@pytest.mark.parametrize("d", DIMS)
def test_rsample_backward(call, d):
    loc, kap, tp, g = inputs(d)
    _, _, saved = rsample(call, loc, kap, save=True)
    gz = torch.randn(ROWS, 2 * d, device=DEV, generator=torch.Generator(device=DEV).manual_seed(d))

    def backward(loc, tprime=None, gnoise=None, tps=None):
        dloc = torch.zeros(ROWS, d, device=DEV)
        dkap = torch.zeros(ROWS, device=DEV)
        call("cvb_clifford_ps_rsample_backward", gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, ROWS, ptr(tprime),
             ptr(gnoise), ptr(tps), dloc.data_ptr(), dkap.data_ptr(), ROWS, d)
        return dloc, dkap

    # injected draws: one kernel serves both calls
    assert_equal(backward(shifted(loc, 4), shifted(tp, 4), shifted(g, 4)), backward(loc, tp, g))
    # saved draws: aligned rows take the training-path kernel, the others the general one
    dloc, dkap = backward(shifted(loc, 4), tps=shifted(saved, 4))
    dloc_ref, dkap_ref = backward(loc, tps=saved)
    assert rel_err(dloc.cpu(), dloc_ref.cpu()) < 2e-5
    assert rel_err(dkap.cpu(), dkap_ref.cpu()) < 3e-4


@pytest.mark.parametrize("injected", [False, True])
@pytest.mark.parametrize("d", DIMS)
def test_rsample_bind(call, d, injected):
    loc, kap, tp, g = inputs(d)
    if not injected:
        tp = g = None
    b = torch.randn(ROWS, 2 * d, device=DEV) / (2 * d) ** 0.5

    def run(loc, tp, g, b):
        z = torch.zeros(ROWS, 2 * d, device=DEV)
        bound = torch.zeros(ROWS, 2 * d, device=DEV)
        kl = torch.zeros(ROWS, device=DEV)
        call("cvb_clifford_ps_rsample_bind", loc.data_ptr(), kap.data_ptr(), ROWS, ptr(tp), ptr(g), 7, 3, b.data_ptr(),
             ROWS, z.data_ptr(), bound.data_ptr(), None, kl.data_ptr(), None, ROWS, d)
        return z, bound, kl

    sh = (lambda t: None if t is None else shifted(t, 4))
    assert_equal(run(shifted(loc, 4), sh(tp), sh(g), shifted(b, 8)), run(loc, tp, g, b))


@pytest.mark.parametrize("mode,tol", [(0, 1e-5), (1, 1e-5), (2, 2e-3), (3, 2e-3), (4, 1e-5)])
def test_vsa_bind_d8192(call, mode, tol):
    """aligned operands take the TMA-staged kernel at this length, the shifted ones the plain-load kernel"""
    rows, d = 1000, 8192
    gen = torch.Generator(device=DEV).manual_seed(mode)
    a = torch.randn(rows, d, device=DEV, generator=gen) / d ** 0.5
    b = torch.randn(rows, d, device=DEV, generator=gen) / d ** 0.5

    def run(a, b):
        out = torch.zeros(rows, d, device=DEV)
        call("cvb_vsa_bind", a.data_ptr(), b.data_ptr(), out.data_ptr(), rows, rows, rows, d, mode)
        return out

    assert rel_err(run(shifted(a, 8), shifted(b, 8)).cpu(), run(a, b).cpu()) < tol
