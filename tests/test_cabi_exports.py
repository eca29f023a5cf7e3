"""CPU-side checks of the drop-in boundary: the shared library loads and exports every symbol that
include/clifford_b200.h declares (no compute without a GPU), the ctypes table matches the header,
and the product path never computes on the host: the distributions refuse CPU tensors, and the VSA ops stage CPU
operands to the GPU when one exists and refuse them when none does."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "clifford_b200.h")


def _declared():
    src = open(HEADER).read()
    return re.findall(r"CVB_API\s+[\w\s\*]+?\b(cvb_\w+)\s*\(", src)


def test_library_exports_every_declared_symbol():
    from clifford_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 28
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
    assert set(names) == set(_lib.EXPORTED_SYMBOLS)
    assert lib.cvb_version() >= 100


def test_ctypes_arity_matches_header():
    from clifford_b200 import _lib
    src = open(HEADER).read()
    for name, (argtypes, _) in _lib._SIGNATURES.items():
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", src, re.S)
        assert m, name
        args = m.group(1).strip()
        n = 0 if args in ("void", "") else args.count(",") + 1
        assert n == len(argtypes), (name, n, len(argtypes))


def test_no_cpu_fallback():
    from clifford_b200 import _lib
    from clifford_b200._lib import CliffordB200Error
    from utils import vsa
    from dists.clifford import CliffordPowerSphericalDistribution, PowerSpherical
    a, b = torch.randn(2, 64), torch.randn(2, 64)
    if torch.cuda.is_available():
        # the VSA ops stage CPU operands to the GPU (tests/test_gpu_boundary.py): the library's kernel computes them
        n0 = _lib.launch_count()
        assert vsa.bind(a, b).device.type == "cpu" and _lib.launch_count() > n0
    else:
        with pytest.raises(CliffordB200Error):
            vsa.bind(a, b)
    with pytest.raises(CliffordB200Error):
        CliffordPowerSphericalDistribution(torch.zeros(2, 16), torch.ones(2, 1)).rsample()
    with pytest.raises(CliffordB200Error):
        PowerSpherical(torch.nn.functional.normalize(torch.randn(2, 8), dim=-1), torch.ones(2)).entropy()
    with pytest.raises(ValueError):
        vsa.unbind(torch.randn(2, 64), torch.randn(2, 64), "nope")


def test_product_path_does_not_import_oracle():
    pkg = os.path.join(ROOT, "clifford-vae_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, os.path.join(dirpath, f)


def test_distribution_metadata_matches_reference_contract():
    from dists.clifford import (CliffordPowerSphericalDistribution, CliffordTorusDistribution, CliffordTorusUniform,
                                PowerSpherical, HypersphericalUniform)
    q = CliffordPowerSphericalDistribution(torch.zeros(3, 8), torch.ones(3, 1))
    assert isinstance(q, CliffordTorusDistribution)
    assert q.batch_shape == (3,) and q.event_shape == (16,) and q.orig_dim == 8 and q.has_rsample
    assert q.concentration.shape == (3, 8) and q.loc.shape == (3, 8)
    p = CliffordTorusUniform(8)
    assert p.event_shape == (16,) and abs(p.entropy() - 7 * 1.8378770664093453) < 1e-12
    kl = torch.distributions.kl._dispatch_kl(type(q), type(p))
    assert kl.__name__ == "_kl_ps_uniform"
    ps = PowerSpherical(torch.nn.functional.normalize(torch.randn(4, 5), dim=-1), torch.ones(4))
    assert ps.batch_shape == (4,) and ps.event_shape == (5,) and ps.dim == 5
    hu = HypersphericalUniform(5)
    assert hu.event_shape == (5,)
    assert torch.distributions.kl._dispatch_kl(type(ps), type(hu)).__name__ == "_kl_powerspherical_uniform"
    with pytest.raises(ValueError):
        CliffordPowerSphericalDistribution(torch.zeros(3, 8), -torch.ones(3, 1))
    from hyperspherical_vae.distributions import VonMisesFisher
    from hyperspherical_vae.distributions.hyperspherical_uniform import HypersphericalUniform as VU
    v = VonMisesFisher(torch.nn.functional.normalize(torch.randn(4, 5), dim=-1), torch.ones(4, 1))
    assert v.batch_shape == (4, 5)
    assert torch.distributions.kl._dispatch_kl(type(v), VU).__name__ == "_kl_vmf_uniform"


def test_only_test_infrastructure_imports_the_oracle():
    """oracle/ may be imported by tests/, __graft_entry__.smoke() and bench.py's CPU legs only."""
    allowed = {os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")}
    for top in ("clifford-vae_b200", "examples", "tools"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith(".py"):
                    path = os.path.join(dirpath, f)
                    txt = open(path).read()
                    assert "from oracle" not in txt and "import oracle" not in txt, path
    for path in allowed:
        assert "oracle" in open(path).read()
