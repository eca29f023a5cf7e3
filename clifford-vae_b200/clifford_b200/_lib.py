"""ctypes binding of libclifford_b200.so (C ABI in include/clifford_b200.h).

There is no CPU fallback: a missing library, a CPU tensor or a non-B200 device raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CLIFFORD_B200_LIB", os.path.join(_HERE, "libclifford_b200.so"))

_lib = None
_lock = threading.Lock()
_inited_devices: set[int] = set()

_f = C.c_void_p      # device pointers are passed as integers / None
_ll = C.c_longlong
_ull = C.c_ulonglong
_i = C.c_int
_fl = C.c_float
_db = C.c_double

_SIGNATURES = {
    "cvb_version": ([], _i),
    "cvb_last_error_string": ([], C.c_char_p),
    "cvb_init": ([], _i),
    "cvb_launch_count": ([], _ll),
    "cvb_clifford_ps_rsample": ([_f, _f, _ll, _i, _ll, _f, _f, _ull, _ull, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_ps_rsample_bind": ([_f, _f, _ll, _f, _f, _ull, _ull, _f, _ll, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_ps_rsample_log_prob": ([_f, _f, _ll, _f, _f, _ull, _ull, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_ps_rsample_backward": ([_f, _f, _f, _ll, _i, _ll, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_ps_log_prob": ([_f, _f, _f, _ll, _i, _ll, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_spectrum_adjoint": ([_f, _f, _ll, _i, _f], _i),
    "cvb_ps_entropy_kl": ([_f, _ll, _i, _ll, _i, _db, _i, _db, _f, _f, _f, _f], _i),
    "cvb_clifford_vm_rsample": ([_f, _f, _ll, _i, _ll, _ull, _ull, _f, _ll, _i, _f], _i),
    "cvb_clifford_vm_rsample_kl": ([_f, _f, _ll, _i, _ll, _ull, _ull, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_vm_rsample_backward": ([_f, _f, _f, _ll, _i, _ll, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_vm_log_prob": ([_f, _f, _f, _ll, _i, _ll, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_phases_to_vector": ([_f, _fl, _ull, _ull, _f, _ll, _i, _f], _i),
    "cvb_vsa_bind": ([_f, _f, _f, _ll, _ll, _ll, _i, _i, _f], _i),
    "cvb_vsa_depth_chain_cosine": ([_f, _f, _ll, _i, _i, _f], _i),
    "cvb_vsa_invert": ([_f, _f, _ll, _i, _f], _i),
    "cvb_vsa_permute": ([_f, _f, _f, _ll, _i, _i, _f], _i),
    "cvb_vsa_bundle_workspace_bytes": ([_ll, _i], _ll),
    "cvb_vsa_bundle": ([_f, _f, _ll, _i, _fl, _f, _f], _i),
    "cvb_vsa_cosine": ([_f, _f, _f, _ll, _ll, _ll, _i, _f], _i),
    "cvb_vsa_cosine_backward": ([_f, _f, _f, _f, _f, _ll, _ll, _ll, _i, _f], _i),
    "cvb_vsa_normalize": ([_f, _f, _ll, _i, _f], _i),
    "cvb_vsa_normalize_backward": ([_f, _f, _f, _ll, _i, _f], _i),
    "cvb_vsa_hrr_init": ([_f, _ll, _i, _ull, _ull, _f], _i),
    "cvb_vsa_unitary_init": ([_f, _ll, _i, _fl, _ull, _ull, _f], _i),
    "cvb_powerspherical_rsample": ([_f, _f, _ll, _f, _f, _ull, _ull, _f, _f, _ll, _i, _f], _i),
    "cvb_powerspherical_rsample_kl": ([_f, _f, _ll, _f, _f, _ull, _ull, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_powerspherical_rsample_backward": ([_f, _f, _f, _ll, _f, _f, _f, _ull, _ull, _f, _f, _ll, _i, _f], _i),
    "cvb_powerspherical_log_prob": ([_f, _f, _f, _ll, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_ps_log_normalizer": ([_f, _ll, _db, _f, _f, _f], _i),
    "cvb_sphere_uniform_rsample": ([_f, _ull, _ull, _f, _ll, _i, _fl, _f], _i),
    "cvb_vmf_rsample": ([_f, _f, _ll, _f, _f, _i, _f, _ull, _ull, _f, _f, _ll, _i, _f], _i),
    "cvb_vmf_rsample_kl": ([_f, _f, _ll, _f, _f, _i, _f, _ull, _ull, _f, _f, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_vmf_rsample_backward": ([_f, _f, _f, _ll, _f, _f, _ull, _ull, _f, _f, _ll, _i, _f], _i),
    "cvb_vmf_entropy_lognorm": ([_f, _ll, _i, _f, _f, _f, _f, _f], _i),
    "cvb_clifford_ps_rsample_head": ([_f, _f, _ll, _fl, _fl, _f, _f, _ull, _ull, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_ps_rsample_backward_head": ([_f, _f, _f, _ll, _fl, _fl, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_powerspherical_rsample_kl_head": ([_f, _f, _ll, _fl, _fl, _f, _f, _ull, _ull, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_powerspherical_rsample_backward_head": ([_f, _f, _f, _ll, _fl, _fl, _f, _f, _f, _ull, _ull, _f, _f, _ll, _i, _f], _i),
    "cvb_vmf_rsample_kl_head": ([_f, _f, _ll, _fl, _fl, _f, _f, _i, _f, _ull, _ull, _f, _f, _f, _f, _f, _f, _f, _ll, _i, _f], _i),
    "cvb_vmf_rsample_backward_head": ([_f, _f, _f, _ll, _fl, _fl, _f, _f, _ull, _ull, _f, _f, _ll, _i, _f], _i),
    "cvb_clifford_vm_entropy": ([_f, _ll, _i, _ll, _i, _f, _f, _f], _i),
    "cvb_vmf_log_prob": ([_f, _f, _f, _f, _ll, _f, _f, _ll, _i, _f], _i),
    "cvb_sphere_logprob_backward": ([_f, _f, _f, _ll, _f, _f, _ll, _i, _f], _i),
    "cvb_set_rng_device_counter": ([_f], _i),
    "cvb_set_rng_device_counter_autobump": ([_f], _i),
    "cvb_ps_halfangle_icdf_table": ([_f, _ll, _f, _f, _f], _i),
    "cvb_philox_fill": ([_f, _ll, _ull, _ull, _f], _i),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class CliffordB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise CliffordB200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C clifford-vae_b200/csrc`). There is no CPU / PyTorch fallback for this path.")
        lib = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in _SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError if the .so does not export a declared symbol
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = lib
    return _lib


def ensure_device(device: torch.device) -> None:
    """cvb_init() on `device` (per-device twiddle table); refuses anything but CUDA."""
    if device.type != "cuda":
        raise CliffordB200Error(
            f"clifford_b200 ops run only on a CUDA (sm_100a) device, got a tensor on '{device}'. "
            "There is deliberately no CPU fallback; move the tensors to the GPU.")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx in _inited_devices:
        return
    lib = load()
    with torch.cuda.device(idx):
        rc = lib.cvb_init()
    if rc != 0:
        raise CliffordB200Error(f"cvb_init failed on cuda:{idx}: {lib.cvb_last_error_string().decode()}")
    _inited_devices.add(idx)


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().cvb_last_error_string().decode()
        if rc == 1:
            raise ValueError(f"{what}: {msg}")
        if rc == 2:
            raise NotImplementedError(f"{what}: {msg}")
        raise CliffordB200Error(f"{what}: {msg}")


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(load().cvb_launch_count())


# ---- Philox (seed, offset) bookkeeping ---------------------------------------------------------
_rng_seed = None
_rng_offset = 0


def _rank_mix(seed: int) -> int:
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        seed ^= (torch.distributed.get_rank() * 0x9E3779B97F4A7C15)
    return seed & 0xFFFFFFFFFFFFFFFF


_graph_counters: dict[int, torch.Tensor] = {}      # device index -> int64 launch counter kept for CUDA-graph capture


def _capturing() -> bool:
    try:
        return torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()
    except Exception:
        return False


def next_rng(device=None):
    """(seed, offset) for the next kernel that draws on the device.

    On a CUDA device the pair comes from torch's own CUDA generator for that device: the seed is
    `torch.manual_seed`'s, the offset is reserved from (and advances) the generator's Philox offset, so
    re-seeding restarts the stream and our draws interleave consistently with torch's.  The seed is
    xor-ed with the distributed rank so DDP ranks draw disjoint streams.  Without a device (CPU unit
    tests of the host logic) a process-local call counter stands in for the offset.

    Under CUDA-graph capture the host values are frozen into the graph, so a device-resident launch counter is
    registered with the library in self-bumping mode (cvb_set_rng_device_counter_autobump): every sampling kernel adds 1
    to it when its last CTA retires, which gives every replay of the graph a fresh stream without a counter-increment
    kernel between the sampling launches.  Outside capture the counter is cleared again (host offsets only).
    """
    global _rng_seed, _rng_offset
    if device is not None and torch.device(device).type == "cuda":
        dev = torch.device(device)
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        lib = load()
        if _capturing():
            ctr = _graph_counters.get(idx)
            if ctr is None:
                raise CliffordB200Error(
                    "sampling inside CUDA-graph capture needs clifford_b200._lib.enable_graph_rng(device) to be called "
                    "BEFORE the capture starts (it allocates the device-resident launch counter)")
            with torch.cuda.device(idx):
                lib.cvb_set_rng_device_counter_autobump(ctr.data_ptr())     # the sampling kernel bumps it itself
            _graph_counters[-idx - 1] = ctr                 # mark: registered, clear it at the next eager call
            seed = _rank_mix(torch.initial_seed())
            # a per-capture host constant keeps distinct captured launches apart; torch's generator state cannot be
            # advanced from inside a capture without registering it with the graph
            _rng_offset += 1
            return seed, (1 << 40) + _rng_offset
        if (-idx - 1) in _graph_counters:                   # leaving capture mode: back to host offsets only
            with torch.cuda.device(idx):
                lib.cvb_set_rng_device_counter(None)
            del _graph_counters[-idx - 1]
        gen = torch.cuda.default_generators[idx]
        off = gen.get_offset()
        gen.set_offset(off + 4)
        return _rank_mix(gen.initial_seed()), off // 4
    seed = _rank_mix(torch.initial_seed())
    if seed != _rng_seed:
        _rng_seed, _rng_offset = seed, 0
    off = _rng_offset
    _rng_offset += 1
    return seed, off


def graph_counter_snapshot(device):
    """Under CUDA-graph capture: a (captured) copy of the launch counter as the NEXT sampling launch will read it, for a
    backward that replays that launch's draws (the sphere samplers regenerate their tangent normals from the counter-
    based generator instead of storing them).  None outside capture (host offsets identify the launch there)."""
    if not _capturing():
        return None
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    ctr = _graph_counters.get(idx)
    return None if ctr is None else ctr.clone()


class replay_counter:
    """with replay_counter(device, snapshot): launches inside read `snapshot` as the device launch counter (no bumping);
    the capture-mode registration is restored afterwards.  snapshot None: no-op."""

    def __init__(self, device, snapshot):
        dev = torch.device(device)
        self.idx = dev.index if dev.index is not None else torch.cuda.current_device()
        self.snap = snapshot

    def __enter__(self):
        if self.snap is not None:
            with torch.cuda.device(self.idx):
                load().cvb_set_rng_device_counter(self.snap.data_ptr())
        return self

    def __exit__(self, *exc):
        if self.snap is not None:
            ctr = _graph_counters.get(self.idx)
            with torch.cuda.device(self.idx):
                if _capturing() and ctr is not None:
                    load().cvb_set_rng_device_counter_autobump(ctr.data_ptr())
                else:
                    load().cvb_set_rng_device_counter(None)
        return False


def enable_graph_rng(device) -> torch.Tensor:
    """Allocate (once per device) the device-resident launch counter that lets the samplers be captured in a CUDA
    graph with fresh draws per replay.  Call before `torch.cuda.graph(...)` / `CUDAGraph.capture_begin()`."""
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    ensure_device(torch.device("cuda", idx))
    if idx not in _graph_counters:
        _graph_counters[idx] = torch.zeros(1, dtype=torch.int64, device=torch.device("cuda", idx))
    return _graph_counters[idx]
