"""torch.autograd.Function wrappers over the C ABI (include/clifford_b200.h).

Everything here is plumbing: shape flattening, output allocation with torch (device memory and
streams are torch's), saving tensors for backward.  The arithmetic lives in the CUDA kernels.
"""
from __future__ import annotations

import math

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr

BIND_MUL, BIND_MUL_CONJ, BIND_DIV, BIND_DIV_CONJ, BIND_NEG_MUL_CONJ = range(5)


def _launch(name, dev, *args, skip=False):
    """Call a C-ABI launcher on device `dev` (a torch.device of one of the call's own tensors) and on that
    device's current stream.  Nothing is remembered between calls: forward and backward (which autograd may run on
    another thread, after any number of unrelated ops) each pass their own device and emptiness.
    skip=True (a launch over zero rows / zero-length vectors) returns without launching: the outputs are
    already-empty tensors, like the reference."""
    if skip:
        return
    lib = _lib.load()
    dev = torch.device(dev)
    _lib.ensure_device(dev)
    if dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):
            rc = getattr(lib, name)(*args, torch.cuda.current_stream().cuda_stream)
    else:
        rc = getattr(lib, name)(*args, stream_ptr())
    check(rc, name)


def _any_empty(*tensors) -> bool:
    return any(t is not None and t.numel() == 0 for t in tensors)


def _f32c(t: torch.Tensor) -> torch.Tensor:
    """contiguous fp32 view/copy of t (the kernels compute in fp32)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _prep(*tensors):
    """Check that all tensors live on one CUDA device (initialising the library there).  Returns (lib, device)."""
    dev = tensors[0].device
    _lib.ensure_device(dev)
    for t in tensors[1:]:
        if t is not None and t.device != dev:
            raise _lib.CliffordB200Error(f"tensors on different devices: {dev} vs {t.device}")
    return _lib.load(), dev


def _kappa_layout(kappa: torch.Tensor, d: int):
    """kappa is (B, 1) [row scalar] or (B, d). Returns (tensor, row_stride, el_stride)."""
    if kappa.shape[-1] == 1:
        k = _f32c(kappa.reshape(-1))
        return k, 1, 0
    k = _f32c(kappa.reshape(-1, d))
    return k, d, 1


class RowScalarOfKappa(torch.autograd.Function):
    """A per-row scalar (entropy, log-normaliser) that a sampler launch already produced, re-attached to the graph as a
    function of the concentration: forward hands back the precomputed value, backward multiplies by the derivative the
    same launch produced.  Its own autograd node (own saved tensors), so the sample and the entropy / KL can be
    differentiated in separate backward passes, like the reference's independent graphs."""

    @staticmethod
    def forward(ctx, kappa, box):
        value, dvalue = box              # plain tensors made inside the sampler's forward (not inputs of this node)
        ctx.save_for_backward(dvalue)
        ctx.kshape = tuple(kappa.shape)
        return value

    @staticmethod
    def backward(ctx, grad):
        (dvalue,) = ctx.saved_tensors
        return (grad.reshape(-1) * dvalue.reshape(-1)).reshape(ctx.kshape), None


def row_scalar(kappa, value, dvalue):
    """value as a differentiable function of kappa when that is wanted, else the bare value."""
    if torch.is_grad_enabled() and torch.is_tensor(kappa) and kappa.requires_grad:
        return RowScalarOfKappa.apply(kappa, (value, dvalue))
    return value


# =================================================================================================
# Clifford torus
# =================================================================================================
class CliffordPSRsample(torch.autograd.Function):
    """z, entropy = f(loc (B,d), kappa (B,1)|(B,d)); rows = n_samples * B.

    draws: None (device Philox) or (tprime, g) each (n_samples*B, d) -- parity mode.
    Returns (z (rows, 2d), entropy (B,), d entropy / d kappa (B,)); the last two are plain values (empty when kappa is per
    element or n_samples > 1) that the distribution re-attaches to kappa with row_scalar().

    head = (floor, kmax): `kappa` is the RAW (B, 1) output of the concentration layer and the kernels evaluate
    kappa = min(softplus(raw) + floor, kmax) themselves (mnist/mlp_vae.py:69-71, cnn/models.py:96,99); every
    kappa-gradient returned is then the gradient with respect to that raw tensor.
    """

    @staticmethod
    def forward(ctx, loc, kappa, n_samples, draws, want_entropy, head=None):
        lib, dev = _prep(loc, kappa)
        B, d = loc.shape
        rows = B * n_samples
        loc_c = _f32c(loc)
        kap_c, krs, kes = _kappa_layout(kappa, d)
        if head is not None and kes != 0:
            raise NotImplementedError("the folded concentration head needs one raw value per row, shape (B, 1)")
        z = torch.empty(rows, 2 * d, device=dev, dtype=torch.float32)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        fused_ent = bool(want_entropy) and kes == 0 and n_samples == 1
        ent = torch.empty(B, device=dev, dtype=torch.float32) if fused_ent else None
        dent = torch.empty(B, device=dev, dtype=torch.float32) if fused_ent else None
        if draws is None:
            tp = g = None
            tp_signed = torch.empty(rows, d, device=dev, dtype=torch.float32) if need_grad else None
            seed, off = _lib.next_rng(dev)
        else:
            tp, g = (_f32c(t.reshape(rows, d)) for t in draws)
            tp_signed = None
            seed, off = 0, 0
        if head is None:
            _launch("cvb_clifford_ps_rsample", dev, ptr(loc_c), ptr(kap_c), krs, kes, B, ptr(tp), ptr(g), seed, off, ptr(z),
                    ptr(tp_signed), ptr(ent), None, ptr(dent), rows, d, skip=rows == 0 or d == 0)
        else:
            _launch("cvb_clifford_ps_rsample_head", dev, ptr(loc_c), ptr(kap_c), B, float(head[0]), float(head[1]), ptr(tp),
                    ptr(g), seed, off, ptr(z), ptr(tp_signed), ptr(ent), None, ptr(dent), rows, d, skip=rows == 0 or d == 0)
        ctx.save_for_backward(loc_c, kap_c, tp, g, tp_signed)
        ctx.head = head
        ctx.meta = (B, d, rows, n_samples, krs, kes, tuple(kappa.shape))
        if ent is None:
            ent, dent = z.new_empty(0), z.new_empty(0)
        ctx.mark_non_differentiable(ent, dent)      # re-attached to kappa by row_scalar(): its own autograd node
        return z, ent, dent

    @staticmethod
    def backward(ctx, grad_z, grad_ent, grad_dent):
        loc_c, kap_c, tp, g, tp_signed = ctx.saved_tensors
        B, d, rows, n_samples, krs, kes, kshape = ctx.meta
        dloc = dkap = None
        if grad_z is not None:
            gz = _f32c(grad_z)
            dloc_rows = torch.empty(rows, d, device=gz.device, dtype=torch.float32)
            dk_rows = torch.empty((rows,) if kes == 0 else (rows, d), device=gz.device, dtype=torch.float32)
            if ctx.head is None:
                _launch("cvb_clifford_ps_rsample_backward", gz.device, ptr(gz), ptr(loc_c), ptr(kap_c), krs, kes, B, ptr(tp),
                        ptr(g), ptr(tp_signed), ptr(dloc_rows), ptr(dk_rows), rows, d, skip=rows == 0 or d == 0)
            else:
                _launch("cvb_clifford_ps_rsample_backward_head", gz.device, ptr(gz), ptr(loc_c), ptr(kap_c), B,
                        float(ctx.head[0]), float(ctx.head[1]), ptr(tp), ptr(g), ptr(tp_signed), ptr(dloc_rows),
                        ptr(dk_rows), rows, d, skip=rows == 0 or d == 0)
            if n_samples > 1:
                dloc_rows = dloc_rows.view(n_samples, B, d).sum(0)
                dk_rows = dk_rows.view(n_samples, B, -1).sum(0) if kes else dk_rows.view(n_samples, B).sum(0)
            dloc = dloc_rows
            dkap = dk_rows.reshape(kshape)
        if dloc is None and ctx.needs_input_grad[0]:
            dloc = torch.zeros_like(loc_c)
        return dloc, dkap, None, None, None, None


def clifford_rsample_bind(loc, kappa, other, n_samples=1, draws=None, want_sample=True):
    """Fused forward-only op: z ~ CliffordPS(loc (B,d), kappa (B,1)) for n_samples * B rows, bound = bind(z, other)
    with other (1 | rows, 2d).  Returns (z | None, bound, entropy (B,) | None).  No autograd (evaluation / VSA
    workloads on fresh latents); raises NotImplementedError for shapes the fused kernel does not cover."""
    lib, dev = _prep(loc, kappa, other)
    B, d = loc.shape
    rows = B * n_samples
    if kappa.shape[-1] != 1:
        raise NotImplementedError("rsample_bind needs one concentration per row")
    loc_c, kap_c, oth_c = _f32c(loc), _f32c(kappa.reshape(-1)), _f32c(other.reshape(-1, 2 * d))
    if oth_c.shape[0] not in (1, rows):
        raise ValueError(f"`other` must have 1 or {rows} rows, got {oth_c.shape[0]}")
    z = torch.empty(rows, 2 * d, device=dev, dtype=torch.float32) if want_sample else None
    bound = torch.empty(rows, 2 * d, device=dev, dtype=torch.float32)
    ent = torch.empty(B, device=dev, dtype=torch.float32) if n_samples == 1 else None
    if draws is None:
        tp = g = None
        seed, off = _lib.next_rng(dev)
    else:
        tp, g = (_f32c(t.reshape(rows, d)) for t in draws)
        seed, off = 0, 0
    _launch("cvb_clifford_ps_rsample_bind", dev, ptr(loc_c), ptr(kap_c), B, ptr(tp), ptr(g), seed, off, ptr(oth_c),
            oth_c.shape[0], ptr(z), ptr(bound), ptr(ent), None, None, rows, d, skip=rows == 0 or d == 0)
    return z, bound, ent


def clifford_rsample_log_prob(loc, kappa, n_samples=1, draws=None):
    """Fused forward-only op for the IWAE / evaluation path: z ~ CliffordPS(loc (B,d), kappa (B,1)) for n_samples * B
    rows together with log q(z) of every row (the sampler knows its own phases: no FFT -> angle pass over z).
    Returns (z (rows, 2d), log_prob (rows,), entropy (B,) | None).  Power-of-two d in [16, 8192]."""
    lib, dev = _prep(loc, kappa)
    B, d = loc.shape
    rows = B * n_samples
    if kappa.shape[-1] != 1:
        raise NotImplementedError("rsample_log_prob needs one concentration per row")
    loc_c, kap_c = _f32c(loc), _f32c(kappa.reshape(-1))
    z = torch.empty(rows, 2 * d, device=dev, dtype=torch.float32)
    lp = torch.empty(rows, device=dev, dtype=torch.float32)
    ent = torch.empty(B, device=dev, dtype=torch.float32) if n_samples == 1 else None
    if draws is None:
        tp = g = None
        seed, off = _lib.next_rng(dev)
    else:
        tp, g = (_f32c(t.reshape(rows, d)) for t in draws)
        seed, off = 0, 0
    _launch("cvb_clifford_ps_rsample_log_prob", dev, ptr(loc_c), ptr(kap_c), B, ptr(tp), ptr(g), seed, off, ptr(z),
            ptr(lp), ptr(ent), None, rows, d, skip=rows == 0 or d == 0)
    return z, lp, ent


class PSEntropy(torch.autograd.Function):
    """Power-spherical entropy per row.  torus=True: sum over circles k>=1 of kappa (B,1)|(B,d)
    (dists/clifford.py:318-322).  torus=False: one D-dim PowerSpherical per row, kappa (B,)."""

    @staticmethod
    def forward(ctx, kappa, d, half_dm1, torus):
        lib, dev = _prep(kappa)
        if torus:
            kap_c, krs, kes = _kappa_layout(kappa, d)
            B = kap_c.shape[0]
        else:
            kap_c, krs, kes = _f32c(kappa.reshape(-1)), 1, 0
            B = kap_c.shape[0]
        ent = torch.empty(B, device=dev, dtype=torch.float32)
        dent = torch.empty((B,) if kes == 0 else (B, d), device=dev, dtype=torch.float32)
        _launch("cvb_ps_entropy_kl", dev, ptr(kap_c), krs, kes, B, d, float(half_dm1), 1 if torus else 0, 0.0, ptr(ent),
                None, ptr(dent), skip=B == 0)
        ctx.save_for_backward(dent)
        ctx.kshape = tuple(kappa.shape)
        ctx.kes = kes
        return ent

    @staticmethod
    def backward(ctx, grad):
        (dent,) = ctx.saved_tensors
        g = grad.reshape(-1)
        dk = g * dent if ctx.kes == 0 else g[:, None] * dent
        return dk.reshape(ctx.kshape), None, None, None


def _torus_log_prob_forward(ctx, entry, value, loc, kappa):
    """The launch of a Clifford-torus log_prob (`entry`: the power-spherical or the von Mises family) with the derivative
    outputs autograd will need, saved on ctx for _torus_log_prob_backward."""
    lib, dev = _prep(value, loc, kappa)
    B, d = loc.shape
    rows = value.shape[0]
    val_c, loc_c = _f32c(value), _f32c(loc)
    kap_c, krs, kes = _kappa_layout(kappa, d)
    lp = torch.empty(rows, device=dev, dtype=torch.float32)
    need = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
    dl = torch.empty(rows, d, device=dev, dtype=torch.float32) if need else None
    dk = torch.empty((rows,) if kes == 0 else (rows, d), device=dev, dtype=torch.float32) if need else None
    dF = torch.empty(rows, d, 2, device=dev, dtype=torch.float32) if ctx.needs_input_grad[0] else None
    _launch(entry, dev, ptr(val_c), ptr(loc_c), ptr(kap_c), krs, kes, B, ptr(lp), ptr(dl), ptr(dk), ptr(dF), rows, d,
            skip=rows == 0 or d == 0)
    ctx.save_for_backward(dl, dk, dF)
    ctx.meta = (B, d, rows, kes, tuple(kappa.shape))
    return lp


def _torus_log_prob_backward(ctx, grad):
    dl, dk, dF = ctx.saved_tensors
    B, d, rows, kes, kshape = ctx.meta
    S = rows // B if B else 0
    g = grad.reshape(rows)
    dval = dloc = dkap = None
    if dF is not None:
        h = (g[:, None, None] * dF).contiguous()
        dval = torch.empty(rows, 2 * d, device=g.device, dtype=torch.float32)
        _launch("cvb_clifford_spectrum_adjoint", g.device, ptr(h), ptr(dval), rows, d, skip=rows == 0 or d == 0)
    if dl is not None:
        dloc = (g[:, None] * dl).view(S, B, d).sum(0)
        dkap = ((g * dk).view(S, B).sum(0) if kes == 0 else (g[:, None] * dk).view(S, B, d).sum(0)).reshape(kshape)
    return dval, dloc, dkap


class CliffordPSLogProb(torch.autograd.Function):
    """log_prob (rows,) of value (rows, 2d) under (loc (B,d), kappa (B,1)|(B,d)); rows = S*B.
    Differentiable in loc, kappa and value (the value gradient goes through the adjoint of the truncated real FFT)."""

    @staticmethod
    def forward(ctx, value, loc, kappa):
        return _torus_log_prob_forward(ctx, "cvb_clifford_ps_log_prob", value, loc, kappa)

    @staticmethod
    def backward(ctx, grad):
        return _torus_log_prob_backward(ctx, grad)


class CliffordVMLogProb(torch.autograd.Function):
    """von Mises torus log_prob (rows,) of value (rows, 2d) under (loc (B,d), kappa (B,1)|(B,d)); rows = S*B: the sum over
    circles k >= 1 of kappa cos(angle(rfft(value)_k) - loc_k) - ln(2 pi I0(kappa)).  Differentiable in value, loc, kappa."""

    @staticmethod
    def forward(ctx, value, loc, kappa):
        return _torus_log_prob_forward(ctx, "cvb_clifford_vm_log_prob", value, loc, kappa)

    @staticmethod
    def backward(ctx, grad):
        return _torus_log_prob_backward(ctx, grad)


class CliffordVMRsample(torch.autograd.Function):
    """z, entropy = f(loc (B,d), kappa (B,1)|(B,d)) for the von Mises torus; rows = n_samples * B.  The same draws as
    clifford_vm_rsample for the same generator state; the launch also saves the drawn offsets phi for the backward
    (the implicit reparameterisation gradient of every von Mises draw, cvb_clifford_vm_rsample_backward).
    Returns (z (rows, 2d), entropy (B,), d entropy / d kappa (B,)); the last two are plain values (empty when kappa is per
    element, n_samples > 1 or want_entropy is false) that the distribution re-attaches to kappa with row_scalar()."""

    @staticmethod
    def forward(ctx, loc, kappa, n_samples, want_entropy):
        lib, dev = _prep(loc, kappa)
        B, d = loc.shape
        rows = B * n_samples
        loc_c = _f32c(loc)
        kap_c, krs, kes = _kappa_layout(kappa, d)
        z = torch.empty(rows, 2 * d, device=dev, dtype=torch.float32)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        phi = torch.empty(rows, d, device=dev, dtype=torch.float32) if need_grad else None
        fused_ent = bool(want_entropy) and kes == 0 and n_samples == 1
        ent = torch.empty(B, device=dev, dtype=torch.float32) if fused_ent else None
        dent = torch.empty(B, device=dev, dtype=torch.float32) if fused_ent else None
        seed, off = _lib.next_rng(dev)
        _launch("cvb_clifford_vm_rsample_kl", dev, ptr(loc_c), ptr(kap_c), krs, kes, B, seed, off, ptr(z), ptr(phi),
                ptr(ent), None, ptr(dent), rows, d, skip=rows == 0 or d == 0)
        ctx.save_for_backward(loc_c, kap_c, phi)
        ctx.meta = (B, d, rows, n_samples, krs, kes, tuple(kappa.shape))
        if ent is None:
            ent, dent = z.new_empty(0), z.new_empty(0)
        ctx.mark_non_differentiable(ent, dent)      # re-attached to kappa by row_scalar(): its own autograd node
        return z, ent, dent

    @staticmethod
    def backward(ctx, grad_z, grad_ent, grad_dent):
        loc_c, kap_c, phi = ctx.saved_tensors
        B, d, rows, n_samples, krs, kes, kshape = ctx.meta
        dloc = dkap = None
        if grad_z is not None and phi is not None:
            gz = _f32c(grad_z)
            dloc_rows = torch.empty(rows, d, device=gz.device, dtype=torch.float32)
            dk_rows = torch.empty((rows,) if kes == 0 else (rows, d), device=gz.device, dtype=torch.float32)
            _launch("cvb_clifford_vm_rsample_backward", gz.device, ptr(gz), ptr(loc_c), ptr(kap_c), krs, kes, B, ptr(phi),
                    ptr(dloc_rows), ptr(dk_rows), rows, d, skip=rows == 0 or d == 0)
            if n_samples > 1:
                dloc_rows = dloc_rows.view(n_samples, B, d).sum(0)
                dk_rows = dk_rows.view(n_samples, B, -1).sum(0) if kes else dk_rows.view(n_samples, B).sum(0)
            dloc = dloc_rows
            dkap = dk_rows.reshape(kshape)
        if dloc is None and ctx.needs_input_grad[0]:
            dloc = torch.zeros_like(loc_c)
        return dloc, dkap, None, None


def clifford_vm_rsample(loc, kappa, n_samples=1):
    """z (n_samples * B, 2d) of the von Mises torus distribution (dists/clifford.py:261-275): phases loc + VonMises(0, kappa)
    drawn on the device, then the Hermitian-spectrum inverse FFT.  loc (B, d), kappa (B, 1) | (B, d).  Forward only (the
    sampling path without a graph); CliffordVMRsample draws the same z with a backward."""
    lib, dev = _prep(loc, kappa)
    B, d = loc.shape
    rows = B * n_samples
    loc_c = _f32c(loc.detach())
    kap_c, krs, kes = _kappa_layout(kappa.detach(), d)
    z = torch.empty(rows, 2 * d, device=dev, dtype=torch.float32)
    seed, off = _lib.next_rng(dev)
    _launch("cvb_clifford_vm_rsample", dev, ptr(loc_c), ptr(kap_c), krs, kes, B, seed, off, ptr(z), rows, d,
            skip=rows == 0 or d == 0)
    return z


def clifford_phases_to_vector(phases, scale, rows, d, device):
    """phases (rows, d) * scale -> (rows, 2d); phases None draws U[0,1) on the device."""
    _lib.ensure_device(torch.device(device))
    z = torch.empty(rows, 2 * d, device=device, dtype=torch.float32)
    dev = z.device
    if phases is None:
        seed, off = _lib.next_rng(dev)
        ph = None
    else:
        ph, seed, off = _f32c(phases.reshape(rows, d)), 0, 0
    _launch("cvb_clifford_phases_to_vector", dev, ptr(ph), float(scale), seed, off, ptr(z), rows, d,
            skip=rows == 0 or d == 0)
    return z


# =================================================================================================
# VSA
# =================================================================================================
def _bind_raw(a2, b2, rows, d, mode):
    out = torch.empty(rows, d, device=a2.device, dtype=torch.float32)
    _launch("cvb_vsa_bind", out.device, ptr(a2), ptr(b2), ptr(out), rows, a2.shape[0], b2.shape[0], d, mode,
            skip=_any_empty(a2, b2, out))
    return out


def _flatten_pair(a, b):
    """Broadcast leading dims of a, b (..., d). Returns (a2 (Ra,d), b2 (Rb,d), rows, out_shape) where
    each operand is fully expanded, a single broadcast row (Rx == 1), or broadcast over leading dims only
    (Rx = product of its trailing batch dims) -- the kernel indexes operand rows modulo Rx."""
    d = a.shape[-1]
    if b.shape[-1] != d:
        raise ValueError(f"last dims differ: {a.shape} vs {b.shape}")
    lead = torch.broadcast_shapes(a.shape[:-1], b.shape[:-1])
    rows = int(math.prod(lead)) if len(lead) else 1

    def flat(x):
        if x.shape[:-1] == lead:
            return _f32c(x).reshape(rows, d)
        if x.numel() == d:
            return _f32c(x).reshape(1, d)
        xl = tuple(x.shape[:-1])
        while xl and xl[0] == 1:
            xl = xl[1:]
        if xl and xl == tuple(lead[len(lead) - len(xl):]):
            return _f32c(x).reshape(-1, d)        # broadcast over leading dims only: row r of the result uses r % Rx
        return _f32c(x.expand(*lead, d)).reshape(rows, d)

    return flat(a), flat(b), rows, tuple(lead) + (d,)


def _reduce_to(grad_rows, shape, out_shape):
    """Sum a (rows, d) gradient of the broadcast result back to an operand of `shape`."""
    g = grad_rows.reshape(out_shape)
    return g.sum_to_size(shape) if tuple(shape) != tuple(out_shape) else g


class Bind(torch.autograd.Function):
    """mode MUL: bind (utils/vsa.py:43-46); MUL_CONJ: unbind 'inv' (vsa.py:56-64); DIV: unbind 'deconv'."""

    @staticmethod
    def forward(ctx, a, b, mode):
        _prep(a, b)
        a2, b2, rows, out_shape = _flatten_pair(a, b)
        out = _bind_raw(a2, b2, rows, a.shape[-1], mode)
        ctx.save_for_backward(a2, b2, out if mode == BIND_DIV else None)
        ctx.meta = (mode, rows, out_shape, tuple(a.shape), tuple(b.shape))
        return out.reshape(out_shape)

    @staticmethod
    def backward(ctx, grad):
        a2, b2, out = ctx.saved_tensors
        mode, rows, out_shape, ashape, bshape = ctx.meta
        d = out_shape[-1]
        g = _f32c(grad).reshape(rows, d)
        da = db = None
        if mode == BIND_MUL:          # d/da = bind(g, invert(b)), d/db = bind(g, invert(a))
            if ctx.needs_input_grad[0]:
                da = _bind_raw(g, b2, rows, d, BIND_MUL_CONJ)
            if ctx.needs_input_grad[1]:
                db = _bind_raw(g, a2, rows, d, BIND_MUL_CONJ)
        elif mode == BIND_MUL_CONJ:   # out = irfft(A conj B): d/da = bind(g, b), d/db = irfft(A conj G)
            if ctx.needs_input_grad[0]:
                da = _bind_raw(g, b2, rows, d, BIND_MUL)
            if ctx.needs_input_grad[1]:
                db = _bind_raw(a2, g, rows, d, BIND_MUL_CONJ)
        else:                         # DIV: d/da = irfft(G / conj(B+eps)), d/db = -irfft(dA conj OUT)
            da_rows = _bind_raw(g, b2, rows, d, BIND_DIV_CONJ)
            if ctx.needs_input_grad[0]:
                da = da_rows
            if ctx.needs_input_grad[1]:
                db = _bind_raw(da_rows, out, rows, d, BIND_NEG_MUL_CONJ)
        if da is not None:
            da = _reduce_to(da, ashape, out_shape)
        if db is not None:
            db = _reduce_to(db, bshape, out_shape)
        return da, db, None


def invert(a):
    lib, dev = _prep(a)
    d = a.shape[-1]
    a2 = _f32c(a).reshape(-1, d)
    out = torch.empty_like(a2)
    _launch("cvb_vsa_invert", dev, ptr(a2), ptr(out), a2.shape[0], d, skip=_any_empty(a2))
    return out.reshape(a.shape)


class Invert(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a):
        return invert(a)

    @staticmethod
    def backward(ctx, grad):
        return invert(grad)   # the index reversal is an involutive permutation


def permute(v, perm, inverse):
    lib, dev = _prep(v, perm)
    d = v.shape[-1]
    if perm.numel() != d:
        raise ValueError("permutation length must equal the vector dimension")
    v2 = _f32c(v).reshape(-1, d)
    pm = perm.to(torch.int64).contiguous()
    out = torch.empty_like(v2)
    _launch("cvb_vsa_permute", dev, ptr(v2), ptr(pm), ptr(out), v2.shape[0], d, 1 if inverse else 0, skip=_any_empty(v2))
    return out.reshape(v.shape)


class Permute(torch.autograd.Function):
    @staticmethod
    def forward(ctx, v, perm, inverse):
        ctx.save_for_backward(perm)
        ctx.inverse = inverse
        return permute(v, perm, inverse)

    @staticmethod
    def backward(ctx, grad):
        (perm,) = ctx.saved_tensors
        return permute(grad, perm, not ctx.inverse), None, None


class Bundle(torch.autograd.Function):
    @staticmethod
    def forward(ctx, vectors, scale):
        lib, dev = _prep(vectors)
        k = vectors.shape[0]
        inner = tuple(vectors.shape[1:])
        d = int(math.prod(inner)) if inner else 1
        v2 = _f32c(vectors).reshape(k, d)
        out = torch.empty(d, device=dev, dtype=torch.float32)
        ws = torch.empty(max(int(lib.cvb_vsa_bundle_workspace_bytes(k, d)) // 4, 1), device=dev, dtype=torch.float32)
        if k == 0:
            out.zero_()           # an empty stack sums to zero (torch.sum over an empty dim)
        _launch("cvb_vsa_bundle", dev, ptr(v2), ptr(out), k, d, float(scale), ptr(ws), skip=_any_empty(v2))
        ctx.meta = (tuple(vectors.shape), float(scale))
        return out.reshape(inner)

    @staticmethod
    def backward(ctx, grad):
        shape, scale = ctx.meta
        return (grad * scale).unsqueeze(0).expand(shape), None


class Cosine(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        lib, dev = _prep(a, b)
        a2, b2, rows, out_shape = _flatten_pair(a, b)
        d = out_shape[-1]
        out = torch.empty(rows, device=dev, dtype=torch.float32)
        if d == 0:
            out.zero_()
        _launch("cvb_vsa_cosine", dev, ptr(a2), ptr(b2), ptr(out), rows, a2.shape[0], b2.shape[0], d,
                skip=_any_empty(a2, b2, out))
        ctx.save_for_backward(a2, b2)
        ctx.meta = (rows, out_shape, tuple(a.shape), tuple(b.shape))
        return out.reshape(out_shape[:-1])

    @staticmethod
    def backward(ctx, grad):
        a2, b2 = ctx.saved_tensors
        rows, out_shape, ashape, bshape = ctx.meta
        d = out_shape[-1]
        g = _f32c(grad).reshape(rows)
        da = torch.empty(rows, d, device=g.device, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        db = torch.empty(rows, d, device=g.device, dtype=torch.float32) if ctx.needs_input_grad[1] else None
        _launch("cvb_vsa_cosine_backward", g.device, ptr(a2), ptr(b2), ptr(g), ptr(da), ptr(db), rows, a2.shape[0],
                b2.shape[0], d, skip=_any_empty(a2, b2, g))
        if da is not None:
            da = _reduce_to(da, ashape, out_shape)
        if db is not None:
            db = _reduce_to(db, bshape, out_shape)
        return da, db


class Normalize(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        lib, dev = _prep(x)
        d = x.shape[-1]
        x2 = _f32c(x).reshape(-1, d)
        out = torch.empty_like(x2)
        _launch("cvb_vsa_normalize", dev, ptr(x2), ptr(out), x2.shape[0], d, skip=_any_empty(x2))
        ctx.save_for_backward(x2)
        ctx.shape = tuple(x.shape)
        return out.reshape(x.shape)

    @staticmethod
    def backward(ctx, grad):
        (x2,) = ctx.saved_tensors
        g = _f32c(grad).reshape(x2.shape)
        dx = torch.empty_like(x2)
        _launch("cvb_vsa_normalize_backward", g.device, ptr(x2), ptr(g), ptr(dx), x2.shape[0], x2.shape[1],
                skip=_any_empty(x2))
        return dx.reshape(ctx.shape)


def hrr_init(n, d, device):
    dev = torch.device(device)
    _lib.ensure_device(dev)
    out = torch.empty(n, d, device=dev, dtype=torch.float32)
    dev = out.device
    seed, off = _lib.next_rng(dev)
    _launch("cvb_vsa_hrr_init", dev, ptr(out), n, d, seed, off, skip=out.numel() == 0)
    return out


def unitary_init(n, d, device, eps):
    dev = torch.device(device)
    _lib.ensure_device(dev)
    out = torch.empty(n, d, device=dev, dtype=torch.float32)
    dev = out.device
    seed, off = _lib.next_rng(dev)
    _launch("cvb_vsa_unitary_init", dev, ptr(out), n, d, float(eps), seed, off, skip=out.numel() == 0)
    return out


# =================================================================================================
# D-dimensional PowerSpherical / vMF / uniform sphere
# =================================================================================================
def sphere_uniform_rsample(rows, D, device, norm_eps, gnoise=None):
    dev = torch.device(device)
    _lib.ensure_device(dev)
    z = torch.empty(rows, D, device=dev, dtype=torch.float32)
    dev = z.device
    if gnoise is None:
        seed, off = _lib.next_rng(dev)
        g = None
    else:
        g, seed, off = _f32c(gnoise.reshape(rows, D)), 0, 0
    _launch("cvb_sphere_uniform_rsample", dev, ptr(g), seed, off, ptr(z), rows, D, float(norm_eps), skip=z.numel() == 0)
    return z


class PowerSphericalRsample(torch.autograd.Function):
    """(z (n*B, D), entropy (B,), d entropy / d kappa (B,)) = PowerSpherical(loc (B,D), kappa (B,)).rsample fused with
    .entropy() in ONE launch (the training step evaluates both, mnist/mlp_vae.py:110-129); the two row scalars are plain
    values re-attached to kappa by row_scalar().  draws None or (tprime (rows,), g (rows, D-1))."""

    @staticmethod
    def forward(ctx, loc, kappa, n_samples, draws, head=None):
        lib, dev = _prep(loc, kappa)
        B, D = loc.shape
        rows = B * n_samples
        loc_c, kap_c = _f32c(loc), _f32c(kappa.reshape(-1))
        z = torch.empty(rows, D, device=dev, dtype=torch.float32)
        ent = torch.empty(B, device=dev, dtype=torch.float32)
        dent = torch.empty(B, device=dev, dtype=torch.float32)
        hd = () if head is None else (float(head[0]), float(head[1]))      # head: kappa is the raw layer output
        sfx = "" if head is None else "_head"
        snap = None
        if draws is None:
            tp = g = None
            save = torch.empty(rows, 2, device=dev, dtype=torch.float32)
            seed, off = _lib.next_rng(dev)
            if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
                snap = _lib.graph_counter_snapshot(dev)     # the backward replays this launch's normals
        else:
            tp = _f32c(draws[0].reshape(rows))
            g = _f32c(draws[1].reshape(rows, D - 1))
            save, seed, off = None, 0, 0
        _launch("cvb_powerspherical_rsample_kl" + sfx, dev, ptr(loc_c), ptr(kap_c), B, *hd, ptr(tp), ptr(g), seed, off, ptr(z),
                ptr(save), ptr(ent), None, ptr(dent), rows, D, skip=z.numel() == 0)
        ctx.save_for_backward(loc_c, kap_c, tp, g, save)
        ctx.head = (sfx, hd)
        ctx.snap = snap
        ctx.meta = (B, D, rows, n_samples, seed, off, tuple(kappa.shape))
        ctx.mark_non_differentiable(ent, dent)
        return z, ent, dent

    @staticmethod
    def backward(ctx, grad_z, grad_ent, grad_dent):
        loc_c, kap_c, tp, g, save = ctx.saved_tensors
        B, D, rows, n_samples, seed, off, kshape = ctx.meta
        dloc = dk = None
        if grad_z is not None:
            gz = _f32c(grad_z).reshape(rows, D)
            dloc = torch.empty(rows, D, device=gz.device, dtype=torch.float32)
            dk = torch.empty(rows, device=gz.device, dtype=torch.float32)
            sfx, hd = ctx.head
            with _lib.replay_counter(gz.device, ctx.snap):
                _launch("cvb_powerspherical_rsample_backward" + sfx, gz.device, ptr(gz), ptr(loc_c), ptr(kap_c), B, *hd, ptr(tp),
                        ptr(g), ptr(save), seed, off, ptr(dloc), ptr(dk), rows, D, skip=gz.numel() == 0)
            if n_samples > 1:
                dloc = dloc.view(n_samples, B, D).sum(0)
                dk = dk.view(n_samples, B).sum(0)
        if dloc is None and ctx.needs_input_grad[0]:
            dloc = torch.zeros_like(loc_c)
        return dloc, (None if dk is None else dk.reshape(kshape)), None, None, None


class PowerSphericalLogProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, value, loc, kappa):
        lib, dev = _prep(value, loc, kappa)
        B, D = loc.shape
        rows = value.shape[0]
        val_c, loc_c, kap_c = _f32c(value), _f32c(loc), _f32c(kappa.reshape(-1))
        lp = torch.empty(rows, device=dev, dtype=torch.float32)
        need = any(ctx.needs_input_grad)
        coef = torch.empty(rows, device=dev, dtype=torch.float32) if need else None
        dk = torch.empty(rows, device=dev, dtype=torch.float32) if need else None
        _launch("cvb_powerspherical_log_prob", dev, ptr(val_c), ptr(loc_c), ptr(kap_c), B, ptr(lp), ptr(coef), ptr(dk),
                rows, D, skip=val_c.numel() == 0)
        ctx.save_for_backward(val_c, loc_c, coef, dk)
        ctx.meta = (B, D, rows, tuple(kappa.shape))
        return lp

    @staticmethod
    def backward(ctx, grad):
        val_c, loc_c, coef, dk = ctx.saved_tensors
        B, D, rows, kshape = ctx.meta
        S = rows // B
        g = _f32c(grad).reshape(rows)
        dval, dloc = _logprob_backward(g * coef, val_c, loc_c, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        dkap = (g * dk).view(S, B).sum(0).reshape(kshape) if ctx.needs_input_grad[2] else None
        return dval, dloc, dkap


def _logprob_backward(w, val_c, loc_c, want_dval, want_dloc):
    """d lp / d value = w loc and d lp / d loc = sum over samples of w value for a row log-density lp = f(<loc, value>),
    w (rows) = upstream gradient times f'.  One kernel (the sample-dimension sum included)."""
    rows, D = val_c.shape
    B = loc_c.shape[0]
    dval = torch.empty(rows, D, device=val_c.device, dtype=torch.float32) if want_dval else None
    dloc = torch.empty(B, D, device=val_c.device, dtype=torch.float32) if want_dloc else None
    if want_dval or want_dloc:
        w = _f32c(w)
        _launch("cvb_sphere_logprob_backward", val_c.device, ptr(w), ptr(val_c), ptr(loc_c), B, ptr(dval), ptr(dloc), rows, D,
                skip=val_c.numel() == 0)
    return dval, dloc


class VMFLogProb(torch.autograd.Function):
    """VonMisesFisher.log_prob (von_mises_fisher.py:193-212): lp (rows,) = kappa <loc, value> - log_norm for value
    (rows, D), loc (B, D), kappa (B,), log_norm (B,) (the fused / cached `_log_normalization`, itself a function of kappa
    in the autograd graph); rows = S * B."""

    @staticmethod
    def forward(ctx, value, loc, kappa, log_norm):
        lib, dev = _prep(value, loc, kappa, log_norm)
        B, D = loc.shape
        rows = value.shape[0]
        val_c, loc_c, kap_c, ln_c = _f32c(value), _f32c(loc), _f32c(kappa.reshape(-1)), _f32c(log_norm.reshape(-1))
        lp = torch.empty(rows, device=dev, dtype=torch.float32)
        dot = torch.empty(rows, device=dev, dtype=torch.float32) if ctx.needs_input_grad[2] else None
        _launch("cvb_vmf_log_prob", dev, ptr(val_c), ptr(loc_c), ptr(kap_c), ptr(ln_c), B, ptr(lp), ptr(dot), rows, D,
                skip=val_c.numel() == 0)
        ctx.save_for_backward(val_c, loc_c, kap_c, dot)
        ctx.meta = (B, D, rows, tuple(kappa.shape), tuple(log_norm.shape))
        return lp

    @staticmethod
    def backward(ctx, grad):
        val_c, loc_c, kap_c, dot = ctx.saved_tensors
        B, D, rows, kshape, lshape = ctx.meta
        S = rows // B
        g = _f32c(grad).reshape(rows)
        w = (g.view(S, B) * kap_c).reshape(rows)
        dval, dloc = _logprob_backward(w, val_c, loc_c, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        dkap = (g * dot).view(S, B).sum(0).reshape(kshape) if ctx.needs_input_grad[2] else None
        dln = (-g.view(S, B).sum(0)).reshape(lshape) if ctx.needs_input_grad[3] else None
        return dval, dloc, dkap, dln


class VMTorusEntropy(torch.autograd.Function):
    """CliffordTorusDistribution.entropy (dists/clifford.py:21-31, :277-278) per row of kappa (B,1)|(B,d): the sum over
    circles k >= 1 of the (eps-regularised) von Mises entropy, with its kappa-derivative for the backward."""

    @staticmethod
    def forward(ctx, kappa, d):
        lib, dev = _prep(kappa)
        kap_c, krs, kes = _kappa_layout(kappa, d)
        B = kap_c.shape[0]
        ent = torch.empty(B, device=dev, dtype=torch.float32)
        dent = torch.empty((B,) if kes == 0 else (B, d), device=dev, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        _launch("cvb_clifford_vm_entropy", dev, ptr(kap_c), krs, kes, B, d, ptr(ent), ptr(dent), skip=B == 0)
        ctx.save_for_backward(dent)
        ctx.kshape = tuple(kappa.shape)
        ctx.kes = kes
        return ent

    @staticmethod
    def backward(ctx, grad):
        (dent,) = ctx.saved_tensors
        g = grad.reshape(-1)
        dk = g * dent if ctx.kes == 0 else g[:, None] * dent
        return dk.reshape(ctx.kshape), None


class PSLogNormalizer(torch.autograd.Function):
    @staticmethod
    def forward(ctx, kappa, dim):
        lib, dev = _prep(kappa)
        k = _f32c(kappa.reshape(-1))
        ln = torch.empty_like(k)
        dln = torch.empty_like(k)
        _launch("cvb_ps_log_normalizer", dev, ptr(k), k.numel(), (dim - 1) / 2, ptr(ln), ptr(dln), skip=k.numel() == 0)
        ctx.save_for_backward(dln)
        ctx.kshape = tuple(kappa.shape)
        return ln.reshape(kappa.shape)

    @staticmethod
    def backward(ctx, grad):
        (dln,) = ctx.saved_tensors
        return (grad.reshape(-1) * dln).reshape(ctx.kshape), None


class VMFRsample(torch.autograd.Function):
    """(z (rows, D), entropy, log_norm, d entropy / d kappa, d log_norm / d kappa (B,) each) = VonMisesFisher(loc (B,D),
    kappa (B,1)).rsample fused with the row's entropy and log-normaliser (von_mises_fisher.py:183-212) in ONE launch; the
    row scalars are plain values re-attached to kappa by row_scalar().
    draws: None or (e_rounds (R, rows) f64 | None for D == 3, u_rounds (R, rows) f64, g (rows, D))."""

    @staticmethod
    def forward(ctx, loc, kappa, n_samples, draws, head=None):
        lib, dev = _prep(loc, kappa)
        B, D = loc.shape
        rows = B * n_samples
        loc_c, kap_c = _f32c(loc), _f32c(kappa.reshape(-1))
        hd = () if head is None else (float(head[0]), float(head[1]))      # head: kappa is the raw layer output
        sfx = "" if head is None else "_head"
        z = torch.empty(rows, D, device=dev, dtype=torch.float32)
        save = torch.empty(rows, 2, device=dev, dtype=torch.float32)
        ent, ln, dent, dln = (torch.empty(B, device=dev, dtype=torch.float32) for _ in range(4))
        snap = None
        if draws is None:
            e = u = g = None
            R = 0
            seed, off = _lib.next_rng(dev)
            if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
                snap = _lib.graph_counter_snapshot(dev)     # the backward replays this launch's normals
        else:
            e, u, g = draws
            u = u.to(torch.float64).reshape(-1, rows).contiguous()
            e = None if e is None else e.to(torch.float64).reshape(-1, rows).contiguous()
            R = u.shape[0]
            g = _f32c(g.reshape(rows, D))
            seed, off = 0, 0
        _launch("cvb_vmf_rsample_kl" + sfx, dev, ptr(loc_c), ptr(kap_c), B, *hd, ptr(e), ptr(u), R, ptr(g), seed, off, ptr(z),
                ptr(save), ptr(ent), None, ptr(dent), ptr(ln), ptr(dln), rows, D, skip=z.numel() == 0)
        ctx.save_for_backward(loc_c, kap_c, g, save)
        ctx.head = (sfx, hd)
        ctx.snap = snap
        ctx.meta = (B, D, rows, n_samples, seed, off, tuple(kappa.shape))
        ctx.mark_non_differentiable(ent, ln, dent, dln)
        return z, ent, ln, dent, dln

    @staticmethod
    def backward(ctx, grad_z, *unused):
        loc_c, kap_c, g, save = ctx.saved_tensors
        B, D, rows, n_samples, seed, off, kshape = ctx.meta
        dloc = dk = None
        if grad_z is not None:
            gz = _f32c(grad_z).reshape(rows, D)
            dloc = torch.empty(rows, D, device=gz.device, dtype=torch.float32)
            dk = torch.empty(rows, device=gz.device, dtype=torch.float32)
            sfx, hd = ctx.head
            with _lib.replay_counter(gz.device, ctx.snap):
                _launch("cvb_vmf_rsample_backward" + sfx, gz.device, ptr(gz), ptr(loc_c), ptr(kap_c), B, *hd, ptr(g), ptr(save),
                        seed, off, ptr(dloc), ptr(dk), rows, D, skip=gz.numel() == 0)
            if n_samples > 1:
                dloc = dloc.view(n_samples, B, D).sum(0)
                dk = dk.view(n_samples, B).sum(0)
        if dloc is None and ctx.needs_input_grad[0]:
            dloc = torch.zeros_like(loc_c)
        return dloc, (None if dk is None else dk.reshape(kshape)), None, None, None


class VMFEntropyLogNorm(torch.autograd.Function):
    """(entropy, log_norm) per row of kappa (B,1) for sphere dimension D."""

    @staticmethod
    def forward(ctx, kappa, D):
        lib, dev = _prep(kappa)
        k = _f32c(kappa.reshape(-1))
        ent, ln, dent, dln = (torch.empty_like(k) for _ in range(4))
        _launch("cvb_vmf_entropy_lognorm", dev, ptr(k), k.numel(), D, ptr(ent), ptr(ln), ptr(dent), ptr(dln),
                skip=k.numel() == 0)
        ctx.save_for_backward(dent, dln)
        ctx.kshape = tuple(kappa.shape)
        return ent, ln

    @staticmethod
    def backward(ctx, g_ent, g_ln):
        dent, dln = ctx.saved_tensors
        out = torch.zeros_like(dent)
        if g_ent is not None:
            out = out + g_ent.reshape(-1) * dent
        if g_ln is not None:
            out = out + g_ln.reshape(-1) * dln
        return out.reshape(ctx.kshape), None
