"""torch.distributions-style classes with the reference's names, constructor signatures, attributes
and KL registrations (reference dists/clifford.py), backed by the sm_100a kernels.

These are re-exported as ``dists.clifford`` so the reference's model files
(mnist/mlp_vae.py:11-16, cnn/models.py:8-15) import them unchanged.
"""
from __future__ import annotations

import math
import weakref
from typing import Dict

import torch
from torch.distributions import Distribution, constraints
from torch.distributions.kl import register_kl
from torch.distributions.utils import broadcast_all

from . import ops, testing

_LOG_2PI = math.log(2 * math.pi)


def head_concentration(raw_scale, floor, kmax):
    """The reference models' concentration head as torch ops (mnist/mlp_vae.py:69-71, cnn/models.py:96,99) -- what the
    ``from_head`` constructors fold into the sampling kernels; used only when a head-built distribution is asked for its
    ``concentration`` / ``scale`` attribute or for a method outside the fused training path."""
    return torch.clamp(torch.nn.functional.softplus(raw_scale) + floor, max=kmax)


def _numel(shape) -> int:
    n = 1
    for s in shape:
        n *= int(s)
    return n


class HypersphericalUniform(Distribution):
    """Uniform distribution on S^(dim-1) in R^dim (reference dists/clifford.py:85-121)."""

    arg_constraints: Dict[str, constraints.Constraint] = {}
    has_rsample = True

    def __init__(self, dim, device="cpu", dtype=torch.float32, validate_args=None):
        self.dim = dim
        self.device, self.dtype = device, dtype
        super().__init__(batch_shape=torch.Size(), event_shape=torch.Size([dim]), validate_args=validate_args)

    def rsample(self, sample_shape=torch.Size()):
        shape = tuple(sample_shape) + tuple(self.event_shape)
        rows = _numel(shape[:-1])
        z = ops.sphere_uniform_rsample(rows, self.dim, self.device, 1e-7)
        return z.reshape(shape).to(self.dtype)

    def _log_density(self):
        return math.lgamma(self.dim / 2) - (math.log(2) + (self.dim / 2) * math.log(math.pi))

    def log_prob(self, value):
        if self.dim <= 0:
            return torch.tensor(float("-inf"), device=self.device, dtype=self.dtype)
        return torch.full_like(value[..., 0], self._log_density())

    def entropy(self):
        if self.dim <= 0:
            return torch.tensor(float("inf"), device=self.device, dtype=self.dtype)
        # 0-d like the reference (-log_prob(zeros(1)) indexes the event dim away, dists/clifford.py:118-121)
        return torch.full((), -self._log_density(), device=self.device, dtype=self.dtype)


class PowerSpherical(Distribution):
    """Power spherical distribution on S^(D-1) (reference dists/clifford.py:162-212).

    loc (..., D) unit vectors, scale (...,) concentrations.  rsample / log_prob / entropy run as
    fused row kernels (Beta draw + tangent normal + T-transform + Householder in one pass).
    """

    arg_constraints: Dict[str, constraints.Constraint] = {}
    has_rsample = True

    def __init__(self, loc, scale, validate_args=None):
        self.loc, self.scale = loc, scale
        self.dim = loc.shape[-1]
        self._fused_entropy = None
        self._head = None
        super().__init__(batch_shape=scale.shape, event_shape=torch.Size([self.dim]), validate_args=False)

    @classmethod
    def from_head(cls, loc, raw_scale, floor=0.8, max=10.0):
        """Extension (SURVEY section 8(f)2): PowerSpherical(loc, clamp(softplus(raw_scale) + floor, max=max)) with the
        softplus + floor + clamp of the models' concentration head (mnist/mlp_vae.py:69-71: floor 0.8; cnn/models.py:96:
        floor 0.5) evaluated INSIDE the sampling kernel and its backward, so rsample() + kl_divergence stay one launch
        from the raw `fc_scale` output.  raw_scale: batch_shape or batch_shape + (1,).  `.scale` is materialised (torch
        ops) only if something asks for it."""
        self = cls.__new__(cls)
        if raw_scale.dim() == loc.dim() and raw_scale.shape[-1] == 1:
            raw_scale = raw_scale.squeeze(-1)
        self.loc = loc
        self.dim = loc.shape[-1]
        self._fused_entropy = None
        self._head = (float(floor), float(max))
        self._raw_scale = raw_scale
        Distribution.__init__(self, batch_shape=raw_scale.shape, event_shape=torch.Size([self.dim]), validate_args=False)
        return self

    def __getattr__(self, name):
        # head-built instances: the concentration as a tensor, evaluated lazily (and differentiably) on first use
        if name == "scale" and self.__dict__.get("_head") is not None:
            self.__dict__["scale"] = head_concentration(self._raw_scale, *self._head)
            return self.__dict__["scale"]
        raise AttributeError(name)

    def _flat(self):
        D = self.dim
        loc2 = self.loc.expand(tuple(self.batch_shape) + (D,)).reshape(-1, D)
        return loc2, self.scale.reshape(-1)

    def rsample(self, sample_shape=torch.Size(), _base_draws=None):
        sample_shape = torch.Size(sample_shape)
        n = _numel(sample_shape)
        if _base_draws is None:
            _base_draws = testing.take()
        if self._head is not None:
            D = self.dim
            loc2 = self.loc.expand(tuple(self.batch_shape) + (D,)).reshape(-1, D)
            param = self._raw_scale
            z, ent, dent = ops.PowerSphericalRsample.apply(loc2, param.reshape(-1), n, _base_draws, self._head)
        else:
            loc2, kap = self._flat()
            param = self.scale
            z, ent, dent = ops.PowerSphericalRsample.apply(loc2, kap, n, _base_draws)
        if ent.numel():                                             # same launch; entropy() / kl_divergence reuse it
            self._fused_entropy = ops.row_scalar(param, ent, dent).reshape(param.shape)
        return z.reshape(tuple(sample_shape) + tuple(self.batch_shape) + (self.dim,)).to(self.loc.dtype)

    def sample(self, sample_shape=torch.Size()):
        with torch.no_grad():
            return self.rsample(sample_shape)

    def log_normalizer(self):
        # log C(kappa) = -((a+b) ln 2 + lgamma(a) - lgamma(a+b) + b ln pi) evaluated on the device
        return ops.PSLogNormalizer.apply(self.scale, self.dim)

    def log_prob(self, value):
        loc2, kap = self._flat()
        D = self.dim
        lead = torch.broadcast_shapes(value.shape[:-1], tuple(self.batch_shape))
        v2 = value.expand(tuple(lead) + (D,)).reshape(-1, D)
        lp = ops.PowerSphericalLogProb.apply(v2, loc2, kap)
        return lp.reshape(lead).to(self.loc.dtype)

    def entropy(self):
        cached = self._fused_entropy
        if cached is not None:
            param = self._raw_scale if self._head is not None else self.scale
            stale = (torch.is_grad_enabled() and torch.is_tensor(param) and param.requires_grad
                     and cached.grad_fn is None and not cached.requires_grad)
            if not stale:
                return cached.to(self.loc.dtype)
        ent = ops.PSEntropy.apply(self.scale, 1, (self.dim - 1) / 2, False)
        return ent.reshape(self.scale.shape).to(self.loc.dtype)


class CliffordTorusUniform(Distribution):
    """Uniform distribution on the Clifford torus (S^1)^d (reference dists/clifford.py:215-242)."""

    arg_constraints: Dict[str, constraints.Constraint] = {}
    has_rsample = True

    def __init__(self, dim, device="cpu", dtype=torch.float32, validate_args=None):
        self.dim = dim
        self.device, self.dtype = device, dtype
        super().__init__(event_shape=torch.Size([2 * self.dim]), validate_args=validate_args)

    def rsample(self, sample_shape=torch.Size(), _base_draws=None):
        sample_shape = tuple(sample_shape)
        rows = _numel(sample_shape)
        z = ops.clifford_phases_to_vector(_base_draws, 2 * math.pi, rows, self.dim, self.device)
        return z.reshape(sample_shape + (2 * self.dim,)).to(self.dtype)

    def log_prob(self, value):
        return -torch.ones_like(value[..., 0]) * self.entropy()

    def entropy(self):
        return (self.dim - 1) * _LOG_2PI


class CliffordTorusDistribution(Distribution):
    """Product of von Mises distributions on the torus (reference dists/clifford.py:245-278).

    ``rsample`` draws the von Mises phases on the device (Best & Fisher rejection, the algorithm of
    torch.distributions.VonMises.sample that the reference calls at :262) and maps them through the same Hermitian
    spectrum -> inverse FFT kernel as the other samplers.  It is reparameterised: under autograd the launch saves the
    drawn offsets and the backward applies the implicit reparameterisation gradient of every von Mises draw (Figurnov et
    al. 2018; DESIGN.md section 6), so the reconstruction term reaches loc and concentration.  For one concentration per
    row the same launch yields the entropy, cached for ``entropy()`` / ``kl_divergence``.  Without a graph it is the
    plain sampling launch (same draws).  The reference's own method never gets that far: its Hermitian-symmetry
    assert (:274) compares against the wrong flip and raises for generic angles, so no driver uses it
    (scripts/sample_viz.py:55-64 restates the sampler inline); this is the working version of what it computes.
    ``log_prob`` sums kappa cos(angle(rfft(value)_k) - loc_k) - ln(2 pi I0(kappa)) over circles k >= 1 -- the circles of
    the entropy and of the uniform prior -- in one kernel with its value / loc / concentration gradients.
    ``entropy`` is one kernel (`cvb_clifford_vm_entropy`: the reference's eps-regularised i0e/i1e expression, evaluated
    from the fp64 log I_v of csrc/special.cuh, with its kappa-derivative).
    """

    arg_constraints: Dict[str, constraints.Constraint] = {}
    has_rsample = True

    def __init__(self, loc, concentration, validate_args=None):
        self._raw_concentration = concentration
        self.loc, self.concentration = broadcast_all(loc, concentration)
        self.orig_dim = loc.shape[-1]
        self._fused_entropy = None
        super().__init__(batch_shape=loc.shape[:-1], event_shape=torch.Size([2 * self.orig_dim]),
                         validate_args=validate_args)

    def _vm_kappa(self, row_scalar_if_expanded=False):
        """(rows, 1) for one concentration per row, else (rows, d).  row_scalar_if_expanded: a stride-0 expanded
        concentration also counts as one per row."""
        d = self.orig_dim
        raw = self._raw_concentration
        if torch.is_tensor(raw) and raw.dim() >= 1 and raw.shape[-1] == 1 and d != 1:
            return raw.expand(tuple(self.batch_shape) + (1,)).reshape(-1, 1)
        conc = self.concentration
        if row_scalar_if_expanded and conc.dim() >= 1 and conc.stride(-1) == 0:
            return conc[..., :1].reshape(-1, 1)
        return conc.reshape(-1, d)

    def rsample(self, sample_shape=torch.Size()):
        sample_shape = torch.Size(sample_shape)
        d = self.orig_dim
        n = _numel(sample_shape)
        loc2 = self.loc.reshape(-1, d)
        kap = self._vm_kappa(row_scalar_if_expanded=True)
        if torch.is_grad_enabled() and (loc2.requires_grad or kap.requires_grad):
            z, ent, dent = ops.CliffordVMRsample.apply(loc2, kap, n, True)
            if ent.numel():                                         # same launch; entropy() / kl_divergence reuse it
                self._fused_entropy = ops.row_scalar(kap, ent, dent).reshape(self.batch_shape)
        else:
            z = ops.clifford_vm_rsample(loc2, self._vm_kappa(), n)
        return z.reshape(tuple(sample_shape) + tuple(self.batch_shape) + (2 * d,)).to(self.loc.dtype)

    def log_prob(self, value):
        d = self.orig_dim
        lead = torch.broadcast_shapes(value.shape[:-1], tuple(self.batch_shape))
        v2 = value.expand(tuple(lead) + (2 * d,)).reshape(-1, 2 * d)
        lp = ops.CliffordVMLogProb.apply(v2, self.loc.reshape(-1, d), self._vm_kappa(row_scalar_if_expanded=True))
        return lp.reshape(lead).to(self.loc.dtype)

    def entropy(self):
        cached = self.__dict__.get("_fused_entropy")
        if cached is not None:
            # a value cached without a graph carries none: recompute when the caller now wants d entropy / d kappa
            kap = self._vm_kappa(row_scalar_if_expanded=True)
            stale = torch.is_grad_enabled() and kap.requires_grad and cached.grad_fn is None and not cached.requires_grad
            if not stale:
                return cached.to(self.loc.dtype)
        # one kernel: sum over circles k >= 1 of ln 2 pi + ln(i0e + eps) + kappa - kappa (i1e + eps) / (i0e + eps)
        d = self.orig_dim
        ent = ops.VMTorusEntropy.apply(self._vm_kappa(), d)
        return ent.reshape(self.batch_shape).to(self.loc.dtype)


class CliffordPowerSphericalDistribution(CliffordTorusDistribution):
    """Clifford-torus distribution with a power-spherical phase on every circle
    (reference dists/clifford.py:281-322).

    ``rsample`` is ONE fused kernel: Beta/sign draws (device Philox, or injected through the private
    ``_base_draws=(tprime, g)`` test hook) -> phases -> Hermitian phasors -> C2R inverse FFT, with the
    row entropy / dH/dkappa produced in the same pass and cached for ``entropy()`` / ``kl_divergence``
    (the reference evaluates the entropy twice per step, mnist/mlp_vae.py:126-129).
    """

    arg_constraints = {"loc": constraints.real, "concentration": constraints.positive}
    has_rsample = True

    def __init__(self, loc, concentration, validate_args=None, normalize_ifft: bool = False):
        super().__init__(loc, concentration, validate_args=validate_args)
        self.normalize_ifft = normalize_ifft
        self.dtype = loc.dtype
        self._fused_entropy = None
        self._sample_log_prob = None      # (weakref to the last no-grad sample, its version, its log_prob)
        self._head = None
        d = self.orig_dim
        conc = self.concentration
        # one concentration per row (every reference driver) vs a full (.., d) tensor
        raw = self._raw_concentration
        if torch.is_tensor(raw) and raw.dim() >= 1 and raw.shape[-1] == 1 and d != 1:
            self._kappa = raw.expand(tuple(self.batch_shape) + (1,))
        elif conc.stride(-1) == 0 or d == 1:
            self._kappa = conc[..., :1]
        else:
            self._kappa = conc

    @classmethod
    def from_head(cls, loc, raw_scale, floor=0.03, max=10.0, normalize_ifft: bool = False):
        """Extension (SURVEY section 8(f)2): CliffordPowerSphericalDistribution(loc, clamp(softplus(raw_scale) + floor,
        max=max)) with the concentration head of the reference models (mnist/mlp_vae.py:69-71: floor 0.03;
        cnn/models.py:99: floor = concentration_floor) evaluated INSIDE the fused sampling kernel and its backward:
        rsample() + kl_divergence stay ONE launch from the raw `fc_scale` / `fc_concentration` output and the gradient
        arrives at that raw tensor with the softplus / clamp chain already applied.  raw_scale: batch_shape + (1,).
        `.concentration` is materialised (torch ops) only if something asks for it."""
        self = cls.__new__(cls)
        d = loc.shape[-1]
        if raw_scale.shape[-1] != 1:
            raise ValueError("from_head needs one raw concentration per row: raw_scale of shape batch_shape + (1,)")
        Distribution.__init__(self, batch_shape=loc.shape[:-1], event_shape=torch.Size([2 * d]), validate_args=False)
        self.loc = loc
        self.orig_dim = d
        self.normalize_ifft = normalize_ifft
        self.dtype = loc.dtype
        self._fused_entropy = None
        self._sample_log_prob = None
        self._head = (float(floor), float(max))
        self._raw_scale = raw_scale.expand(tuple(self.batch_shape) + (1,))
        return self

    def __getattr__(self, name):
        # head-built instances: the concentration tensors, evaluated lazily (and differentiably) on first use
        if name in ("_kappa", "concentration", "_raw_concentration") and self.__dict__.get("_head") is not None:
            kap = head_concentration(self._raw_scale, *self._head)
            self.__dict__["_kappa"] = kap
            self.__dict__["_raw_concentration"] = kap
            self.__dict__["concentration"] = kap.expand_as(self.loc)
            return self.__dict__[name]
        raise AttributeError(name)

    def _flat(self):
        d = self.orig_dim
        return self.loc.reshape(-1, d), self._kappa.reshape(-1, self._kappa.shape[-1])

    def rsample(self, sample_shape=torch.Size(), _base_draws=None) -> torch.Tensor:
        sample_shape = torch.Size(sample_shape)
        n = _numel(sample_shape)
        d = self.orig_dim
        out_shape = tuple(sample_shape) + tuple(self.batch_shape) + (2 * d,)
        if _base_draws is None:
            _base_draws = testing.take()
        if self._head is not None and torch.is_grad_enabled() and (self.loc.requires_grad or self._raw_scale.requires_grad):
            # training path from the raw head output: softplus + floor + clamp inside the kernel
            raw2 = self._raw_scale.reshape(-1, 1)
            z, ent, dent = ops.CliffordPSRsample.apply(self.loc.reshape(-1, d), raw2, n, _base_draws, True, self._head)
            if ent.numel():
                self._fused_entropy = ops.row_scalar(raw2, ent, dent).reshape(self.batch_shape)
            return z.reshape(out_shape).to(self.dtype)
        loc2, kap2 = self._flat()
        no_grad = not (torch.is_grad_enabled() and (loc2.requires_grad or kap2.requires_grad))
        if (no_grad and len(sample_shape) > 0 and kap2.shape[-1] == 1 and 16 <= d <= 8192 and (d & (d - 1)) == 0
                and loc2.shape[0] > 0 and n > 0):
            # evaluation path (IWAE, mnist/mlp_vae.py:161,181: q_z.rsample(torch.Size([n_samples])) then
            # q_z.log_prob(z)): the same launch also yields log q(z) of the sample, which log_prob() returns when it
            # is handed this very tensor back.  A plain rsample() (empty sample_shape) skips it.
            z, lp, ent = ops.clifford_rsample_log_prob(loc2.detach(), kap2.detach(), n, _base_draws)
            if ent is not None:
                self._fused_entropy = ent.reshape(self.batch_shape)
            z = z.reshape(out_shape).to(self.dtype)
            self._sample_log_prob = (weakref.ref(z), z._version, lp.reshape(out_shape[:-1]))
            return z
        z, ent, dent = ops.CliffordPSRsample.apply(loc2, kap2, n, _base_draws, True)
        if ent.numel():
            self._fused_entropy = ops.row_scalar(kap2, ent, dent).reshape(self.batch_shape)
        return z.reshape(out_shape).to(self.dtype)

    def rsample_bind(self, other, sample_shape=torch.Size(), return_sample=True, _base_draws=None):
        """Extension (not in the reference): draw z and return bind(z, other); with return_sample=False from ONE
        kernel.  The sample's spectrum is the unit phasors themselves, so binding it costs one forward FFT of `other`
        and one inverse FFT, and z is never materialised.  `other`: (2d,), (1, 2d) or sample_shape + batch_shape + (2d,).  Forward only
        (under autograd use rsample() and utils.vsa.bind).  Returns (z, bound), or bound if return_sample=False."""
        from . import vsa
        sample_shape = torch.Size(sample_shape)
        loc2, kap2 = self._flat()
        d = self.orig_dim
        n = _numel(sample_shape)
        out_shape = tuple(sample_shape) + tuple(self.batch_shape) + (2 * d,)
        # the one-kernel path pays off when z itself is not wanted (its inverse FFT and 8d bytes of writes are skipped:
        # 12-17 % faster than rsample + bind); with z written the two specialised kernels are faster than the fused one
        fast = (not return_sample) and kap2.shape[-1] == 1 and d >= 16 and d <= 8192 and (d & (d - 1)) == 0
        if not fast:
            z = self.rsample(sample_shape, _base_draws=_base_draws)
            bound = vsa.bind(z, other)
            return (z, bound) if return_sample else bound
        oth = other if other.numel() == 2 * d else other.expand(out_shape)
        with torch.no_grad():
            z, bound, ent = ops.clifford_rsample_bind(loc2, kap2, oth, n, _base_draws, return_sample)
        if ent is not None and not (kap2.requires_grad and torch.is_grad_enabled()):
            self._fused_entropy = ent.reshape(self.batch_shape)     # forward-only value: never cached under autograd
        bound = bound.reshape(out_shape).to(self.dtype)
        return (z.reshape(out_shape).to(self.dtype), bound) if return_sample else bound

    def log_prob(self, value):
        cached = self._sample_log_prob
        if cached is not None and cached[0]() is value and value._version == cached[1] and not (
                torch.is_grad_enabled() and (value.requires_grad or self.loc.requires_grad or self._kappa.requires_grad)):
            return cached[2].to(self.dtype)
        loc2, kap2 = self._flat()
        n = 2 * self.orig_dim
        lead = torch.broadcast_shapes(value.shape[:-1], tuple(self.batch_shape))
        v2 = value.expand(tuple(lead) + (n,)).reshape(-1, n)
        lp = ops.CliffordPSLogProb.apply(v2, loc2, kap2)
        return lp.reshape(lead).to(self.dtype)

    def entropy(self):
        cached = self._fused_entropy
        if cached is not None:
            # a value cached by a no-grad rsample (evaluation path) carries no graph: recompute when the caller now
            # wants d entropy / d kappa
            param = self._raw_scale if self._head is not None else self._kappa
            stale = (torch.is_grad_enabled() and param.requires_grad and cached.grad_fn is None
                     and not cached.requires_grad)
            if not stale:
                return cached.to(self.dtype)
        _, kap2 = self._flat()
        ent = ops.PSEntropy.apply(kap2, self.orig_dim, 0.5, True)
        return ent.reshape(self.batch_shape).to(self.dtype)


@register_kl(CliffordPowerSphericalDistribution, CliffordTorusUniform)
def _kl_ps_uniform(p, q):
    return -p.entropy() + q.entropy()


@register_kl(CliffordTorusDistribution, CliffordTorusUniform)
def _kl_vm_uniform(p, q):
    return -p.entropy() + q.entropy()


@register_kl(PowerSpherical, HypersphericalUniform)
def _kl_powerspherical_uniform(p, q):
    return -p.entropy() + q.entropy()
