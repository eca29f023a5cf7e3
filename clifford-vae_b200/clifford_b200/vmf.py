"""von Mises-Fisher distribution and its uniform prior with the reference's class names and
constructor signatures (reference vmf/hyperspherical_vae/distributions/{von_mises_fisher,
hyperspherical_uniform}.py), backed by the sm_100a kernels: the Wood rejection loop runs on the
device (no host RNG, no `while mask.sum()` sync) and log I_v replaces the host SciPy call.
"""
from __future__ import annotations

import math

import torch
from torch.distributions.kl import register_kl

from . import ops, testing
from .distributions import _keep_fused, _stale, head_concentration


class HypersphericalUniform(torch.distributions.Distribution):
    """Uniform on S^dim (dim = m - 1), reference hyperspherical_uniform.py:5-54."""

    arg_constraints = {}
    support = torch.distributions.constraints.real
    has_rsample = False
    _mean_carrier_measure = 0

    @property
    def dim(self):
        return self._dim

    @property
    def device(self):
        return self._device

    @device.setter
    def device(self, val):
        self._device = val if isinstance(val, torch.device) else torch.device(val)

    def __init__(self, dim, validate_args=None, device="cpu"):
        super().__init__(torch.Size([dim]), validate_args=validate_args)
        self._dim = dim
        # the reference ignores `device` and picks cuda when available (:27)
        self.device = torch.device("cuda" if torch.cuda.is_available() else "cpu")

    def sample(self, shape=torch.Size()):
        shape = shape if isinstance(shape, torch.Size) else torch.Size([shape])
        rows = 1
        for s in shape:
            rows *= int(s)
        z = ops.sphere_uniform_rsample(rows, self._dim + 1, self.device, 0.0)
        return z.reshape(tuple(shape) + (self._dim + 1,))

    def entropy(self):
        return self.__log_surface_area()

    def log_prob(self, x):
        return -torch.ones(x.shape[:-1], device=self.device) * self.__log_surface_area()

    def __log_surface_area(self):
        val = math.log(2) + ((self._dim + 1) / 2) * math.log(math.pi) - math.lgamma((self._dim + 1) / 2)
        return torch.full((1,), val, device=self.device, dtype=torch.float32)


class VonMisesFisher(torch.distributions.Distribution):
    """reference von_mises_fisher.py:11-217.  loc (..., m) unit rows, scale (..., 1)."""

    arg_constraints = {
        "loc": torch.distributions.constraints.real,
        "scale": torch.distributions.constraints.positive,
    }
    support = torch.distributions.constraints.real
    has_rsample = True
    _mean_carrier_measure = 0

    def __init__(self, loc, scale, validate_args=None, k=1):
        self.dtype = loc.dtype
        self.loc = loc
        self.scale = scale
        self.device = loc.device
        self._m = loc.shape[-1]
        self.k = k
        self._fused = None
        self._head = None
        super().__init__(self.loc.size(), validate_args=validate_args)   # batch_shape quirk kept (:44)

    @classmethod
    def from_head(cls, loc, raw_scale, floor=0.8, max=10.0, k=1):
        """Extension (SURVEY section 8(f)2): VonMisesFisher(loc, clamp(softplus(raw_scale) + floor, max=max)) with the
        concentration head of mnist/mlp_vae.py:69-71 evaluated INSIDE the sampling kernel and its backward (one launch
        from the raw `fc_scale` output; gradients arrive at raw_scale).  raw_scale: loc.shape[:-1] + (1,).  `.scale` is
        materialised (torch ops) only if something asks for it."""
        self = cls.__new__(cls)
        self.dtype = loc.dtype
        self.loc = loc
        self.device = loc.device
        self._m = loc.shape[-1]
        self.k = k
        self._fused = None
        self._head = (float(floor), float(max))
        self._raw_scale = raw_scale
        torch.distributions.Distribution.__init__(self, self.loc.size(), validate_args=False)
        return self

    def __getattr__(self, name):
        if name == "scale" and self.__dict__.get("_head") is not None:
            self.__dict__["scale"] = head_concentration(self._raw_scale, *self._head)
            return self.__dict__["scale"]
        raise AttributeError(name)

    @property
    def mean(self):
        ratio = _ive_fraction_approx2(torch.tensor(self._m / 2, dtype=torch.float64, device=self.device),
                                      self.scale.to(torch.float64))
        return (self.loc.to(torch.float64) * ratio).type(self.dtype)

    @property
    def stddev(self):
        return self.scale

    def sample(self, shape=torch.Size()):
        with torch.no_grad():
            return self.rsample(shape)

    def rsample(self, shape=torch.Size(), _base_draws=None):
        shape = shape if isinstance(shape, torch.Size) else torch.Size([shape])
        m = self._m
        loc2 = self.loc.reshape(-1, m)
        param = self._raw_scale if self._head is not None else self.scale       # head: the kernels apply softplus/floor/clamp
        kap = param.expand(tuple(self.loc.shape[:-1]) + (1,)).reshape(-1, 1)
        n = 1
        for s in shape:
            n *= int(s)
        if _base_draws is None:
            _base_draws = testing.take()
        z, ent, ln, dent, dln = ops.VMFRsample.apply(loc2, kap, n, _base_draws, self._head)
        if tuple(param.shape) == tuple(self.loc.shape[:-1]) + (1,):
            _keep_fused(self, "_fused", param, param.shape[:-1], (ent, dent), (ln, dln))
        return z.reshape(tuple(shape) + tuple(self.loc.shape)).type(self.dtype)

    def _ent_ln(self):
        cached = self._fused
        if cached is not None and not _stale(cached[0], self._raw_scale if self._head is not None else self.scale):
            return cached
        ent, ln = ops.VMFEntropyLogNorm.apply(self.scale, self._m)
        shp = self.scale.shape[:-1]
        return ent.reshape(shp), ln.reshape(shp)

    def entropy(self):
        return self._ent_ln()[0].type(self.dtype)

    def log_prob(self, x):
        # one kernel: kappa <loc, x> - log_norm per row (von_mises_fisher.py:193-212)
        m = self._m
        lead = tuple(self.loc.shape[:-1])
        if tuple(self.scale.shape) != lead + (1,) or tuple(x.shape[-len(lead) - 1:]) != lead + (m,):
            return self._log_unnormalized_prob(x) - self._log_normalization()       # exotic broadcasting: torch ops
        lp = ops.VMFLogProb.apply(x.reshape(-1, m), self.loc.reshape(-1, m), self.scale.reshape(-1),
                                  self._log_normalization().reshape(-1))
        return lp.reshape(x.shape[:-1]).type(self.dtype)

    def _log_unnormalized_prob(self, x):
        # kappa * <loc, x>: a row dot product -- the cosine kernel's numerator; use the PS log-prob
        # kernel's dot path is overkill here, this is a (B,) op outside every reference driver's loop
        output = self.scale * (self.loc * x).sum(-1, keepdim=True)
        return output.view(*(output.shape[:-1]))

    def _log_normalization(self):
        return self._ent_ln()[1].type(self.dtype)


def _ive_fraction_approx2(v, z, eps=1e-20):
    def delta_a(a):
        lamb = v + (a - 1.0) / 2.0
        return (v - 0.5) + lamb / (2 * torch.sqrt((torch.pow(lamb, 2) + torch.pow(z, 2)).clamp(eps)))

    d0, d2 = delta_a(0.0), delta_a(2.0)
    b0 = z / (d0 + torch.sqrt((torch.pow(d0, 2) + torch.pow(z, 2))).clamp(eps))
    b2 = z / (d2 + torch.sqrt((torch.pow(d2, 2) + torch.pow(z, 2))).clamp(eps))
    return (b0 + b2) / 2.0


@register_kl(VonMisesFisher, HypersphericalUniform)
def _kl_vmf_uniform(vmf, hyu):
    return -vmf.entropy() + hyu.entropy()
