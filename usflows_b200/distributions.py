"""Base distributions as modules with constrained learnable parameters -- drop-in mirrors of the reference's
`DistributionModule`, `Laplace`, `Normal`, `Independent` (src/usflows/distributions.py:117-238, 709-728) and of the
Lp-radial family `RadialDistribution` with `LogNormal` / `GammaMM` radius distributions (:181-197, 327-372, 478-549,
674-707) that the reference's image configurations use as the base (experiments/mnist/mnist.yaml:79-92).

Parameter names match the reference (`loc`, `scale_unconstrained`, scale = softplus(scale_unconstrained)).
`log_prob` and `sample` run the fused base-density / Philox sampling kernels; no torch.distributions object is
rebuilt per call (the reference does that on every access, distributions.py:129-138).
"""
from __future__ import annotations

import math
from typing import Iterable, Optional

import torch
from torch.nn import Module, Parameter

from . import ops
from .utils import inv_softplus


class DistributionModule(Module):
    base_kind: int = -1

    def __init__(self, n_batch_dims: int = 0):
        super().__init__()
        self.n_batch_dims = n_batch_dims

    # -- prepared parameters (scale = softplus(scale_unconstrained)), cached per weight version ------
    def _prepared(self):
        key = tuple((p.data_ptr(), p._version) for p in (self.loc, self.scale_unconstrained))
        if getattr(self, "_prep_key", None) != key:
            ops.require_cuda(self.loc, "base_distribution.loc")
            with torch.no_grad(), ops.on_device(self.loc):
                raw = self.scale_unconstrained.detach()
                if raw.dim() == 0:                                 # scalar scale expands to loc's shape (:228-232)
                    raw = raw.expand_as(self.loc)
                raw = raw.reshape(-1).contiguous()
                scale = torch.empty_like(raw)
                ops.softplus(raw, scale)
                loc = self.loc.detach().reshape(-1).contiguous()
            self._prep_cache, self._prep_key = (loc, scale), key
        return self._prep_cache

    def _permuted(self, perm: torch.Tensor):
        """Prepared parameters re-ordered for an event held in another element order (channels-last images)."""
        loc, scale = self._prepared()
        key = (self._prep_key, perm.data_ptr())
        if getattr(self, "_perm_key", None) != key:
            self._perm_cache, self._perm_key = (loc[perm].contiguous(), scale[perm].contiguous()), key
        return self._perm_cache

    def _density_into(self, z: "ops.Act", add_const: float, out: torch.Tensor, perm: Optional[torch.Tensor] = None) -> None:
        """out[r] = log p(z[r, :]) + add_const on the current stream (the tail of `Flow.log_prob`); with `perm`, column j
        of z holds event element perm[j]."""
        loc, scale = self._prepared() if perm is None else self._permuted(perm)
        ops.base_logprob(z, loc, scale, self.base_kind, add_const, out)

    def _sample_into(self, out: torch.Tensor, draw: "ops.Draw") -> None:
        loc, scale = self._prepared()
        a = ops.Act(out.shape[0], out.shape[1], f32=out)
        if draw.plain:
            ops.base_sample(a, loc, scale, self.base_kind, draw.seed, draw.offset)
        else:
            ops.base_sample_at(a, loc, scale, self.base_kind, draw)

    @property
    def event_shape(self) -> torch.Size:
        return torch.Size(self.loc.shape[self.n_batch_dims:])

    @property
    def batch_shape(self) -> torch.Size:
        return torch.Size(self.loc.shape[:self.n_batch_dims])

    def _get_distribution_params(self):
        """Current constrained parameters (distributions.py:141-143, 211-215, 234-238)."""
        raw = self.scale_unconstrained
        if raw.dim() == 0:
            raw = raw.expand_as(self.loc)
        return {"loc": self.loc, "scale": torch.nn.functional.softplus(raw)}

    @property
    def distribution(self) -> torch.distributions.Distribution:
        """The `torch.distributions` object the reference rebuilds on every access (distributions.py:129-138), for callers
        that want it (entropy, cdf, ...); `log_prob` / `sample` of this module run the fused kernels instead."""
        cls = torch.distributions.Laplace if self.base_kind == ops.BASE_LAPLACE else torch.distributions.Normal
        d = cls(**self._get_distribution_params())
        extra = len(d.batch_shape) - self.n_batch_dims
        return torch.distributions.Independent(d, extra) if extra > 0 else d

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.log_prob(x)

    def log_prob(self, x: torch.Tensor) -> torch.Tensor:
        """sum over the event dims of the Laplace / Normal log-density (distributions.py:150-151)."""
        from . import engine
        return engine.base_log_prob(self, x)

    def sample(self, sample_shape: Optional[Iterable[int]] = None) -> torch.Tensor:
        from . import engine
        return engine.base_sample(self, sample_shape)


class Laplace(DistributionModule):
    base_kind = ops.BASE_LAPLACE

    def __init__(self, loc: torch.Tensor, scale: torch.Tensor, device: str = "cpu"):
        super().__init__()
        self.loc = Parameter(loc)
        self.scale_unconstrained = Parameter(inv_softplus(scale))
        self.to(device)


class Normal(DistributionModule):
    base_kind = ops.BASE_NORMAL

    def __init__(self, loc: torch.Tensor, scale: torch.Tensor, device: str = "cpu"):
        super().__init__()
        self.loc = Parameter(loc)
        self.scale_unconstrained = Parameter(inv_softplus(scale))
        self.to(device)


class _FrozenBase(DistributionModule):
    """A plain `torch.distributions.Laplace` / `Normal` object (optionally inside `torch.distributions.Independent`) as
    the base -- the reference's `Flow` takes any object with `log_prob` / `sample` / `batch_shape` and makes the batch dims
    event dims (flows.py:97-101); its older configurations pass `pyro.distributions.Laplace(loc, scale)` this way.  The
    values are read once into non-persistent buffers: no parameters and no state-dict keys, as in the reference."""

    def __init__(self, dist):
        super().__init__()
        D = torch.distributions
        while isinstance(dist, D.Independent):
            dist = dist.base_dist
        if isinstance(dist, D.Laplace):
            self.base_kind = ops.BASE_LAPLACE
        elif isinstance(dist, D.Normal):
            self.base_kind = ops.BASE_NORMAL
        else:
            raise NotImplementedError(f"usflows_b200.Flow: base distribution {type(dist).__name__} is not built (Laplace, "
                                      "Normal, RadialDistribution modules and torch Laplace / Normal objects are)")
        loc, scale = torch.broadcast_tensors(torch.as_tensor(dist.loc, dtype=torch.float32),
                                             torch.as_tensor(dist.scale, dtype=torch.float32))
        self._torch_dist = dist
        self.register_buffer("loc", loc.detach().clone(), persistent=False)
        self.register_buffer("scale_unconstrained", inv_softplus(scale.detach().clone()), persistent=False)

    @property
    def distribution(self) -> torch.distributions.Distribution:
        d = self._torch_dist
        return torch.distributions.Independent(d, len(d.batch_shape)) if len(d.batch_shape) else d


class Independent(Module):
    """Reinterprets batch dims of a DistributionModule as event dims (distributions.py:709-728).  The fused
    base-density kernel already sums over every non-batch dim, so this is bookkeeping only."""

    def __init__(self, base_distribution: DistributionModule, reinterpreted_batch_ndims: int = 0):
        super().__init__()
        if isinstance(base_distribution, torch.distributions.Distribution):   # the reference's wraps torch objects (:712-728)
            # a torch Laplace / Normal [d] has batch_shape [d]; the frozen module treats those dims as the event already
            base_distribution, reinterpreted_batch_ndims = _FrozenBase(base_distribution), 0
        self._base_distribution = base_distribution
        self.reinterpreted_batch_ndims = reinterpreted_batch_ndims

    @property
    def base_dist(self):
        return self._base_distribution

    @property
    def batch_shape(self):
        bs = self._base_distribution.batch_shape
        return torch.Size(bs[:len(bs) - self.reinterpreted_batch_ndims])

    @property
    def event_shape(self):
        bs = self._base_distribution.batch_shape
        return torch.Size(bs[len(bs) - self.reinterpreted_batch_ndims:]) + self._base_distribution.event_shape

    def log_prob(self, x):
        return self._base_distribution.log_prob(x)

    def sample(self, sample_shape=None):
        return self._base_distribution.sample(sample_shape)


# --------------------------------------------------------------------------------------------------
# Lp-radial base distributions (distributions.py:327-549)
# --------------------------------------------------------------------------------------------------
class _RadiusDistribution(Module):
    """Distribution of the radial component: a parameter container (reference parameter names) whose density is
    evaluated inside the radial kernels (`usf_radial_logprob` / `usf_radial_sample`)."""

    norm_kind: int = -1

    def _params(self):
        raise NotImplementedError

    def _norm_params(self):
        """(kind, n_components, device fp32 vector in the layout of USF_NORM_*), cached per weight version."""
        ps = self._params()
        key = tuple((p.data_ptr(), p._version) for p in ps)
        if getattr(self, "_prep_key", None) != key:
            for p in ps:
                ops.require_cuda(p, "norm_distribution parameter")
            with torch.no_grad():
                self._prep_cache = self._pack()
            self._prep_key = key
        return self._prep_cache

    def log_prob(self, r: torch.Tensor) -> torch.Tensor:
        """log f_R(r) on its own (the reference's `DistributionModule.log_prob`, distributions.py:150-151): the radial
        density kernel on a one-dimensional event -- ||r||_inf = |r|, volume term switched off."""
        ops.require_cuda(r, "radius")
        kind, K, params = self._norm_params()
        flat = r.reshape(-1, 1).contiguous()
        out = torch.empty(flat.shape[0], dtype=torch.float32, device=flat.device)
        if flat.shape[0]:
            with ops.on_device(flat):
                ops.radial_logprob(ops.Act(flat.shape[0], 1, f32=flat), torch.zeros(1, device=flat.device), ops.LP_INF, kind,
                                   params, K, 0.0, 0.0, out)
        shape = r.shape[:-1] if r.dim() and r.shape[-1] == 1 else r.shape      # the radius arrives as [..., 1] (:508)
        return out.reshape(shape)

    def sample(self, sample_shape=None) -> torch.Tensor:
        """Draws of R (the radial sampling kernel on a one-dimensional event: the Lp-sphere direction is +1)."""
        from . import engine
        kind, K, params = self._norm_params()
        shape = [int(n) for n in (sample_shape if sample_shape is not None else [])]
        out = torch.empty(max(1, math.prod(shape)), 1, dtype=torch.float32, device=params.device)
        seed, offset = engine.philox_call_stream(out.device)
        with ops.on_device(out):
            ops.radial_sample(out, torch.zeros(1, device=out.device), ops.LP_INF, kind, params, K, seed, offset)
        return out.reshape(*shape, 1)


def _softplus_vec(raw: torch.Tensor) -> torch.Tensor:
    raw = raw.detach().reshape(-1).contiguous()
    out = torch.empty_like(raw)
    with ops.on_device(raw):
        ops.softplus(raw, out)
    return out


class LogNormal(_RadiusDistribution):
    """log R ~ Normal(loc, softplus(scale_unconstrained))  (distributions.py:181-197); one-element loc / scale."""

    norm_kind = ops.NORM_LOGNORMAL

    def __init__(self, loc: torch.Tensor, scale: torch.Tensor, device: str = "cpu"):
        super().__init__()
        if loc.numel() != 1 or scale.numel() != 1:
            raise NotImplementedError("usflows_b200.LogNormal: one radius distribution per flow (1-element loc / scale)")
        self.loc = Parameter(loc)
        self.scale_unconstrained = Parameter(inv_softplus(scale))
        self.to(device)

    def _params(self):
        return (self.loc, self.scale_unconstrained)

    def _pack(self):
        buf = torch.empty(2, dtype=torch.float32, device=self.loc.device)
        buf[0:1].copy_(self.loc.detach().reshape(-1))
        buf[1:2].copy_(_softplus_vec(self.scale_unconstrained))
        return ops.NORM_LOGNORMAL, 1, buf

    def _lognormals(self):
        mu = self.loc.reshape(1)
        return torch.zeros_like(mu), mu, torch.nn.functional.softplus(self.scale_unconstrained).reshape(1)


class _GammaFamily(_RadiusDistribution):
    """Radius distributions that are a mixture of (generalised) Gammas: R = scale_k * S^(1 / power_k), S ~ Gamma(a_k, b_k).
    `_mixture()` hands the constrained values (logits [K], concentration [K], rate [K], scale [K] or None, power [K] or
    None) over as differentiable tensors -- the radial kernels read them packed (USF_NORM_GAMMA_MIXTURE without scale /
    power, USF_NORM_GENGAMMA_MIXTURE with), the training route and the exportable module evaluate them with torch."""

    def _mixture(self):
        raise NotImplementedError

    def _pack(self):
        logits, conc, rate, scale, power = self._mixture()
        K = logits.numel()
        parts = [logits, conc, rate] + ([] if scale is None else [scale, power])
        buf = torch.empty(len(parts) * K, dtype=torch.float32, device=logits.device)
        for i, t in enumerate(parts):
            buf[i * K:(i + 1) * K].copy_(t.detach().reshape(-1))
        return (ops.NORM_GAMMA_MIXTURE if scale is None else ops.NORM_GENGAMMA_MIXTURE), K, buf


class _LogNormalFamily(_RadiusDistribution):
    """Radius distributions that are a mixture of log-normals: `_lognormals()` -> (logits [K], mu [K], sigma [K])."""

    def _lognormals(self):
        raise NotImplementedError

    def _pack(self):
        logits, mu, sigma = self._lognormals()
        K = logits.numel()
        if K == 1:                                           # the single log-normal keeps its own kernel branch
            buf = torch.cat([mu.detach().reshape(-1), sigma.detach().reshape(-1)]).to(torch.float32)
            return ops.NORM_LOGNORMAL, 1, buf
        buf = torch.cat([t.detach().reshape(-1) for t in (logits, mu, sigma)]).to(torch.float32)
        return ops.NORM_LOGNORMAL_MIXTURE, K, buf


def _mixture_args(*tensors):
    if any(t.dim() != 1 or t.shape != tensors[0].shape for t in tensors):
        raise NotImplementedError("usflows_b200: radius mixtures take 1-D [K] parameter tensors")


class GammaMM(_GammaFamily):
    """Mixture of K Gamma(concentration_k, rate_k) with weights softmax(mixture_logits)  (distributions.py:674-707)."""

    norm_kind = ops.NORM_GAMMA_MIXTURE

    def __init__(self, concentration: torch.Tensor, rate: torch.Tensor, mixture_weights: torch.Tensor, device: str = "cpu"):
        super().__init__()
        if concentration.dim() != 1 or rate.shape != concentration.shape or mixture_weights.shape != concentration.shape:
            raise NotImplementedError("usflows_b200.GammaMM: 1-D [K] concentration / rate / mixture_weights")
        self.concentration_unconstrained = Parameter(inv_softplus(concentration))
        self.rate_unconstrained = Parameter(inv_softplus(rate))
        self.mixture_logits = Parameter(mixture_weights)      # used as logits, as the reference does (:701)
        self.to(device)

    def _params(self):
        return (self.mixture_logits, self.concentration_unconstrained, self.rate_unconstrained)

    def _mixture(self):
        sp = torch.nn.functional.softplus
        return self.mixture_logits, sp(self.concentration_unconstrained), sp(self.rate_unconstrained), None, None


class _MixtureModel:
    """Parameter layout of the reference's `MixtureModel` (distributions.py:730-795): `unconstrained_params` (a
    ParameterList in the order of the component's arguments, positive ones stored through inv_softplus) and
    `mixture_logits` -- state-dict keys `unconstrained_params.0`, `unconstrained_params.1`, `mixture_logits`."""

    def _init_mixture(self, params, positive, mixture_weights, device):
        _mixture_args(*params, mixture_weights)
        self.unconstrained_params = torch.nn.ParameterList(
            [Parameter(inv_softplus(p) if pos else p) for p, pos in zip(params, positive)])
        self._positive = tuple(positive)
        self.mixture_logits = Parameter(mixture_weights)
        self.to(device)

    def _params(self):
        return (self.mixture_logits, *self.unconstrained_params)

    def _constrained(self):
        sp = torch.nn.functional.softplus
        return [sp(p) if pos else p for p, pos in zip(self.unconstrained_params, self._positive)]


class WeibullMM(_MixtureModel, _GammaFamily):
    """Mixture of K Weibull(scale_k, concentration_k) (distributions.py:835-848): R = scale * E^(1 / concentration),
    E ~ Exponential(1) = Gamma(1, 1)."""

    norm_kind = ops.NORM_GENGAMMA_MIXTURE

    def __init__(self, scale: torch.Tensor, concentration: torch.Tensor, mixture_weights: torch.Tensor, device: str = "cpu"):
        _GammaFamily.__init__(self)
        self._init_mixture((scale, concentration), (True, True), mixture_weights, device)

    def _mixture(self):
        scale, conc = self._constrained()
        one = torch.ones_like(scale)
        return self.mixture_logits, one, one, scale, conc


class LogNormalMM(_MixtureModel, _LogNormalFamily):
    """Mixture of K LogNormal(loc_k, scale_k) (distributions.py:821-833)."""

    norm_kind = ops.NORM_LOGNORMAL_MIXTURE

    def __init__(self, loc: torch.Tensor, scale: torch.Tensor, mixture_weights: torch.Tensor, device: str = "cpu"):
        _LogNormalFamily.__init__(self)
        self._init_mixture((loc, scale), (False, True), mixture_weights, device)

    def _lognormals(self):
        loc, scale = self._constrained()
        return self.mixture_logits, loc, scale


class Gamma(_GammaFamily):
    """Gamma(softplus(concentration_unconstrained), softplus(rate_unconstrained)) radius (distributions.py:162-179);
    one-element concentration / rate -- a one-component mixture for the kernels."""

    norm_kind = ops.NORM_GAMMA_MIXTURE

    def __init__(self, concentration: torch.Tensor, rate: torch.Tensor, device: str = "cpu"):
        super().__init__()
        if concentration.numel() != 1 or rate.numel() != 1:
            raise NotImplementedError("usflows_b200.Gamma: one radius distribution per flow (1-element concentration / rate)")
        self.concentration_unconstrained = Parameter(inv_softplus(concentration))
        self.rate_unconstrained = Parameter(inv_softplus(rate))
        self.to(device)

    def _params(self):
        return (self.concentration_unconstrained, self.rate_unconstrained)

    def _mixture(self):
        sp = torch.nn.functional.softplus
        conc = sp(self.concentration_unconstrained).reshape(1)
        return torch.zeros_like(conc), conc, sp(self.rate_unconstrained).reshape(1), None, None


class Chi(_GammaFamily):
    """R = scale * sqrt(S), S ~ Chi2(df) = Gamma(df / 2, 1 / 2)  (distributions.py:55-115; the radius of a `scale`-scaled
    standard normal in `df` dimensions).  No learnable parameters, as in the reference; `df` / `scale` are buffers so that
    `.to(device)` moves them."""

    norm_kind = ops.NORM_GENGAMMA_MIXTURE

    def __init__(self, df, scale: float = 1.0, validate_args=None, device: str = "cpu"):
        super().__init__()
        df_t = torch.as_tensor(df, dtype=torch.float32).reshape(-1)
        if df_t.numel() != 1:
            raise NotImplementedError("usflows_b200.Chi: one radius distribution per flow (scalar df)")
        if not (float(df_t) > 0 and float(scale) > 0):
            raise ValueError("Chi: df and scale must be positive")
        self.df, self.scale = df, scale
        self.register_buffer("_df", df_t, persistent=False)
        self.register_buffer("_scale", torch.full((1,), float(scale)), persistent=False)
        self.to(device)

    def _params(self):
        return (self._df, self._scale)

    def _mixture(self):
        return (torch.zeros_like(self._df), self._df / 2, torch.full_like(self._df, 0.5), self._scale,
                torch.full_like(self._df, 2.0))

    # the two closed forms the reference's class adds to log_prob / sample (distributions.py:98-115); accessors, evaluated
    # through torch's Chi2 like there
    def cdf(self, value: torch.Tensor) -> torch.Tensor:
        return torch.distributions.Chi2(self._df.to(value.device)).cdf((value / self.scale) ** 2)

    def entropy(self) -> torch.Tensor:
        return torch.distributions.Chi2(self._df).entropy() / 2 + math.log(2.0) + math.log(float(self.scale))


def _frozen(t) -> torch.Tensor:
    return torch.as_tensor(t, dtype=torch.float32).detach().reshape(-1).clone()


class _TorchGammaRadius(_GammaFamily):
    """A frozen `torch.distributions` object as the radius distribution -- the reference's configurations pass them straight
    into `RadialDistribution` (experiments/mnist/mnist_digits_minimal_radial_{chi2,weilbul,exponential}.yaml,
    mnist_digits_minimal_radialdists.yaml:81-95).  Chi2(df) = Gamma(df / 2, 1 / 2); Exponential(rate) = Gamma(1, rate);
    HalfNormal(s) = s sqrt(Chi2(1)); Weibull(scale, k) = scale Exponential(1)^(1 / k); `torch.distributions.Gamma` as is.
    Values are read at construction (these objects carry no parameters in the reference either)."""

    def __init__(self, dist):
        super().__init__()
        D = torch.distributions
        scale = power = None
        if isinstance(dist, D.Chi2):                # before Gamma: Chi2 is a Gamma subclass
            conc = _frozen(dist.df) / 2
            rate = torch.full_like(conc, 0.5)
        elif isinstance(dist, D.Gamma):
            conc, rate = _frozen(dist.concentration), _frozen(dist.rate)
        elif isinstance(dist, D.Exponential):
            rate = _frozen(dist.rate)
            conc = torch.ones_like(rate)
        elif isinstance(dist, D.HalfNormal):
            scale = _frozen(dist.scale)
            conc, rate, power = torch.full_like(scale, 0.5), torch.full_like(scale, 0.5), torch.full_like(scale, 2.0)
        elif isinstance(dist, D.Weibull):
            scale, power = _frozen(dist.scale), _frozen(dist.concentration)
            conc, rate = torch.ones_like(scale), torch.ones_like(scale)
        else:
            raise NotImplementedError(type(dist).__name__)
        if conc.numel() != 1:
            raise NotImplementedError("usflows_b200.RadialDistribution: one radius distribution per flow (scalar parameters)")
        self.distribution = dist
        self.norm_kind = ops.NORM_GAMMA_MIXTURE if scale is None else ops.NORM_GENGAMMA_MIXTURE
        for name, t in (("_conc", conc), ("_rate", rate), ("_scale", scale), ("_power", power)):
            self.register_buffer(name, t, persistent=False)

    def _params(self):
        return (self._conc, self._rate)

    def _mixture(self):
        return torch.zeros_like(self._conc), self._conc, self._rate, self._scale, self._power


class _TorchLogNormalRadius(_LogNormalFamily):
    """A frozen `torch.distributions.LogNormal` (pyro's is a subclass) as the radius distribution
    (experiments/mnist/mnist_digits_minimal_radial_lognormal.yaml)."""

    norm_kind = ops.NORM_LOGNORMAL

    def __init__(self, dist):
        super().__init__()
        mu, sigma = _frozen(dist.loc), _frozen(dist.scale)
        if mu.numel() != 1 or sigma.numel() != 1:
            raise NotImplementedError("usflows_b200.RadialDistribution: one radius distribution per flow (scalar parameters)")
        self.distribution = dist
        self.register_buffer("_mu", mu, persistent=False)
        self.register_buffer("_sigma", sigma, persistent=False)

    def _params(self):
        return (self._mu, self._sigma)

    def _lognormals(self):
        return torch.zeros_like(self._mu), self._mu, self._sigma


def _wrap_torch_radius(dist):
    D = torch.distributions
    if isinstance(dist, D.LogNormal):
        return _TorchLogNormalRadius(dist)
    if isinstance(dist, (D.Gamma, D.Exponential, D.HalfNormal, D.Weibull)):
        return _TorchGammaRadius(dist)
    raise NotImplementedError(f"usflows_b200.RadialDistribution: radius distribution {type(dist).__name__} is not built "
                              "(LogNormal, LogNormalMM, GammaMM, Gamma, WeibullMM, Chi, torch LogNormal / Gamma / Chi2 / "
                              "Exponential / HalfNormal / Weibull are)")


class RadialDistribution(Module):
    """Lp-radial distribution: x = loc + R u, R ~ norm_distribution, u uniform on the unit Lp sphere, p in {1, 2, inf}
    (distributions.py:327-372).  log_prob(x) = log f_R(||x - loc||_p) - log dV_p^d/dr (:501-549)."""

    def __init__(self, loc: torch.Tensor, norm_distribution: _RadiusDistribution, p: float, n_batch_dims: int = 0,
                 device: str = "cpu"):
        super().__init__()
        if not isinstance(p, float):
            raise ValueError("p must be a float.")
        if p <= 0:
            raise ValueError("p must be positive.")
        if p not in (1.0, 2.0, math.inf):
            raise ValueError(f"p={p} not implemented. Use p=1,2, or infinity")
        if n_batch_dims != 0:
            raise NotImplementedError("usflows_b200.RadialDistribution: n_batch_dims > 0 is not built")
        if isinstance(norm_distribution, torch.distributions.Distribution):
            norm_distribution = _wrap_torch_radius(norm_distribution)
        self.norm_distribution = norm_distribution
        self.event_shape = loc.shape[n_batch_dims:]
        self.batch_shape = loc.shape[:n_batch_dims]
        self.device = device
        self.loc = Parameter(loc.to(device))
        self.p = p
        self.n_batch_dims = n_batch_dims
        self.dim = int(math.prod(loc.shape[n_batch_dims:]))
        self.shape = loc.shape
        self.to(device)

    @property
    def _p_kind(self) -> int:
        return ops.LP_1 if self.p == 1.0 else ops.LP_2 if self.p == 2.0 else ops.LP_INF

    @staticmethod
    def _dv_const(p: float, d: int) -> float:
        if p == 1.0:             # (2r)^(d-1) 2 / (d-1)!   as written at :527-531
            return math.log(2) * d - sum(math.log(i) for i in range(1, d))
        if p == 2.0:             # d pi^(d/2) r^(d-1) / Gamma(d/2 + 1)
            return math.log(d) + (d / 2) * math.log(math.pi) - math.lgamma(d / 2 + 1)
        if p == math.inf:
            return math.log(d) + d * math.log(2)
        raise ValueError(f"p={p} not implemented. Use p=1,2, or infinity")

    def log_delta_volume_const(self) -> float:
        """r-independent part of log dV_p^d/dr (distributions.py:514-549): the full value is this + (d - 1) log r."""
        return self._dv_const(self.p, self.dim)

    def log_delta_volume(self, p: float, r):
        """log dV_p^d/dr at radius r (distributions.py:514-549): the constant above + (d - 1) log r."""
        return self._dv_const(float(p), self.dim) + (self.dim - 1) * torch.log(torch.as_tensor(r))

    def _prepared(self):
        ops.require_cuda(self.loc, "base_distribution.loc")
        kind, K, params = self.norm_distribution._norm_params()
        key = (self.loc.data_ptr(), self.loc._version)
        if getattr(self, "_loc_key", None) != key:
            self._loc_flat, self._loc_key = self.loc.detach().reshape(-1).contiguous(), key
        return self._loc_flat, kind, K, params

    def _density_into(self, z: "ops.Act", add_const: float, out: torch.Tensor, perm: Optional[torch.Tensor] = None) -> None:
        loc, kind, K, params = self._prepared()
        if perm is not None:                         # the Lp norm does not depend on the element order; loc does
            key = (self._loc_key, perm.data_ptr())
            if getattr(self, "_perm_key", None) != key:
                self._perm_loc, self._perm_key = loc[perm].contiguous(), key
            loc = self._perm_loc
        ops.radial_logprob(z, loc, self._p_kind, kind, params, K, self.log_delta_volume_const(), add_const, out)

    def _sample_into(self, out: torch.Tensor, draw: "ops.Draw") -> None:
        loc, kind, K, params = self._prepared()
        if draw.plain:
            ops.radial_sample(out, loc, self._p_kind, kind, params, K, draw.seed, draw.offset)
        else:
            ops.radial_sample_at(out, loc, self._p_kind, kind, params, K, draw)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.log_prob(x)

    def log_prob(self, x: torch.Tensor) -> torch.Tensor:
        from . import engine
        return engine.base_log_prob(self, x)

    def sample(self, sample_shape: Optional[Iterable[int]] = None) -> torch.Tensor:
        from . import engine
        if sample_shape is None:                     # the reference peels the sample dim again in this case (:480-497)
            return engine.base_sample(self, [1]).squeeze(0)
        return engine.base_sample(self, sample_shape)
