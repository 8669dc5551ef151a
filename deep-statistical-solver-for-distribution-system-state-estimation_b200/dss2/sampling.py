"""Synthetic scenario sampler of the reference's offline generator (scope row 8f-3): the 24-hour load / generation profiles and the
Monte-Carlo perturbation of `toy_network.py:83-126` with the samplers of `loadsampling.py:75-107`, evaluated by two CUDA kernels
(`dss2_load_profiles`, `dss2_mc_sample`, csrc/dataset.cu).  The power-flow solve that turns the sampled loads into labels (pandapower
`runpp`, toy_network.py:160-250) is `dss2.powerflow` (the reference's pi-model, on the device): sum the samples into bus injections and
call `powerflow.solved_scenarios` (INTEGRATION.md 2).

Random draws: by default they are taken from numpy's legacy global stream exactly like the reference's `np.random.rand` /
`np.random.normal` calls (row-major over the Monte-Carlo matrix), so after `np.random.seed(s)` the samples equal the reference's bit for
bit; `draws=` accepts a device tensor instead (e.g. torch.randn on the GPU for the 1 M-scenario case)."""
import numpy as np
import torch

from . import _lib

# toy_network.py:83-88
HOUSEHOLD = (0.25, 0.2, 0.2, 0.2, 0.2, 0.25, 0.4, 0.65, 0.65, 0.65, 0.7, 0.6, 0.7, 0.65, 0.55, 0.5, 0.45, 0.6, 0.8, 0.9, 0.8, 0.7, 0.55, 0.3)
INDUSTRY = (0.35, 0.35, 0.3, 0.3, 0.4, 0.5, 0.6, 0.9, 1., 1., 1., 0.9, 0.85, 0.85, 0.85, 0.85, 0.8, 0.55, 0.5, 0.45, 0.4, 0.4, 0.35, 0.35)
SUN = (0., 0., 0., 0., 0., 0., 0.1, 0.25, 0.4, 0.7, 0.9, 1., 1., 1.0, 1.0, 1.0, 0.9, 0.8, 0.6, 0.4, 0.3, 0.1, 0., 0.)
WIND = (0.6, 0.6, 0.7, 0.5, 0.4, 0.4, 0.5, 0.7, 0.8, 0.7, 0.5, 0.5, 0.4, 0.5, 0.4, 0.5, 0.6, 0.6, 0.3, 0.4, 0.7, 0.6, 0.4, 0.5)
DIST = {"uniform": 0, "normal": 1}


def _f64(a, device):
    return torch.as_tensor(np.asarray(a, dtype=np.float64) if not torch.is_tensor(a) else a, dtype=torch.float64, device=device).contiguous()


def mc_sample(arg_a, arg_b, numbersamples, dist, draws=None, device="cuda"):
    """dist='uniform': arg_a + rand * (arg_b - arg_a) (samplermontecarlo(LB, UB, n), loadsampling.py:75-93); dist='normal':
    arg_a + arg_b * gauss (samplermontecarlo_normal(MU, SIG, n), loadsampling.py:94-107).  Returns a float64 CUDA tensor [U, n]."""
    if dist not in DIST:
        raise NotImplementedError(f"mc_sample: dist={dist!r}; the reference's runnable choices are 'normal' and 'uniform'")
    if not torch.cuda.is_available():
        raise _lib.Dss2Error("dss2: no CUDA device; this package has no CPU fallback")
    lib = _lib.load()
    a, b = _f64(arg_a, device).reshape(-1), _f64(arg_b, device).reshape(-1)
    u = a.numel()
    assert b.numel() == u
    if draws is None:   # the reference's stream: np.random.rand(U, n) / np.random.normal(size=(U, n)) on the legacy global generator
        draws = np.random.rand(u, numbersamples) if dist == "uniform" else np.random.standard_normal((u, numbersamples))
    draws = _f64(draws, device)
    assert draws.numel() == u * numbersamples
    out = torch.empty(u, numbersamples, dtype=torch.float64, device=device)
    with torch.cuda.device(out.device):
        _lib.check(lib.dss2_mc_sample(_lib.ptr(a), _lib.ptr(b), u, numbersamples, DIST[dist], _lib.ptr(draws), _lib.ptr(out), _lib.stream()),
                   "dss2_mc_sample")
    return out


def sample_profiles(base, weight_a, weight_b, profile_a, profile_b, iterations, dist="normal", spread=0.15, draws=None, device="cuda"):
    """mu[l,h] = weight_a[l]*(base[l]*profile_a[h]) + weight_b[l]*(base[l]*profile_b[h]) (toy_network.py:106-107) perturbed `iterations`
    times per (l,h).  dist='normal': N(mu, mu*spread) (LOAD_DIST default, spread = PM_NOISE / SGEN_NOISE, toy_network.py:122-123);
    dist='uniform': U(mu(1-spread), mu(1+spread)) (spread = PM_ERROR / SGEN_ERROR, :119-120).  Returns a float64 CUDA tensor
    [L, H*iterations] in the reference's layout (toy_network.py:129).  'kumaraswamy' is not offered: the reference's own call passes 3 of
    the sampler's 6 arguments (toy_network.py:125 vs loadsampling.py:108) and cannot run."""
    if dist not in DIST:
        raise NotImplementedError(f"sample_profiles: dist={dist!r}; the reference's runnable choices are 'normal' and 'uniform'")
    if not torch.cuda.is_available():
        raise _lib.Dss2Error("dss2: no CUDA device; this package has no CPU fallback")
    lib = _lib.load()
    base, wa, wb, pa, pb = (_f64(t, device) for t in (base, weight_a, weight_b, profile_a, profile_b))
    L, H = base.numel(), pa.numel()
    assert wa.numel() == L and wb.numel() == L and pb.numel() == H
    a, b = torch.empty(L * H, dtype=torch.float64, device=device), torch.empty(L * H, dtype=torch.float64, device=device)
    with torch.cuda.device(a.device):
        _lib.check(lib.dss2_load_profiles(_lib.ptr(base), _lib.ptr(wa), _lib.ptr(wb), _lib.ptr(pa), _lib.ptr(pb), L, H, DIST[dist], float(spread),
                                          _lib.ptr(a), _lib.ptr(b), _lib.stream()), "dss2_load_profiles")
    return mc_sample(a, b, iterations, dist, draws, device).reshape(L, H * iterations)


def sample_loads(p_mw, household_mask, industry_mask, iterations, dist="normal", spread=0.15, draws=None, device="cuda"):
    """Active-power loads of toy_network.py:106 (residential + LV loads follow the household profile, commercial/industrial + MV loads the
    industry profile); reactive power is POWER_COEF times the result (toy_network.py:135)."""
    return sample_profiles(p_mw, household_mask, industry_mask, HOUSEHOLD, INDUSTRY, iterations, dist, spread, draws, device)


def sample_sgen(p_mw, sun_mask, wind_mask, iterations, dist="normal", spread=0.125, draws=None, device="cuda"):
    """Static generation of toy_network.py:107 (PV + 'Static' units follow the sun profile, wind units the wind profile)."""
    return sample_profiles(p_mw, sun_mask, wind_mask, SUN, WIND, iterations, dist, spread, draws, device)
