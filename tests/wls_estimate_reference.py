"""Host reference of the WLS state estimator (dss2.estimation), test infrastructure only: it minimises the ORACLE's `wls_loss`
(lam_reg = 0) of one scenario in fp64 by Gauss-Newton, with the Jacobian of a residual vector built on the oracle's `get_pflow` taken by
torch autograd and each step solved as a dense least-squares problem.  It shares nothing with the kernel's hand-derived partials, its
gain-matrix pattern or its block LU.  Classical weighting = lam_v = lam_p = N, lam_pf = E in wls_loss (w = 1 after its means)."""
import numpy as np
import torch

import dss2_oracle as orc


def weights(N, E, reg_coefs=None):
    """(lam_v, lam_p, lam_pf) of wls_loss for one scenario: classical WLS (None) or the loss's own coefficients."""
    if reg_coefs is None:
        return float(N), float(N), float(E)
    return float(reg_coefs["lam_v"]), float(reg_coefs["lam_p"]), float(reg_coefs["lam_pf"])


def loss_coefs(N, E, reg_coefs=None):
    lv, lp, lpf = weights(N, E, reg_coefs)
    return {"lam_v": lv, "lam_p": lp, "lam_pf": lpf, "lam_reg": 0.0, "mu_v": 0.0, "mu_theta": 0.0}


def residuals(x, ea, ei, stats, reg_coefs=None):
    """r(V, th) for one scenario (fp64 tensors): sqrt(lam / N * R) (Z - h) over the bus measurements (V, th, p, q), then
    sqrt(lam_pf / E * R') (Z' - h') over the branch measurements, the terms of wls_loss in its own formulas; sum(r^2) = wls_loss."""
    N, E = x.shape[0], ea.shape[0]
    xm, xs, em, es = stats
    feat, node_param, efeat, edge_param = x[:, :8], x[:, 8:], ea[:, :6], ea[:, 6:]
    z, r, ez, er = feat[:, 0::2], feat[:, 1::2], efeat[:, 0:4:2], efeat[:, 1:4:2]
    meas = (z * xs[0::2] + xm[0::2]) * (z != 0)
    wgt = (r * xs[1::2] + xm[1::2]) * (r != 0)
    emeas = (ez * es[0:4:2] + em[0:4:2]) * (ez != 0)
    ewgt = (er * es[1:4:2] + em[1:4:2]) * (er != 0)
    lv, lp, lpf = weights(N, E, reg_coefs)
    sw = torch.sqrt(wgt * torch.tensor([lv, lv, lp, lp], dtype=x.dtype) / N)
    swe = torch.sqrt(ewgt * lpf / E)
    keep = 1.0 - node_param[:, 1]

    def fn(v, th):
        th = th * keep
        _, _, pf, qf, pt, qt, _, _ = orc.get_pflow(torch.stack([v, th], 1), ei, node_param, edge_param)
        p = -orc.segment_sum(pt, ei[1], N) - orc.segment_sum(pf, ei[0], N)
        q = -orc.segment_sum(qt, ei[1], N) - orc.segment_sum(qf, ei[0], N)
        h = torch.stack([v, th, p, q], 1)
        return torch.cat([(sw * (meas - h)).reshape(-1), (swe * (emeas - torch.stack([pf, qf], 1))).reshape(-1)])
    return fn


def estimate(x, ea, ei, stats, reg_coefs=None, tol=1e-10, max_iter=30):
    """Gauss-Newton from a flat start for one scenario, each step halved until the objective does not grow: x [N,11], ea [E,13], ei [2,E] local, stats = (x_mean, x_std, edge_mean, edge_std).
    Returns (V [N], th [N], iterations, converged) as numpy fp64; th at the slack is 0."""
    x, ea = torch.as_tensor(x).double(), torch.as_tensor(ea).double()
    ei = torch.as_tensor(ei).long()
    stats = [torch.as_tensor(s).double() for s in stats]
    N = x.shape[0]
    fn = residuals(x, ea, ei, stats, reg_coefs)
    free = (x[:, 9] != 1.0).numpy()
    v, th = torch.ones(N, dtype=torch.float64), torch.zeros(N, dtype=torch.float64)
    j = float((fn(v, th) ** 2).sum())
    for it in range(1, max_iter + 1):
        jv, jt = torch.autograd.functional.jacobian(fn, (v, th))
        J = torch.cat([jt[:, free], jv], 1).numpy()
        step = np.linalg.lstsq(J, -fn(v, th).numpy(), rcond=None)[0]
        dth = np.zeros(N)
        dth[free] = step[:free.sum()]
        dth, dv = torch.from_numpy(dth), torch.from_numpy(step[free.sum():])
        # the step halved until the objective does not grow (plain Gauss-Newton can diverge from the flat start)
        for h in range(40):
            a = 0.5 ** h
            jn = float((fn(v + a * dv, th + a * dth) ** 2).sum())
            if jn <= j + 1e-12 * j:
                break
        else:
            return v.numpy(), th.numpy(), it, False
        v, th, j = v + a * dv, th + a * dth, jn
        if np.abs(step).max() <= tol:
            return v.numpy(), th.numpy(), it, True
    return v.numpy(), th.numpy(), max_iter, False


def loss(x, ea, ei, stats, vm, va, reg_coefs=None, dtype=torch.float64, grad=False):
    """The oracle's wls_loss (lam_reg = 0) of one scenario at the state (vm, va), with the model output (V - x_mean0) / x_std0;
    with grad=True also its gradient w.r.t. that output."""
    x, ea = torch.as_tensor(x).to(dtype), torch.as_tensor(ea).to(dtype)
    stats = [torch.as_tensor(s).to(dtype) for s in stats]
    out = torch.stack([(torch.as_tensor(vm).to(dtype) - stats[0][0]) / stats[1][0], torch.as_tensor(va).to(dtype)], 1)
    out.requires_grad_(grad)
    l = orc.wls_loss(x, ea, out, *stats, torch.as_tensor(ei).long(), loss_coefs(x.shape[0], ea.shape[0], reg_coefs))
    if not grad:
        return float(l)
    l.backward()
    return float(l), out.grad
