"""CPU reference for the batched AC power flow (dss2.powerflow) - TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A plain dense fp64 Newton-Raphson (numpy) on the reference's pi-model, independent of the kernel's sparse block formulation: the
Jacobian comes from the complex derivatives dS/dtheta, dS/dV and is solved densely.  tests/test_powerflow.py holds it to pandapower's
CIGRE-14 labels and to synthetic states, and compares the kernel's iteration counts with it; tools/powerflow_bench.py runs it as the
host baseline.  The product package never imports it.
"""
import numpy as np
def powerflow_nr(bus_param, edge_param, p_mw, q_mvar, v_slack=1.03, tol_mva=1e-8, max_iter=10):
    """Plain dense Newton-Raphson in polar form, float64, one scenario at a time.  bus_param [N,3] (vn_kv, slack, zero_inj),
    edge_param [E_all,9]; p_mw, q_mvar [S,N] load-positive (data.py:428-429), the slack's entries ignored; v_slack float or [S].

    Y from the closed edges with the pi-model of data.py:370-376 (phase shift ignored): Y_ff, Y_tt += y + ys/2, Y_ft, Y_tf -= y.
    S_calc = V_lv^2 U conj(Y U) with V_lv = min(vn_kv); mismatch S_calc + (p + j q) over the PQ buses.  Flat start (V = 1, theta = 0,
    the slack at (v_slack, 0)).  `iterations` counts the Newton updates applied: convergence (max |mismatch| <= tol_mva) is tested
    before each update, and max_iter updates without it, or a singular Jacobian, give converged = False.
    Returns numpy vm, va [S,N], iterations [S] int, converged [S] bool, max_mismatch_mva [S]."""
    bus, edge = np.asarray(bus_param, dtype=np.float64), np.asarray(edge_param, dtype=np.float64)
    p_mw, q_mvar = np.atleast_2d(np.asarray(p_mw, dtype=np.float64)), np.atleast_2d(np.asarray(q_mvar, dtype=np.float64))
    S, N = p_mw.shape
    slack = np.nonzero(bus[:, 1] == 1.0)[0]
    assert slack.size == 1, "one slack bus"
    slack = int(slack[0])
    pq = np.array([i for i in range(N) if i != slack])
    Y = np.zeros((N, N), dtype=np.complex128)
    for e in edge[edge[:, 6] == 1.0]:
        f, t = int(e[0]), int(e[1])
        y, ys = e[2] + 1j * e[3], e[4] + 1j * e[5]
        Y[f, f] += y + ys / 2
        Y[t, t] += y + ys / 2
        Y[f, t] -= y
        Y[t, f] -= y
    Y *= bus[:, 0].min() ** 2
    vs = np.broadcast_to(np.asarray(v_slack, dtype=np.float64), (S,))
    vm, va = np.ones((S, N)), np.zeros((S, N))
    its, conv, mism = np.zeros(S, dtype=np.int64), np.zeros(S, dtype=bool), np.zeros(S)
    n = pq.size
    for s in range(S):
        V, th = np.ones(N), np.zeros(N)
        V[slack] = vs[s]
        s_spec = -(p_mw[s] + 1j * q_mvar[s])
        for it in range(max_iter + 1):
            U = V * np.exp(1j * th)
            I = Y @ U
            mis = (U * np.conj(I) - s_spec)[pq]
            F = np.r_[mis.real, mis.imag]
            mism[s] = np.abs(F).max()
            its[s] = it
            if mism[s] <= tol_mva:
                conv[s] = True
                break
            if it == max_iter:
                break
            dS_dth = 1j * np.diag(U) @ np.conj(np.diag(I) - Y @ np.diag(U))
            dS_dV = np.diag(U) @ np.conj(Y @ np.diag(U / V)) + np.diag(U / V) @ np.conj(np.diag(I))
            J = np.block([[dS_dth.real[np.ix_(pq, pq)], dS_dV.real[np.ix_(pq, pq)]],
                          [dS_dth.imag[np.ix_(pq, pq)], dS_dV.imag[np.ix_(pq, pq)]]])
            try:
                dx = np.linalg.solve(J, -F)
            except np.linalg.LinAlgError:
                break
            th[pq] += dx[:n]
            V[pq] += dx[n:]
        vm[s], va[s] = V, th
    return vm, va, its, conv, mism
