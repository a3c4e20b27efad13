"""ORACLE (test infrastructure, not product code): numpy twin of the
primal-dual interior-point method the CUDA kernel implements.

It restates, for the NLP  min f(x,p) s.t. lbg <= g(x,p) <= ubg  (no bounds on
x, exactly what the reference passes to CasADi at problem.py:113), the published
IPOPT algorithm (Waechter & Biegler, Math. Prog. 106, 2006) with the option
values the reference selects (problem.py:57-60: tol=1e-3,
warm_start_init_point=yes) and IPOPT's documented defaults:

  * slack formulation g(x)-s=0, log barrier on the slack bounds (eq. 3)
  * monotone barrier update mu+ = max(min(tol,compl_inf_tol)/11, min(0.2 mu, mu^1.5)), barrier
    stop test E_mu <= 10 mu, tau = max(0.99, 1-mu)          (eq. 7, 8)
  * optimality error E_mu with s_d, s_c scaling, s_max=100  (eq. 5, 6)
  * condensed Newton system, inertia correction by delta_w escalation
    (1e-4, x100 first time, x8 after, /3 decay)             (sec. 3.1, alg. IC)
  * fraction-to-boundary, filter line search with switching/Armijo
    conditions (gamma_theta=1e-5, gamma_phi=1e-8, eta_phi=1e-8, s_theta=1.1,
    s_phi=2.3, delta=1)                                      (sec. 2.3, alg. A)
  * gradient-based scaling (nlp_scaling_max_gradient=100), bound relaxation
    1e-8, warm-start pushes 1e-3, multiplier safeguard kappa_Sigma=1e10.

Deviations from IPOPT (documented in DESIGN.md): no second-order correction,
no restoration phase (a feasibility restart -- slacks re-centred, multipliers
and filter reset, mu = 1 -- is tried up to 5 times, then Restoration_Failed), inertia is checked on the
condensed matrix H = W + J_d^T Sigma J_d (Cholesky) instead of the full
augmented system.  parity unpinned: no IPOPT binary is available here.

The C restatement oracle/ipm.c follows this file statement by statement.
"""
import numpy as np

from .nlp_eval import TableEval

STATUS = {0: 'Solve_Succeeded', 1: 'Maximum_Iterations_Exceeded',
          2: 'Restoration_Failed', 3: 'Error_In_Step_Computation',
          4: 'Invalid_Number_Detected', 5: 'Infeasible_Problem_Detected'}

DEFAULTS = dict(
    tol=1e-3, max_iter=3000, mu_init=0.1, constr_viol_tol=1e-4,
    dual_inf_tol=1.0, compl_inf_tol=1e-4, bound_push=1e-3, bound_frac=1e-3,
    mult_bound_push=1e-3, bound_relax_factor=1e-8, scaling_max_gradient=100.0,
    kappa_eps=10.0, kappa_mu=0.2, theta_mu=1.5, tau_min=0.99, s_max=100.0,
    kappa_sigma=1e10, gamma_theta=1e-5, gamma_phi=1e-8, eta_phi=1e-8,
    s_theta=1.1, s_phi=2.3, delta=1.0, gamma_alpha=0.05, theta_max_fact=1e4,
    theta_min_fact=1e-4, delta_w0=1e-4, delta_w_min=1e-20, delta_w_max=1e40,
    kappa_w_plus_first=100.0, kappa_w_plus=8.0, kappa_w_minus=1.0 / 3.0,
    delta_c_val=1e-8, delta_c_exp=0.25, piv_tol=1e-12, inf_bound=1e19,
    soft_resto_factor=0.9999, soft_resto=1, max_filter=32, max_ls=40,
    max_restarts=5, restart_mu=1.0, restart_push=1e-1, inertia_mode=0)

EPS = np.finfo(float).eps


def _cmp_le(lhs, rhs, base):
    return lhs - rhs <= 10.0 * EPS * abs(base)


class Result(object):
    pass


def solve(tb, x0, p, lbg=None, ubg=None, options=None, lam_g0=None,
          trace=False):
    o = dict(DEFAULTS)
    o.update(options or {})
    ev = TableEval(tb)
    n, m = tb.n, tb.m
    lbg = tb.lbg if lbg is None else np.asarray(lbg, dtype=float)
    ubg = tb.ubg if ubg is None else np.asarray(ubg, dtype=float)
    V = ev.tape(p)
    x = np.array(x0, dtype=float)

    big = o['inf_bound']
    is_eq = (lbg == ubg)
    hasL = (lbg > -big) & ~is_eq
    hasU = (ubg < big) & ~is_eq
    ineq = ~is_eq
    eq_idx = np.nonzero(is_eq)[0]
    n_eq = len(eq_idx)
    if n_eq != tb.kkt_n_eq or np.any(eq_idx != tb.kkt_eq_rows):
        res = Result()           # equality pattern differs from the structure
        res.x, res.lam_g, res.f = x, np.zeros(m), 0.0
        res.status, res.return_status, res.iters, res.mu, res.log = \
            3, STATUS[3], 0, o['mu_init'], []
        return res
    kperm = np.argsort(np.r_[tb.kkt_pos_var, tb.kkt_pos_eq])
    ksign = tb.kkt_sign.astype(float)

    # ---- gradient-based scaling at x0 ---------------------------------
    jv = np.abs(ev.jac_vals(x, V))
    gmax = np.zeros(m)
    np.maximum.at(gmax, tb.jrow, jv)
    smg = o['scaling_max_gradient']
    dsc = np.where(gmax > smg, np.maximum(smg / np.maximum(gmax, 1e-300), 1e-8), 1.0)
    fmax = np.abs(ev.gradf(x, V)).max() if n else 0.0
    fsc = max(smg / fmax, 1e-8) if fmax > smg else 1.0

    sL = np.where(hasL, lbg * dsc, -np.inf)
    sU = np.where(hasU, ubg * dsc, np.inf)
    beq = lbg * dsc
    brf = o['bound_relax_factor']
    sL = np.where(hasL, sL - brf * np.maximum(1.0, np.abs(sL)), sL)
    sU = np.where(hasU, sU + brf * np.maximum(1.0, np.abs(sU)), sU)

    def evaluate(xx):
        return fsc * ev.f(xx, V), dsc * ev.g(xx, V)

    # ---- starting point ---------------------------------------------------
    f, g = evaluate(x)
    s = g.copy()
    k1, k2 = o['bound_push'], o['bound_frac']
    both = hasL & hasU
    pL = np.where(both, np.minimum(k1 * np.maximum(1, np.abs(sL)), k2 * (sU - sL)),
                  k1 * np.maximum(1, np.abs(sL)))
    pU = np.where(both, np.minimum(k1 * np.maximum(1, np.abs(sU)), k2 * (sU - sL)),
                  k1 * np.maximum(1, np.abs(sU)))
    with np.errstate(invalid='ignore'):      # -inf + inf on rows without that bound (masked)
        s = np.where(hasL, np.maximum(s, sL + pL), s)
        s = np.where(hasU, np.minimum(s, sU - pU), s)
    y = np.zeros(m)
    if lam_g0 is not None:
        y = np.asarray(lam_g0, dtype=float) * fsc / dsc
    mbp = o['mult_bound_push']
    zL = np.where(hasL, np.maximum(mbp, -y), 0.0)
    zU = np.where(hasU, np.maximum(mbp, y), 0.0)
    mu = o['mu_init']
    tau = max(o['tau_min'], 1.0 - mu)
    n_bounds = int(hasL.sum() + hasU.sum())

    filt = []
    theta_max = theta_min = None
    delta_w_last = 0.0
    n_restarts = 0
    status, it = 1, 0
    log = []

    for it in range(o['max_iter'] + 1):
        jvals = dsc[tb.jrow] * ev.jac_vals(x, V)
        J = np.zeros((m, n))
        J[tb.jrow, tb.jcol] = jvals
        gf = fsc * ev.gradf(x, V)
        dL = np.where(hasL, s - sL, 1.0)
        dU = np.where(hasU, sU - s, 1.0)
        r_x = gf + J.T.dot(y)
        r_s = np.where(ineq, -y - zL + zU, 0.0)
        c = np.where(is_eq, g - beq, np.where(ineq, g - s, 0.0))

        def err(mu_):
            dinf = max(np.abs(r_x).max(), np.abs(r_s).max() if m else 0.0)
            cinf = np.abs(c).max() if m else 0.0
            cmpl = 0.0
            if n_bounds:
                cmpl = max(np.abs(np.where(hasL, dL * zL - mu_, 0.0)).max(),
                           np.abs(np.where(hasU, dU * zU - mu_, 0.0)).max())
            zsum = zL.sum() + zU.sum()
            s_d = max(o['s_max'], (np.abs(y).sum() + zsum) / max(1, m + n_bounds)) / o['s_max']
            s_c = max(o['s_max'], zsum / max(1, n_bounds)) / o['s_max']
            return max(dinf / s_d, cinf, cmpl / s_c), dinf, cinf, cmpl

        E0, dinf, cinf, cmpl0 = err(0.0)
        # unscaled side conditions
        g_un = g / dsc
        viol = max(0.0, np.max(np.where(hasU | is_eq, g_un - ubg, 0.0)),
                   np.max(np.where(hasL | is_eq, lbg - g_un, 0.0))) if m else 0.0
        dinf_un = max(np.abs(r_x).max(), (np.abs(r_s) * dsc).max() if m else 0.0) / fsc
        if trace:
            # (iter, f, cinf, dinf, mu, E0, alpha, delta_w): the last two belong to the step
            # taken FROM this iterate and are filled in below (0.0 while there is none)
            log.append((it, f / fsc, cinf, dinf, mu, E0, 0.0, 0.0))
        if not np.isfinite(E0):
            status = 4
            break
        if (E0 <= o['tol'] and dinf_un <= o['dual_inf_tol'] and
                viol <= o['constr_viol_tol'] and cmpl0 / fsc <= o['compl_inf_tol']):
            status = 0
            break
        if it == o['max_iter']:
            status = 1
            break

        # ---- barrier parameter update ---------------------------------
        # floor as implemented by IPOPT's monotone update (IpMonotoneMuUpdate:
        # min(tol, compl_inf_tol)/(kappa_eps+1)), not the paper's tol/10
        mu_min = min(o['tol'], o['compl_inf_tol'] * fsc) / (o['kappa_eps'] + 1.0)
        while True:
            Emu = err(mu)[0]
            if Emu <= o['kappa_eps'] * mu and mu > mu_min:
                mu = max(mu_min, min(o['kappa_mu'] * mu, mu ** o['theta_mu']))
                tau = max(o['tau_min'], 1.0 - mu)
                filt = []
            else:
                break

        theta = np.abs(c).sum()
        if theta_max is None:
            theta_max = o['theta_max_fact'] * max(1.0, theta)
            theta_min = o['theta_min_fact'] * max(1.0, theta)
        phi = f - mu * (np.log(dL[hasL]).sum() + np.log(dU[hasU]).sum())

        # ---- Newton system -------------------------------------------------
        sigL = np.where(hasL, zL / dL, 0.0)
        sigU = np.where(hasU, zU / dU, 0.0)
        Sig = sigL + sigU
        phis = np.where(hasL, -mu / dL, 0.0) + np.where(hasU, mu / dU, 0.0)
        r_d = np.where(ineq, g - s, 0.0)
        W = ev.hess_dense(x, V, y * dsc, fsc)
        Jd = J * ineq[:, None]
        Jc = J[eq_idx]
        H0 = W + Jd.T.dot(Sig[:, None] * Jd)
        rhs1 = -(gf + Jc.T.dot(y[eq_idx]) + Jd.T.dot(Sig * r_d + phis))
        rhs2 = -c[eq_idx]

        delta_w, delta_c = 0.0, 0.0
        first_try = True
        sol = None
        while True:
            K = np.zeros((n + n_eq, n + n_eq))
            K[:n, :n] = H0 + delta_w * np.eye(n)
            K[n:, :n] = Jc
            K[:n, n:] = Jc.T
            K[n:, n:] = -delta_c * np.eye(n_eq)
            # symmetric permutation of lowering.build_kkt_structure: equality
            # rows interleaved, K = L S L^T with S = diag(kkt_sign)
            ok, L, eq_fail, S_piv = _signed_cholesky(K[np.ix_(kperm, kperm)], ksign,
                                                     o['piv_tol'], o['inertia_mode'])
            if ok:
                sol = np.empty(n + n_eq)
                sol[kperm] = _signed_solve(L, S_piv, np.r_[rhs1, rhs2][kperm])
                break
            if eq_fail:
                delta_c = o['delta_c_val'] * mu ** o['delta_c_exp']
            if first_try:
                delta_w = o['delta_w0'] if delta_w_last == 0.0 else \
                    max(o['delta_w_min'], o['kappa_w_minus'] * delta_w_last)
                first_try = False
            else:
                delta_w *= o['kappa_w_plus_first'] if delta_w_last == 0.0 \
                    else o['kappa_w_plus']
            if delta_w > o['delta_w_max']:
                break
        if sol is None:
            status = 3
            break
        if delta_w > 0.0:
            delta_w_last = delta_w
        dx, dyc = sol[:n], sol[n:]
        ds = np.where(ineq, J.dot(dx) + r_d, 0.0)
        dy = np.where(ineq, Sig * ds + phis - y, 0.0)
        dy[eq_idx] = dyc
        dzL = np.where(hasL, mu / dL - zL - sigL * ds, 0.0)
        dzU = np.where(hasU, mu / dU - zU + sigU * ds, 0.0)

        # ---- fraction to the boundary -------------------------------------
        def max_step(val, dval, mask):
            sel = mask & (dval < 0.0)
            if not sel.any():
                return 1.0
            return min(1.0, np.min(-tau * val[sel] / dval[sel]))
        a_p = min(max_step(dL, ds, hasL), max_step(dU, -ds, hasU))
        a_d = min(max_step(zL, dzL, hasL), max_step(zU, dzU, hasU))

        # ---- filter line search --------------------------------------------
        gphi = gf.dot(dx) + phis.dot(ds)
        if gphi < 0.0:
            a_min = min(o['gamma_theta'], o['gamma_phi'] * theta / (-gphi))
            if theta <= theta_min:
                a_min = min(a_min, o['delta'] * theta ** o['s_theta'] /
                            (-gphi) ** o['s_phi'])
        else:
            a_min = o['gamma_theta']
        a_min *= o['gamma_alpha']

        def trial(alpha):
            xt, st = x + alpha * dx, s + alpha * ds
            ft, gt = evaluate(xt)
            ct = np.where(is_eq, gt - beq, np.where(ineq, gt - st, 0.0))
            dLt = np.where(hasL, st - sL, 1.0)
            dUt = np.where(hasU, sU - st, 1.0)
            pht = ft - mu * (np.log(dLt[hasL]).sum() + np.log(dUt[hasU]).sum())
            return xt, st, ft, gt, np.abs(ct).sum(), pht

        alpha = a_p
        accepted = False
        n_ls = 0
        while alpha >= a_min and n_ls < o['max_ls']:
            n_ls += 1
            xt, st, ft, gt, tht, pht = trial(alpha)
            ok = np.isfinite(pht) and np.isfinite(tht) and tht <= theta_max
            if ok:
                for (tf_, pf_) in filt:
                    if not (tht < tf_ or pht < pf_):
                        ok = False
                        break
            ftype = False
            if ok:
                switching = (theta <= theta_min and gphi < 0.0 and
                             alpha * (-gphi) ** o['s_phi'] >
                             o['delta'] * theta ** o['s_theta'])
                if switching:
                    ok = _cmp_le(pht - phi, o['eta_phi'] * alpha * gphi, phi)
                    ftype = ok
                else:
                    ok = (_cmp_le(tht, (1.0 - o['gamma_theta']) * theta, theta) or
                          _cmp_le(pht - phi, -o['gamma_phi'] * theta, phi))
            if ok:
                accepted = True
                if not ftype:
                    _filter_add(filt, (1.0 - o['gamma_theta']) * theta,
                                phi - o['gamma_phi'] * theta, o['max_filter'])
                break
            alpha *= 0.5

        if not accepted and o['soft_resto']:
            # soft restoration: accept a step that reduces the primal-dual error
            pd0 = _pd_error(r_x, r_s, c, dL, zL, dU, zU, hasL, hasU, mu)
            alpha = a_p
            n_try = 0
            while n_try < 12:
                n_try += 1
                xt, st, ft, gt, tht, pht = trial(alpha)
                yt = y + alpha * dy
                zLt = zL + min(alpha, a_d) * dzL
                zUt = zU + min(alpha, a_d) * dzU
                Jt = np.zeros((m, n))
                Jt[tb.jrow, tb.jcol] = dsc[tb.jrow] * ev.jac_vals(xt, V)
                rxt = fsc * ev.gradf(xt, V) + Jt.T.dot(yt)
                rst = np.where(ineq, -yt - zLt + zUt, 0.0)
                ct = np.where(is_eq, gt - beq, np.where(ineq, gt - st, 0.0))
                pdt = _pd_error(rxt, rst, ct, np.where(hasL, st - sL, 1.0), zLt,
                                np.where(hasU, sU - st, 1.0), zUt, hasL, hasU, mu)
                if np.isfinite(pdt) and pdt <= o['soft_resto_factor'] * pd0:
                    accepted = True
                    filt = []
                    break
                alpha *= 0.5
        if trace:
            log[-1] = log[-1][:6] + (alpha if accepted else 0.0, delta_w)
        if not accepted:
            if n_restarts < o['max_restarts']:
                # feasibility restart (stand-in for IPOPT's restoration phase): keep x,
                # re-centre the slacks, forget the multipliers and the filter, and
                # continue from a large barrier parameter
                n_restarts += 1
                mu = o['restart_mu']
                tau = max(o['tau_min'], 1.0 - mu)
                kp = o['restart_push']
                s = g.copy()
                s = np.where(hasL, np.maximum(s, sL + kp * np.maximum(1, np.abs(sL))), s)
                s = np.where(hasU, np.minimum(s, sU - kp * np.maximum(1, np.abs(sU))), s)
                y = np.zeros(m)
                zL = np.where(hasL, mu / np.where(hasL, s - sL, 1.0), 0.0)
                zU = np.where(hasU, mu / np.where(hasU, sU - s, 1.0), 0.0)
                filt = []
                theta_max = None
                delta_w_last = 0.0
                continue
            status = 2
            break

        # ---- accept ---------------------------------------------------------
        x, s, f, g = xt, st, ft, gt
        y = y + alpha * dy
        zL = zL + a_d * dzL
        zU = zU + a_d * dzU
        ks = o['kappa_sigma']
        dLn = np.where(hasL, s - sL, 1.0)
        dUn = np.where(hasU, sU - s, 1.0)
        zL = np.where(hasL, np.clip(zL, mu / (ks * dLn), ks * mu / dLn), 0.0)
        zU = np.where(hasU, np.clip(zU, mu / (ks * dUn), ks * mu / dUn), 0.0)

    res = Result()
    res.x = x
    res.lam_g = y * dsc / fsc
    res.f = f / fsc
    res.status = status
    res.return_status = STATUS[status]
    res.iters = it
    res.mu = mu
    res.log = log
    return res


def _pd_error(r_x, r_s, c, dL, zL, dU, zU, hasL, hasU, mu):
    return (np.abs(r_x).sum() + np.abs(r_s).sum() + np.abs(c).sum() +
            np.abs(np.where(hasL, dL * zL - mu, 0.0)).sum() +
            np.abs(np.where(hasU, dU * zU - mu, 0.0)).sum())


def _filter_add(filt, th, ph, cap):
    filt[:] = [(t, p) for (t, p) in filt if not (t >= th and p >= ph)]
    if len(filt) >= cap:
        filt.pop(0)
    filt.append((th, ph))


def _signed_cholesky(K, sign, piv_tol, mode=0):
    """K = L S L^T in the permuted order, lower-triangular L.

    mode 0 (IPOPT's inertia test): S[j] is the sign of pivot j as it comes and the
    factorisation is accepted when the NUMBER of negative pivots equals the number
    of equality rows (Sylvester's law of inertia).  mode 1: S fixed to ``sign``
    (+1 variables, -1 equality rows); a pivot of the other sign fails -- stricter
    than necessary, it over-regularises problems with non-convex constraints.
    Returns (ok, L, regularise_constraint_block, S)."""
    N = K.shape[0]
    A = np.tril(K).copy()
    d0 = np.abs(np.diag(K)).copy()
    S = np.zeros(N)
    n_neg = int((np.asarray(sign) < 0).sum())
    for j in range(N):
        if mode:
            sgn = float(sign[j])
        else:
            sgn = 1.0 if A[j, j] > 0 else -1.0
        piv = sgn * A[j, j]
        thr = 0.0 if (mode and sgn < 0) else piv_tol * max(d0[j], 1e-300)
        if not (piv > thr) or not np.isfinite(piv):
            return False, None, sign[j] < 0, None
        S[j] = sgn
        ljj = np.sqrt(piv)
        A[j, j] = ljj
        if j + 1 < N:
            A[j + 1:, j] = A[j + 1:, j] / (sgn * ljj)
            col = A[j + 1:, j]
            A[j + 1:, j + 1:] -= sgn * np.tril(np.outer(col, col))
    neg = int((S < 0).sum())
    if neg != n_neg:
        return False, None, neg < n_neg, None
    return True, A, False, S


def _signed_solve(L, sign, rhs):
    N = L.shape[0]
    w = np.array(rhs, dtype=float)
    for j in range(N):
        w[j] /= L[j, j]
        w[j + 1:] -= L[j + 1:, j] * w[j]
    w = w * sign
    for j in range(N - 1, -1, -1):
        w[j] /= L[j, j]
        w[:j] -= L[j, :j] * w[j]
    return w


FEAS_STEPS = 30


def feasibility_lm(tb, x0, p, lbg=None, ubg=None, max_steps=FEAS_STEPS):
    """Feasibility phase the host runs on an instance that ended in Restoration_Failed
    (stand-in for the feasibility part of IPOPT's restoration phase): Levenberg-Marquardt
    on the violation v(x) = g - clip(g, lbg, ubg),
        (Jv^T Jv + lam I) dx = -Jv^T v,   Jv = rows with v != 0,
    lam from 1e-3, /10 after an accepted step, x10 (at most 12 times) after a rejected
    one; stops when max|v| <= 1e-8.  Returns (x, max|v|, steps).  oracle/ipm.c
    (oracle_feas_batch) and the CUDA kernel omg_feas_kernel follow this function."""
    ev = TableEval(tb)
    lbg = tb.lbg if lbg is None else np.asarray(lbg, dtype=float)
    ubg = tb.ubg if ubg is None else np.asarray(ubg, dtype=float)
    V = ev.tape(p)
    x = np.array(x0, dtype=float)
    n = tb.n

    def residual(xx):
        g = ev.g(xx, V)
        v = np.where(g < lbg, g - lbg, np.where(g > ubg, g - ubg, 0.0))
        return v, 0.5 * v.dot(v), (np.abs(v).max() if len(v) else 0.0)

    v, phi, vmax = residual(x)
    lam, steps = 1e-3, 0
    while steps < max_steps and vmax > 1e-8:
        J = ev.jac_dense(x, V)
        act = v != 0.0
        A = J[act].T.dot(J[act])
        rhs = -J[act].T.dot(v[act])
        accepted = False
        for _ in range(12):
            try:
                Lc = np.linalg.cholesky(A + lam * np.eye(n))
                dx = np.linalg.solve(Lc.T, np.linalg.solve(Lc, rhs))
                vt, pt, vmt = residual(x + dx)
                ok = pt < phi
            except np.linalg.LinAlgError:
                ok = False
            if ok:
                x, v, phi, vmax = x + dx, vt, pt, vmt
                lam = max(lam / 10.0, 1e-12)
                accepted = True
                break
            lam *= 10.0
        if not accepted:
            break
        steps += 1
    return x, vmax, steps


def solve_with_feasibility(tb, x0, p, lbg=None, ubg=None, options=None, feas_steps=FEAS_STEPS):
    """What B200Solver.solve_batch does per instance: solve; on Restoration_Failed run the
    feasibility phase from the returned point and solve once more from there."""
    res = solve(tb, x0, p, lbg, ubg, options)
    if res.status == 2 and feas_steps > 0:
        x1, _, _ = feasibility_lm(tb, res.x, p, lbg, ubg, feas_steps)
        r2 = solve(tb, x1, p, lbg, ubg, options)
        r2.iters += res.iters
        return r2
    return res
