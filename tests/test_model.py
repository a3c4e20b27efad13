"""Model layer + lowering: sizes and flat layouts of the BASELINE configs
(SURVEY.md section 8 table and appendix A), table evaluation against direct
polynomial evaluation and finite differences, warm-start shift."""
import numpy as np
import pytest

from omg_tools_b200 import scenarios as sc
from omg_tools_b200.basics import poly as pl
from omg_tools_b200.basics.spline_extra import shiftoverknot_T
from oracle.nlp_eval import TableEval


@pytest.fixture(scope='module')
def cfg1():
    return sc.config1(build_solver=False)


@pytest.mark.parametrize('name,n,m,n_par', [('config1', 98, 325, 17),
                                            ('config2', 190, 563, 35),
                                            ('config5', 184, 862, 58)])
def test_problem_dimensions(name, n, m, n_par):
    pr = getattr(sc, name)(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_par) == (n, m, n_par)
    assert tb.degree == 2
    assert int((tb.lbg == tb.ubg).sum()) == 10     # 4 initial + 6 terminal rows


def test_flat_layout_config1(cfg1):
    f = cfg1.father
    names = [k[1] for k in f._var_struct.keys()]
    assert names == ['splines_seg0', 'eps_00', 'g0', 'g1',
                     'a_%s_seg0_00' % cfg1.vehicles[0].label,
                     'b_%s_seg0_00' % cfg1.vehicles[0].label]
    pnames = [k[1] for k in f._par_struct.keys()]
    assert pnames == ['state0', 'input0', 'poseT', 'x', 'v', 'a', 'checkpoints',
                      'rad', 'T', 't']
    rows = [v[1] for v in f._con_struct.entries.values()]
    assert rows == [12] * 4 + [11] * 4 + [13, 13, 41] + [13] * 4 + [31] + \
        [1] * 4 + [13] * 4 + [1] * 6 + [21]
    # cold start = linear interpolation of the vehicle spline, zeros elsewhere
    x0 = f.get_variables().cat
    assert np.allclose(x0[:13], np.linspace(-1.5, 2., 13))
    assert np.allclose(x0[13:26], np.linspace(-1.5, 2., 13))
    assert np.all(x0[26:] == 0.)
    p = f.set_parameters(0.37).cat
    assert np.allclose(p[:6], [-1.5, -1.5, 0, 0, 2, 2])
    assert np.allclose(p[-2:], [10., 0.37])


def test_tables_match_polynomials_and_derivatives(cfg1):
    f, tb = cfg1.father, cfg1.father.tables
    ev = TableEval(tb)
    rng = np.random.default_rng(3)
    x = f.get_variables().cat + 0.1 * rng.standard_normal(tb.n)
    p = f.set_parameters(0.37).cat.copy()
    V = ev.tape(p)
    vals = {pl.resolve(s): v for s, v in zip(f._var_ids, x)}
    vals.update({pl.resolve(s): v for s, v in zip(f._par_ids, p)})
    rows, _, _ = f.construct_constraints()
    direct = np.array([r.evaluate(dict(vals)) for r in rows])
    assert np.abs(ev.g(x, V) - direct).max() < 1e-12
    obj = f.construct_objective()
    assert abs(ev.f(x, V) - obj.evaluate(dict(vals))) < 1e-13
    h = 1e-6
    J = ev.jac_dense(x, V)
    lam = rng.standard_normal(tb.m)
    W = ev.hess_dense(x, V, lam)
    for j in rng.choice(tb.n, 12, replace=False):
        e = np.zeros(tb.n)
        e[j] = h
        assert np.abs((ev.g(x + e, V) - ev.g(x - e, V)) / (2 * h) - J[:, j]).max() < 1e-5
        dj = (ev.jac_dense(x + e, V).T @ lam - ev.jac_dense(x - e, V).T @ lam) / (2 * h)
        assert np.abs(dj - W[:, j]).max() < 1e-5
    g0 = ev.gradf(x, V)
    assert abs((ev.f(x + 1e-6 * g0, V) - ev.f(x, V)) / 1e-6 - g0 @ g0) < 1e-6


def test_collision_rows_are_the_pointwise_constraint(cfg1):
    """Property independent of the reference: the 41 vehicle-side rows are the
    B-spline coefficients of a(t).(x(t),y(t)) - b(t) + r + sd - eps(t)."""
    from omg_tools_b200.basics.spline import BSpline, BSplineBasis
    f, tb = cfg1.father, cfg1.father.tables
    ev = TableEval(tb)
    rng = np.random.default_rng(5)
    x = rng.standard_normal(tb.n)
    p = f.set_parameters(0.).cat
    g = ev.g(x, ev.tape(p))
    off, size, _ = f._con_struct.entries[(None, 'c_10_%s' % cfg1.vehicles[0].label)]
    assert size == 41
    veh = cfg1.vehicles[0]
    b3 = veh.basis
    b1 = BSplineBasis(np.r_[0., veh.knots[3:-3], 1.], 1)
    xs, ys, eps = (BSpline(b3, x[k * 13:(k + 1) * 13]) for k in (0, 1, 2))
    a0, a1, b = (BSpline(b1, x[65 + k * 11:65 + (k + 1) * 11]) for k in (0, 1, 2))
    con = a0 * xs + a1 * ys + (-b + 0.1 + 0.1 - eps)
    assert np.abs(con.coeffs - g[off:off + 41]).max() < 1e-11
    tt = np.linspace(0, 1, 50)
    point = a0(tt) * xs(tt) + a1(tt) * ys(tt) - b(tt) + 0.2 - eps(tt)
    assert np.abs(con(tt) - point).max() < 1e-11


def test_knot_shift_of_seg0_variables(cfg1):
    f = cfg1.father
    blocks = f.shifted_entries()
    names = [b[1] for b in blocks]
    assert names[0] == 'splines_seg0' and all('seg0' in n for n in names)
    assert not any(n.startswith('g') or n.startswith('eps') for n in names)
    rng = np.random.default_rng(2)
    before = rng.standard_normal(f.tables.n)
    f.set_variables(before)
    cfg1.initialize(0.)
    cfg1.init_step(1.0, 0.1)          # passes the first knot (knot_time = 1 s)
    after = f.get_variables().cat
    T3 = shiftoverknot_T(cfg1.vehicles[0].basis)
    assert np.allclose(after[:13], T3 @ before[:13])
    assert np.allclose(after[13:26], T3 @ before[13:26])
    assert np.array_equal(after[26:65], before[26:65])     # eps, g untouched
    f.init_variables()
    cfg1.reinitialize()


def test_rotating_obstacle_rows_config5():
    pr = sc.config5(build_solver=False)
    f = pr.father
    rows = {k[1]: v[1] for k, v in f._con_struct.entries.items()}
    lab = [o.label for o in pr.environment.obstacles]
    assert rows['c_0_' + lab[0]] == 31 and rows['c_1_' + lab[0]] == 31
    assert rows['c_0_' + lab[2]] == 71 and rows['c_1_' + lab[2]] == 71
    # theta enters through cos/sin atoms of the parameter tape
    assert 4 in f.tables.tape_func and 5 in f.tables.tape_func


def test_holonomic3d_example_dimensions_and_rows():
    """examples/p2p_holonomic_3d.py: 3 position splines, 3 terminal-objective
    slacks, 2 obstacles x (a[3], b) degree-1 hyperplanes; obstacle checkpoints
    are parameters (obstacle.py:191-193).  The collision rows must be the
    pointwise separation a.(chk + p(t)) - b + r <= 0 in coefficient form."""
    pr = sc.config_holonomic3d(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_par) == (166, 1536, 109)
    ent = pr.father._var_struct.entries
    shapes = sorted(v[2] for v in ent.values())
    assert shapes == sorted([(13, 3)] + [(13, 1)] * 3 + [(11, 3), (11, 1)] * 2)
    # 6 initial + 3 terminal position + 9 terminal derivative equalities
    assert int((tb.lbg == tb.ubg).sum()) == 18
    # tables evaluate consistently with finite differences
    rng = np.random.default_rng(0)
    X0, P = sc.instance_data(pr, 1)
    x = X0[0] + 0.1 * rng.standard_normal(tb.n)
    ev = TableEval(tb)
    v = ev.tape(P[0])
    g0 = ev.g(x, v)
    J = ev.jac_dense(x, v)
    h = 1e-6
    for k in rng.choice(tb.n, 12, replace=False):
        xp = x.copy()
        xp[k] += h
        xm = x.copy()
        xm[k] -= h
        fd = (ev.g(xp, v) - ev.g(xm, v)) / (2 * h)
        assert np.abs(fd - J[:, k]).max() < 1e-6
    assert np.isfinite(g0).all()


def test_holonomic1d_problem_solves_on_oracle():
    """Smallest member of the family (holonomic1d.py): one spline, no
    collision rows; the oracle must reach the target with zero end velocity."""
    from omg_tools_b200 import Holonomic1D, Environment, Square
    from oracle import ipm_ref
    veh = Holonomic1D()
    veh.set_initial_conditions([0.])
    veh.set_terminal_conditions([2.])
    pr = sc._p2p(veh, Environment(room={'shape': Square(10.)}), None, False)
    tb = pr.father.tables
    assert tb.n == 26          # 13 spline + 13 objective slack coefficients
    X0, P = sc.instance_data(pr, 1)
    res = ipm_ref.solve(tb, X0[0], P[0])
    assert res.status == 0
    assert abs(res.x[12] - 2.) < 1e-6 and abs(res.x[0]) < 1e-6
    # velocity bound 0.5 m/s over T=10 s: derivative coefficients within bound
    basis = veh.basis
    Bd, P1 = basis.derivative(1)
    assert (P1.dot(res.x[:13]) / 10. <= 0.5 + 1e-6).all()


class _OracleSolver(object):
    """Stand-in for the solver callable of Problem.solve() (reference
    problem.py:113) backed by the CPU oracle: lets the host loop run without a
    GPU.  Test infrastructure only."""

    def __init__(self, tb):
        from oracle import ipm_c
        self.tb, self.ipm_c = tb, ipm_c

    def __call__(self, x0, p, lbg, ubg, lam_g0=None, **kw):
        r = self.ipm_c.solve_batch_full(
            self.tb, np.asarray(x0, float)[None], np.asarray(p, float)[None], threads=1,
            lbg=np.asarray(lbg, float)[None], ubg=np.asarray(ubg, float)[None])
        self.last = r
        return {'x': r['x'][0], 'lam_g': r['lam_g'][0], 'f': r['f'][0]}

    def stats(self):
        ok = self.last['status'][0] == 0
        return {'return_status': 'Solve_Succeeded' if ok else 'Restoration_Failed',
                'iter_count': int(self.last['iters'][0])}


def test_quadrotor3d_config4_tables_and_receding_horizon():
    """BASELINE config 4 (examples/p2p_3dquadrotor.py).  Sizes as surveyed
    (n=238, m=1319), 236 shared intermediates; derivatives of the chain-rule
    tables against finite differences; then the reference's MPC loop
    (predict/init_step/solve/store/simulate, update_time 0.4 s) flies the
    quadrotor to the goal with every solve converged."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config4(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_mid, tb.degree) == (238, 1319, 236, 5)
    ev = TableEval(tb)
    rng = np.random.default_rng(1)
    X0, P = sc.instance_data(pr, 1)
    x = X0[0] + 0.05 * rng.standard_normal(tb.n)
    V = ev.tape(P[0])
    J = ev.jac_dense(x, V)
    lam = rng.standard_normal(tb.m)
    W = ev.hess_dense(x, V, lam)
    h = 1e-6
    for j in rng.choice(tb.n, 8, replace=False):
        e = np.zeros(tb.n)
        e[j] = h
        assert np.abs((ev.g(x + e, V) - ev.g(x - e, V)) / (2 * h) - J[:, j]).max() < 1e-5
        dj = (ev.jac_dense(x + e, V).T @ lam - ev.jac_dense(x - e, V).T @ lam) / (2 * h)
        assert np.abs(dj - W[:, j]).max() < 1e-5
    # rows evaluate to the model's polynomials (intermediates expanded)
    f = pr.father
    vals = {pl.resolve(s): v for s, v in zip(f._var_ids, x)}
    vals.update({pl.resolve(s): v for s, v in zip(f._par_ids, P[0])})
    rows, _, _ = f.construct_constraints()
    direct = np.array([r.evaluate(dict(vals)) if isinstance(r, pl.Poly) else float(r)
                       for r in rows])
    assert np.abs(direct - ev.g(x, V)).max() < 1e-11
    # receding horizon
    pr.problem = _OracleSolver(tb)
    pr.initialize(0.)
    t, dt = 0., 0.4
    for k in range(13):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        assert pr.problem.stats()['return_status'] == 'Solve_Succeeded', k
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t += dt
    assert np.abs(pr.vehicles[0].signals['state'][:3, -1] - [3., 2., 0.5]).max() < 1e-2


def test_freeT_point2point_receding_horizon():
    """FreeTPoint2point (reference point2point.py:269-374): T is a decision
    variable and the objective, rows are cubic.  The reference's loop
    (init_step re-expresses the remaining spline piece on a fresh basis and
    shortens T) drives the vehicle to the goal; every solve converges and the
    motion time decreases by the update time."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_freeT(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.degree) == (126, 622, 3)
    pr.problem = _OracleSolver(tb)
    pr.initialize(0.)
    t, dt = 0., 0.5
    Ts = []
    for k in range(20):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        assert pr.problem.stats()['return_status'] == 'Solve_Succeeded', k
        Ts.append(pr.horizon_time())
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t += dt
        if pr.stop_criterium(t, dt):
            break
    assert 9. < Ts[0] < 10.                      # ~7 s of travel at 0.5 m/s + acceleration
    assert np.abs(np.diff(Ts) + dt).max() < 0.15  # the plan is executed as predicted
    assert np.abs(pr.vehicles[0].signals['state'][:, -1] - [2., 2.]).max() < 1e-2


def test_freeT_with_a_moving_obstacle_receding_horizon():
    """FreeTPoint2point with the example's moving circular obstacle (bilinear T * tau * v
    terms in the obstacle rows): every MPC step converges and the vehicle arrives."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_freeT(build_solver=False, moving=True)
    pr.problem = _OracleSolver(pr.father.tables)
    pr.initialize(0.)
    t, dt = 0., 0.5
    for k in range(24):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        assert pr.problem.stats()['return_status'] == 'Solve_Succeeded', k
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t = np.round(t + dt, 6)
        if pr.stop_criterium(t, dt):
            break
    assert k < 23
    assert np.abs(pr.vehicles[0].signals['state'][:, -1] - [2., 2.]).max() < 1e-2


def test_freeT_with_safety_distance_and_dubins_freeT():
    """Free end time with a safety-distance slack (the slack objective starts at t/T = 0:
    basics/poly.py rel_time) -- the MPC loop converges at every step, arrives, and keeps the
    obstacle at more than its radius; and examples/p2p_dubins.py as written (substitution,
    freeT): the motion time multiplies the intermediates.  From a rolling speed guess the
    oracle converges to a motion time between the straight-line bound and 10 s; from the
    reference's zero-speed guess the Jacobian of the position rows is rank deficient and
    the line search gives up -- IPOPT's restoration phase; here the host-level feasibility
    phase followed by a second solve, DESIGN.md section 2."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_freeT_safety(build_solver=False)
    pr.problem = _OracleSolver(pr.father.tables)
    pr.initialize(0.)
    t, dt = 0., 0.5
    for k in range(24):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        assert pr.problem.stats()['return_status'] == 'Solve_Succeeded', k
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t = np.round(t + dt, 6)
        if pr.stop_criterium(t, dt):
            break
    pos = pr.vehicles[0].signals['state']
    assert np.abs(pos[:, -1] - [2., 2.]).max() < 1e-2
    assert np.hypot(pos[0] - 0.3, pos[1] - 0.2).min() > 0.6 - 1e-3
    pr = sc.config_dubins_freeT(build_solver=False)
    tb, f = pr.father.tables, pr.father
    assert tb.n_mid > 0 and tb.nnz_wx > 0
    x0, p0 = f.get_variables().cat[None], f.set_parameters(0.).cat[None]
    r = ipm_c.solve_batch_full(tb, x0, p0, threads=1, options={'feas_steps': 0})
    assert r['status'][0] == 2                     # the reference's zero-speed guess, line search alone
    r = ipm_c.solve_batch_full(tb, x0, p0, threads=1)
    assert r['status'][0] == 0 and 7. < r['f'][0] < 8.     # with the feasibility phase (DESIGN.md section 2)
    # vehicle option init_v_til: rolling initial guess; the example's whole MPC loop
    pr = sc.config_dubins_freeT(build_solver=False, init_v_til=0.3)
    pr.problem = _OracleSolver(pr.father.tables)
    pr.initialize(0.)
    t, dt, Ts = 0., 0.5, []
    for k in range(30):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        assert pr.problem.stats()['return_status'] == 'Solve_Succeeded', k
        Ts.append(pr.horizon_time())
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t = np.round(t + dt, 6)
        if pr.stop_criterium(t, dt):
            break
    assert np.hypot(3., 3.) / 0.7 < Ts[0] < 10.
    assert np.abs(pr.vehicles[0].signals['state'][:, -1] - [3., 3., 0.]).max() < 1e-2


def test_trailer_solves():
    """vehicles/trailer.py (examples/p2p_trailer.py: Dubins vehicle + trailer on a 0.6 m hitch,
    free end time, the lead vehicle added to the problem a second time): from a rolling guess
    the oracle converges; the hitch kinematics hold along the solution and the articulation
    angle stays within +-45 degrees."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = _cached_problem('config_trailer')
    tb, f = pr.father.tables, pr.father
    assert (tb.n, tb.m, tb.n_par) == (61, 3081, 12)
    X0 = f.get_variables().cat[None].copy()
    for veh, col in ((pr.vehicles[0], 1), (pr.vehicles[1], 0)):      # option init_v_til = 0.3
        off = f._var_struct.entries[(veh.label, 'splines_seg0')][0]
        X0[0, off + 12 * col:off + 12 * (col + 1)] = 0.3
    r = ipm_c.solve_batch_full(tb, X0, f.set_parameters(0.).cat[None], threads=1)
    assert r['status'][0] == 0
    x = r['x'][0]
    T = x[f._var_struct.entries[(pr.label, 'T')][0]]
    assert np.hypot(3.4, 3.) / 0.8 < T < 20.
    C = x[:36].reshape(3, 12)                       # tg_tr, v~, tg of the trailer problem
    basis = pr.vehicles[0].basis
    tau = np.linspace(0., 1., 201)
    S = basis.eval_basis(tau)
    Bd, P1 = basis.derivative(1)
    tg_tr, v, tg = S.dot(C[0]), S.dot(C[1]), S.dot(C[2])
    dtg_tr = Bd.eval_basis(tau).dot(P1.dot(C[0]))
    hitch = T * v * (2 * tg * (1 - tg_tr**2) - (1 - tg**2) * 2 * tg_tr)
    assert np.abs(2 * dtg_tr * 0.6 - hitch).max() < T * 1e-3 + 0.05     # band + spline relaxation
    assert np.abs(2 * np.arctan(tg) - 2 * np.arctan(tg_tr)).max() < np.pi / 4. + 0.02
    assert abs(tg_tr[-1]) < 1e-6 and abs(tg[-1]) < 1e-6


def test_intermediates_small_example_and_guards():
    """lowering.py with 'mid' symbols on a hand-checkable NLP:
    c = x0*x1 (shared), rows  p*c + x2 <= 1  and  2*c - x0 = 0."""
    from omg_tools_b200.basics.lowering import lower
    x = [pl.new_symbol('mx%d' % k, 'var') for k in range(3)]
    p = pl.new_symbol('mp', 'par')
    c = pl.new_mid('mc', x[0] * x[1])
    sid = lambda e: e.single_symbol()
    rows = [p * c + x[2], 2. * c - x[0]]
    tb = lower([sid(v) for v in x], [sid(p)], rows, x[2] * x[2], [-np.inf, 0.], [1., 0.])
    assert (tb.n, tb.m, tb.n_mid) == (3, 2, 1)
    ev = TableEval(tb)
    xv, pv, lam = np.array([0.5, -2., 3.]), np.array([4.]), np.array([0.7, -1.3])
    V = ev.tape(pv)
    assert np.allclose(ev.g(xv, V), [4. * (0.5 * -2.) + 3., 2. * (0.5 * -2.) - 0.5])
    J = ev.jac_dense(xv, V)
    assert np.allclose(J, [[4. * -2., 4. * 0.5, 1.], [2. * -2. - 1., 2. * 0.5, 0.]])
    W = ev.hess_dense(xv, V, lam)
    # Hessian of lam0*p*x0*x1 + lam1*2*x0*x1 + x2^2
    ref = np.zeros((3, 3))
    ref[0, 1] = ref[1, 0] = 0.7 * 4. + (-1.3) * 2.
    ref[2, 2] = 2.
    assert np.allclose(W, ref)
    # guards: rows must be affine in intermediates, intermediates must not nest
    with pytest.raises(NotImplementedError):
        lower([sid(v) for v in x], [sid(p)], [c * c * c], x[2], [0.], [0.])
    c2 = pl.new_mid('mc2', c * x[2])
    with pytest.raises(NotImplementedError):
        lower([sid(v) for v in x], [sid(p)], [c2 + x[0]], x[2], [0.], [0.])


def test_intermediates_with_x_dependent_coefficients():
    """Rows whose mid coefficient depends on x (hyperplane normal times an integrated
    position: Dubins without substitution, AGV, trailer) or on another mid (products of two
    shared product splines: the steering-rate rows of the bicycle).  The Jacobian needs
    A(x, mids) C, the Hessian the terms X^T C + C^T X + C^T M C: a small NLP with every
    combination against finite differences."""
    from omg_tools_b200.basics.lowering import lower
    x = [pl.new_symbol('nx%d' % k, 'var') for k in range(4)]
    p = pl.new_symbol('np', 'par')
    c = pl.new_mid('nc', x[0] * x[1] + p * x[1] * x[1])
    d = pl.new_mid('nd', x[1] * x[2] * x[2])
    sid = lambda e: e.single_symbol()
    rows = [x[3] * c + x[0], x[3] * x[3] * d - 2. * c * x[0] + p * d + 0.5 * c * d - p * x[2] * d * d,
            3. * c - x[2] + c * c]
    tb = lower([sid(v) for v in x], [sid(p)], rows, x[3] * x[3],
               [-np.inf, -np.inf, 0.], [1., 0., 0.])
    assert (tb.n, tb.m, tb.n_mid) == (4, 3, 2) and tb.nnz_wx > 0 and tb.n_xq > 0
    ev = TableEval(tb)
    rng = np.random.default_rng(5)
    xv, pv, lam = rng.standard_normal(4), np.array([0.7]), rng.standard_normal(3)
    V = ev.tape(pv)

    def g(z):
        cc = z[0] * z[1] + pv[0] * z[1] * z[1]
        dd = z[1] * z[2] * z[2]
        return np.array([z[3] * cc + z[0], z[3] * z[3] * dd - 2. * cc * z[0] + pv[0] * dd
                         + 0.5 * cc * dd - pv[0] * z[2] * dd * dd, 3. * cc - z[2] + cc * cc])

    assert np.allclose(ev.g(xv, V), g(xv))
    h = 1e-5
    J = ev.jac_dense(xv, V)
    Jfd = np.array([(g(xv + h * e) - g(xv - h * e)) / (2 * h) for e in np.eye(4)]).T
    assert np.abs(J - Jfd).max() < 1e-8
    W = ev.hess_dense(xv, V, lam, 0.5)

    def lag_grad(z):
        Vz = ev.tape(pv)
        return ev.jac_dense(z, Vz).T.dot(lam) + 0.5 * ev.gradf(z, Vz)

    Wfd = np.array([(lag_grad(xv + h * e) - lag_grad(xv - h * e)) / (2 * h) for e in np.eye(4)])
    assert np.abs(W - Wfd).max() < 1e-8 and np.abs(W - W.T).max() == 0.


def test_planar_quadrotor_receding_horizon():
    """examples/p2p_quadrotor.py (vehicles/quadrotor.py): flat outputs x, y of
    degree 4, thrust and pitch-rate limits as quadratic rows.  Sizes, table
    derivatives, and the reference's MPC loop to the goal with the oracle."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_quadrotor2d(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_par, tb.degree) == (103, 496, 28, 2)
    ev = TableEval(tb)
    rng = np.random.default_rng(2)
    X0, P = sc.instance_data(pr, 1)
    x = X0[0] + 0.05 * rng.standard_normal(tb.n)
    V = ev.tape(P[0])
    J = ev.jac_dense(x, V)
    h = 1e-6
    for j in rng.choice(tb.n, 8, replace=False):
        e = np.zeros(tb.n)
        e[j] = h
        fd = (ev.g(x + e, V) - ev.g(x - e, V)) / (2 * h)
        assert np.abs(fd - J[:, j]).max() < 1e-6 * max(1., np.abs(J[:, j]).max())
    pr.problem = _OracleSolver(tb)
    pr.initialize(0.)
    t, dt = 0., 0.25
    n_ok = 0
    for k in range(21):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        n_ok += pr.problem.stats()['return_status'] == 'Solve_Succeeded'
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t += dt
    # The thrust lower bound is a non-convex quadratic: while it is active the reduced
    # Hessian has negative curvature, the inertia correction adds delta_w ~ 1e3 and the
    # solve crawls (one step of this run hits the iteration limit; its iterate is
    # feasible and the loop recovers at the next step).
    assert n_ok >= 19
    veh = pr.vehicles[0]
    assert np.abs(veh.signals['state'][:2, -1] - [4., 4.]).max() < 5e-2
    u1 = veh.signals['input'][0]
    assert u1.min() > 2. - 1e-2 and u1.max() < 15. + 1e-2      # thrust limits hold along the flight


def test_batch_mpc_quadrotor_prediction_matches_reference_loop():
    """execution/batch_mpc.py: the Quadrotor3D adapter predicts position and
    velocity by exact Gauss-Legendre quadrature of the flat-output accelerations;
    it must reproduce the reference-style Vehicle.store/predict bookkeeping
    (splines2signals + integrate_twice), including a step across a knot."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    from omg_tools_b200.execution import batch_mpc as bm

    class HostTensor(object):          # what the adapter needs from a CUDA tensor
        def __init__(self, a):
            self.a = a

        def cpu(self):
            return self

        def numpy(self):
            return self.a

    pr = sc.config4(build_solver=False)
    pr.problem = _OracleSolver(pr.father.tables)
    pr.initialize(0.)
    veh = pr.vehicles[0]
    ad = bm._Quadrotor3DAdapter(None, veh, 1, 0., np.random.default_rng(0))
    t, dt = 0., 0.4
    for k in range(3):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        if k > 0:
            assert np.abs(ad.state[0] - veh.prediction['state']).max() < 1e-11
            assert np.abs(ad.inp[0] - veh.prediction['input']).max() < 1e-11
        pr.solve(t, dt)
        x = pr.father.get_variables().cat
        ad.predict(HostTensor(x[None]), np.round(t, 6) % pr.knot_time, dt, 5.0, device=False)
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t += dt
    # parameter packing of the adapter == the model's set_parameters
    P = np.zeros((1, pr.father.tables.n_par))
    ent = pr.father._par_struct.entries
    ad.state, ad.inp = veh.prediction['state'][None].copy(), veh.prediction['input'][None].copy()
    ad.pack(P, {key: ent[key][0] for key in ent})
    ref = pr.father.set_parameters(t).cat
    for key, (off, size, _) in ent.items():
        if key[0] == veh.label:
            assert np.abs(P[0, off:off + size] - ref[off:off + size]).max() < 1e-12, key


def test_dubins_substitution_receding_horizon():
    """vehicles/dubins.py (examples/p2p_dubins.py with a fixed end time): flat
    outputs v~, tan(theta/2); the position band rows share 116 intermediates.
    Table derivatives, then the MPC loop drives the vehicle to (3, 3, 0) within the
    speed and turn-rate limits, every solve converged."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_dubins(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_mid, tb.degree) == (126, 554, 116, 3)
    ev = TableEval(tb)
    rng = np.random.default_rng(3)
    X0, P = sc.instance_data(pr, 1)
    x = X0[0] + 0.05 * rng.standard_normal(tb.n)
    V = ev.tape(P[0])
    J = ev.jac_dense(x, V)
    lam = rng.standard_normal(tb.m)
    W = ev.hess_dense(x, V, lam)
    h = 1e-6
    for j in rng.choice(tb.n, 8, replace=False):
        e = np.zeros(tb.n)
        e[j] = h
        fd = (ev.g(x + e, V) - ev.g(x - e, V)) / (2 * h)
        assert np.abs(fd - J[:, j]).max() < 1e-6 * max(1., np.abs(J[:, j]).max())
        dj = (ev.jac_dense(x + e, V).T @ lam - ev.jac_dense(x - e, V).T @ lam) / (2 * h)
        assert np.abs(dj - W[:, j]).max() < 1e-5 * max(1., np.abs(W[:, j]).max())
    pr.problem = _OracleSolver(tb)
    pr.initialize(0.)
    t, dt = 0., 0.5
    for k in range(22):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        assert pr.problem.stats()['return_status'] == 'Solve_Succeeded', k
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t = np.round(t + dt, 6)
    veh = pr.vehicles[0]
    assert np.abs(veh.signals['state'][:, -1] - [3., 3., 0.]).max() < 1e-2
    assert veh.signals['input'][0].max() < 0.7 + 1e-3
    assert np.abs(veh.signals['input'][1]).max() < np.pi / 3. + 1e-3


def test_dubins_default_formulation_receding_horizon():
    """Dubins as the reference defines it by default (substitution=False, dubins.py:63,
    235-251): the integrated position enters the terminal and collision rows, so the
    hyperplane normal multiplies the shared intermediates -- cross-Hessian slots of
    lowering.py.  Table derivatives by finite differences, numpy and C oracle agree, and
    the MPC loop reaches (3, 3, 0) with every solve converged."""
    from oracle import ipm_c, ipm_ref
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_dubins_plain(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_mid, tb.degree) == (190, 856, 118, 3)
    assert tb.nnz_wx == 308 and tb.W.n_out == tb.nnz_w + tb.nnz_wx
    ev = TableEval(tb)
    rng = np.random.default_rng(3)
    X0, P = sc.instance_data(pr, 1)
    x = X0[0] + 0.05 * rng.standard_normal(tb.n)
    V = ev.tape(P[0])
    J = ev.jac_dense(x, V)
    lam = rng.standard_normal(tb.m)
    W = ev.hess_dense(x, V, lam)
    assert np.abs(W - W.T).max() == 0.
    h = 1e-6
    for j in rng.choice(tb.n, 8, replace=False):
        e = np.zeros(tb.n)
        e[j] = h
        fd = (ev.g(x + e, V) - ev.g(x - e, V)) / (2 * h)
        assert np.abs(fd - J[:, j]).max() < 1e-6 * max(1., np.abs(J[:, j]).max())
        dj = (ev.jac_dense(x + e, V).T @ lam - ev.jac_dense(x - e, V).T @ lam) / (2 * h)
        assert np.abs(dj - W[:, j]).max() < 1e-5 * max(1., np.abs(W[:, j]).max())
    # the two oracles take the same path
    rc = ipm_c.solve_batch_full(tb, X0, P, threads=1)
    rn = ipm_ref.solve(tb, X0[0], P[0])
    assert rc['status'][0] == 0 == rn.status and abs(int(rc['iters'][0]) - rn.iters) <= 1
    assert np.abs(rc['x'][0] - rn.x)[:26].max() < 1e-5
    pr.problem = _OracleSolver(tb)
    pr.initialize(0.)
    t, dt = 0., 0.5
    for k in range(22):
        pr.predict(t, dt, 0.01)
        pr.init_step(t, dt)
        pr.solve(t, dt)
        assert pr.problem.stats()['return_status'] == 'Solve_Succeeded', k
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t = np.round(t + dt, 6)
    veh = pr.vehicles[0]
    assert np.abs(veh.signals['state'][:, -1] - [3., 3., 0.]).max() < 1e-2
    assert veh.signals['input'][0].max() < 0.7 + 1e-3
    assert np.abs(veh.signals['input'][1]).max() < np.pi / 3. + 1e-3


def test_dubins_exact_substitution_solves():
    """exact_substitution (dubins.py:95-101): dx, dy on the product basis tied by
    equality rows; no intermediates."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_dubins_exact(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_mid) == (166, 517, 0)
    X0, P = sc.instance_data(pr, 1)
    r = ipm_c.solve_batch_full(tb, X0, P, threads=1)
    assert r['status'][0] == 0
    ev = TableEval(tb)
    g = ev.g(r['x'][0], ev.tape(P[0]))
    assert (g <= tb.ubg + 1e-4).all() and (g >= tb.lbg - 1e-4).all()


def test_bicycle_tables_and_solve():
    """vehicles/bicycle.py (examples/p2p_bicycle.py, fixed end time): steering-rate rows with
    products of two shared product splines (mid-mid Hessian slots), integrated position
    times hyperplane normal (cross slots).  Table derivatives against finite differences;
    from a rolling initial guess (v~ = 0.3; the reference's all-zero speed guess sits on a
    degenerate point of the steering rows, where only IPOPT's restoration phase gets away)
    both oracles converge to the same point."""
    from oracle import ipm_c, ipm_ref
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_bicycle(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_par, tb.n_mid, tb.degree) == (85, 646, 25, 167, 5)
    assert tb.nnz_wx > 0 and (tb.xq_b >= 0).any() and (tb.xq_b < 0).any()
    ev = TableEval(tb)
    rng = np.random.default_rng(4)
    X0, P = sc.instance_data(pr, 1)
    X0[0, :7] = 0.3
    x = X0[0] + 0.05 * rng.standard_normal(tb.n)
    V = ev.tape(P[0])
    J = ev.jac_dense(x, V)
    lam = rng.standard_normal(tb.m)
    W = ev.hess_dense(x, V, lam)
    h = 1e-6
    for j in rng.choice(tb.n, 8, replace=False):
        e = np.zeros(tb.n)
        e[j] = h
        fd = (ev.g(x + e, V) - ev.g(x - e, V)) / (2 * h)
        assert np.abs(fd - J[:, j]).max() < 1e-6 * max(1., np.abs(J[:, j]).max())
        dj = (ev.jac_dense(x + e, V).T @ lam - ev.jac_dense(x - e, V).T @ lam) / (2 * h)
        assert np.abs(dj - W[:, j]).max() < 1e-5 * max(1., np.abs(W[:, j]).max())
    rc = ipm_c.solve_batch_full(tb, X0, P, threads=1)
    rn = ipm_ref.solve(tb, X0[0], P[0])
    assert rc['status'][0] == 0 == rn.status and abs(int(rc['iters'][0]) - rn.iters) <= 1
    assert np.abs(rc['x'][0] - rn.x)[:14].max() < 1e-5
    g = ev.g(rc['x'][0], V)
    assert (g <= tb.ubg + 1e-4).all() and (g >= tb.lbg - 1e-4).all()


def test_simple_quadrotor3d_solves():
    """vehicles/quadrotor3d_simple.py: quadratic (non-convex) thrust / body-rate / tilt rows;
    the oracle converges to a feasible trajectory that reaches the goal."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_quadrotor3d_simple(build_solver=False)
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_par, tb.degree, tb.n_mid) == (200, 913, 64, 2, 0)
    X0, P = sc.instance_data(pr, 1)
    r = ipm_c.solve_batch_full(tb, X0, P, threads=1)
    assert r['status'][0] == 0
    ev = TableEval(tb)
    g = ev.g(r['x'][0], ev.tape(P[0]))
    assert (g <= tb.ubg + 1e-4).all() and (g >= tb.lbg - 1e-4).all()
    L = len(pr.vehicles[0].basis)
    assert np.abs(r['x'][0][[L - 1, 2 * L - 1, 3 * L - 1]] - [3., 2., 0.5]).max() < 1e-2


def test_formation_central_solves():
    """problems/formation_central.py (examples/formation_holonomic_central.py): four vehicles
    in one NLP with soft formation constraints; the fleet shares the terminal and formation
    slack splines (the reference's name-based composition).  The oracle converges to a
    feasible (local) solution through the gap, in formation from mid-horizon on."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = sc.config_formation_central(build_solver=False)
    tb, f = pr.father.tables, pr.father
    assert (tb.n, tb.m, tb.n_par) == (420, 2468, 70)
    names = [k[1] for k in f._var_struct.entries.keys()]
    assert names.count('g0') == 1 and names.count('eps_form_00') == 1
    r = ipm_c.solve_batch_full(tb, f.get_variables().cat[None], f.set_parameters(0.).cat[None], threads=1)
    assert r['status'][0] == 0
    x = r['x'][0]
    ent = f._var_struct.entries
    C = np.array([x[ent[(v.label, 'splines_seg0')][0]:][:26] for v in pr.vehicles]).reshape(4, 2, 13)
    ev = TableEval(tb)
    g = ev.g(x, ev.tape(f.set_parameters(0.).cat))
    assert (g <= tb.ubg + 1e-4).all() and (g >= tb.lbg - 1e-4).all()
    goals = np.array([v.poseT for v in pr.vehicles])
    assert np.abs(C[:, 1, -1] - goals[:, 1]).max() < 1e-2     # through the gap, y reached
    centre = C + np.array([v.rel_pos_c for v in pr.vehicles])[:, :, None]
    # (the vehicles start in a row; the soft constraints pull them into formation)
    # and let it deform by a few cm while squeezing through the 0.5 m gap
    err = np.abs(centre - centre.mean(0)).max(axis=(0, 1))
    assert err[3:].max() < 0.15 and err[8:].max() < 1e-3


def test_holonomic_orient_solves():
    """vehicles/holonomicorient.py (examples/p2p_holonomic_orient.py, fixed end time):
    rectangular vehicle with free heading, degree-4 collision rows; the oracle converges to a
    feasible trajectory."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    pr = _cached_problem('config_holonomic_orient')
    tb = pr.father.tables
    assert (tb.n, tb.m, tb.n_par, tb.degree, tb.n_mid) == (189, 3035, 56, 3, 232)
    X0, P = sc.instance_data(pr, 1)
    r = ipm_c.solve_batch_full(tb, X0, P, threads=1)
    assert r['status'][0] == 0
    ev = TableEval(tb)
    g = ev.g(r['x'][0], ev.tape(P[0]))
    assert (g <= tb.ubg + 1e-4).all() and (g >= tb.lbg - 1e-4).all()
    # (fixed 10 s horizon: the soft terminal position is not reached, the vehicle stops on
    # the way; rest-to-rest with the initial heading kept by the regularisation)
    x = r['x'][0]
    assert np.abs(x[26:39] - np.tan(np.pi / 8.)).max() < 1e-3
    assert x[12] > 1. and x[25] > 1.


def test_more_reference_examples_lower_and_solve():
    """examples/p2p_holonomic_octroom.py (octagonal room -> half-plane room rows)
    and a Holonomic with Euclidean (norm_2) velocity/acceleration limits: tables
    build and the oracle converges to a feasible trajectory."""
    from omg_tools_b200 import (Holonomic, Environment, Obstacle, Rectangle, Circle,
                                RegularPolyhedron, Square)
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')

    def octroom():
        vehicle = Holonomic()
        vehicle.set_options({'safety_distance': 0.1})
        vehicle.set_initial_conditions([-1.5, -1.5])
        vehicle.set_terminal_conditions([1.0, 1.5])
        environment = Environment(room={'shape': RegularPolyhedron(2.5, 8)})
        rectangle = Rectangle(width=3., height=0.2)
        environment.add_obstacle(Obstacle({'position': [-2.1, -0.5]}, shape=rectangle))
        environment.add_obstacle(Obstacle({'position': [1.7, -0.5]}, shape=rectangle))
        traj = {'velocity': {'time': [3., 4.], 'values': [[-0.15, 0.0], [0., 0.15]]}}
        environment.add_obstacle(Obstacle({'position': [1.5, 0.5]}, shape=Circle(0.4),
                                          simulation={'trajectories': traj}))
        return sc._p2p(vehicle, environment, None, False)

    def norm2():
        vehicle = Holonomic(options={'syslimit': 'norm_2'}, bounds={'vmax': 0.6, 'amax': 1.2})
        vehicle.set_initial_conditions([-1.5, -1.5])
        vehicle.set_terminal_conditions([2., 2.])
        environment = Environment(room={'shape': Square(5.)})
        environment.add_obstacle(Obstacle({'position': [0.3, 0.2]}, shape=Circle(0.6)))
        return sc._p2p(vehicle, environment, None, False)

    for build, m_expected in ((octroom, 801), (norm2, None)):
        pr = build()
        tb = pr.father.tables
        if m_expected:
            assert tb.m == m_expected
        X0, P = sc.instance_data(pr, 1)
        r = ipm_c.solve_batch_full(tb, X0, P, threads=1)
        assert r['status'][0] == 0
        ev = TableEval(tb)
        g = ev.g(r['x'][0], ev.tape(P[0]))
        assert (g <= tb.ubg + 1e-4).all() and (g >= tb.lbg - 1e-4).all()
    # norm_2 limits: the speed along the solution stays below vmax
    veh = pr.vehicles[0]
    basis = veh.basis
    tau = np.linspace(0, 1, 201)
    Bd, P1 = basis.derivative(1)
    D = Bd.eval_basis(tau).dot(P1) / 10.
    x = r['x'][0]
    speed = np.hypot(D.dot(x[:13]), D.dot(x[13:26]))
    assert speed.max() < 0.6 + 1e-3


EXT_GOLDEN = ('config_dubins_plain', 'config_dubins_rect', 'config_dubins_exact',
              'config_holonomic_orient', 'config_bicycle', 'config_agv',
              'config_quadrotor3d_simple', 'config_formation_central', 'config_interveh',
              'config_free_end', 'config_freeT', 'config_freeT_moving', 'config_freeT_safety',
              'config_dubins_freeT', 'config_trailer', 'config_formation_central_example',
              'config_warehouse', 'config_revolving_door_diffdrive',
              'config_revolving_door_quadrotor')


_PROBLEMS = {}


def _cached_problem(name):
    """Scenario built once per test session for the tests that only READ the problem (the
    large models take 10-30 s to lower)."""
    if name not in _PROBLEMS:
        _PROBLEMS[name] = getattr(sc, name)(build_solver=False)
    return _PROBLEMS[name]


def _model_golden(name):
    """The fixture file holding `name` (make_model_golden.py --ext splits the ext models over three
    files, each below 1 MB)."""
    import os
    files = ('model_golden_ext1.npz', 'model_golden_ext2.npz', 'model_golden_ext3.npz') \
        if name in EXT_GOLDEN else ('model_golden.npz',)
    for fn in files:
        M = np.load(os.path.join(os.path.dirname(__file__), 'golden', fn))
        if name + '_var_layout' in M.files:
            return M
    raise KeyError(name)


@pytest.mark.parametrize('name', ['config1', 'config2', 'config4', 'config5', 'config_holonomic3d',
                                  'config_quadrotor2d', 'config_dubins'] + list(EXT_GOLDEN))
def test_nlp_definition_equals_the_references_own_model_code(name):
    """tests/golden/model_golden.npz holds g_ref(x, p), f_ref(x, p), the bounds and the
    flat layout produced by the REFERENCE's modelling code itself (vehicles, environment,
    obstacles, Point2point.construct, spline algebra) run on a numeric stand-in for
    casadi.MX (tests/golden/make_model_golden.py).  This framework's lowered tables --
    including the chain-rule tables of Quadrotor3D -- must give the same numbers: every
    constraint row, in the same order, with the same bounds, and the objective."""
    import re
    M = _model_golden(name)
    pr = _cached_problem(name)
    tb, f = pr.father.tables, pr.father
    norm = lambda s: re.sub(r'(vehicle|obstacle|p2p|environment)\d+', r'\1#', str(s))
    layout = lambda st: [norm('%s|%s|%dx%d' % (k[0], k[1], v[2][0], v[2][1]))
                         for k, v in st.entries.items()]
    assert layout(f._var_struct) == [norm(s) for s in M[name + '_var_layout']]
    ref_par = [norm(s) for s in M[name + '_par_layout']]
    keep = np.ones(M[name + '_P'].shape[1], dtype=bool)
    if 'freeT' in name or name in ('config_trailer', 'config_warehouse'):
        # The reference defines T twice under one name: as a parameter handed to the vehicle
        # and environment rows and -- afterwards -- as the variable of the objective
        # (point2point.py:53-62, 281-284); the parameter is never set.  Here T is the variable
        # in every row (problems/point2point.py); the golden holds the same value for both.
        k_T = ref_par.index('p2p#|T|1x1')
        keep[sum(int(e.split('|')[2].split('x')[0]) * int(e.split('|')[2].split('x')[1])
                 for e in ref_par[:k_T])] = False
        ref_par.pop(k_T)
    assert layout(f._par_struct) == ref_par
    assert np.array_equal(tb.lbg, M[name + '_lb']) and np.array_equal(tb.ubg, M[name + '_ub'])
    ev = TableEval(tb)
    for k in range(M[name + '_X'].shape[0]):
        x, p = M[name + '_X'][k], M[name + '_P'][k][keep]
        V = ev.tape(p)
        g_ref = M[name + '_G'][k]
        err = np.abs(ev.g(x, V) - g_ref) / np.maximum(1., np.abs(g_ref))
        assert err.max() < 1e-7, (k, int(np.argmax(err)))
        # (degree-9..16 product splines in the ext fixtures: a few more ulps of rounding)
        assert np.median(err) < (1e-12 if name in EXT_GOLDEN else 1e-13)
        assert abs(ev.f(x, V) - M[name + '_F'][k]) < (1e-10 if name in EXT_GOLDEN else 1e-12)
    # what the host feeds the solver: the parameter vector at t = 0.37 (every child's
    # set_parameters, optilayer.py:427-445) and the initial guess of the vehicle splines
    assert np.array_equal(f.set_parameters(0.37).cat, M[name + '_host_P'][keep])
    assert np.array_equal(f.get_variables().cat, M[name + '_host_X0'])


@pytest.mark.parametrize('name', ['config1', 'config4', 'config5', 'config_holonomic3d',
                                  'config_quadrotor2d', 'config_dubins', 'config_dubins_plain',
                                  'config_holonomic_orient', 'config_bicycle',
                                  'config_quadrotor3d_simple', 'config_trailer'])
def test_trajectory_extraction_equals_the_references(name):
    """Post-solve extraction (SURVEY 8f item 1): the reference's Vehicle.store ->
    concat_splines / splines2signals / sample_splines, run from /root/reference on a
    perturbed initial-guess spline (tests/golden/make_model_golden.py), against this
    framework's Vehicle.store on the same coefficients and time axis -- every signal the
    reference produces (state, input, and the model specific ones)."""
    from omg_tools_b200.basics.spline import BSpline
    M = _model_golden(name)
    pr = getattr(sc, name)(build_solver=False)
    veh = pr.vehicles[0]
    C, tax = M[name + '_traj_C'], M[name + '_traj_time']
    splines = [BSpline(veh.basis, C[:, k]) for k in range(C.shape[1])]
    veh.store(1.3, 0.01, [splines], pr.options.get('horizon_time', 10.), tax)   # (free T: the generator's 10 s)
    assert len(M[name + '_traj_keys']) >= 2
    for key in M[name + '_traj_keys']:
        ref = M[name + '_traj_' + str(key)]
        mine = np.atleast_2d(veh.trajectories[str(key)])
        assert mine.shape == ref.shape, key
        assert np.abs(mine - ref).max() < 1e-12 * max(1., np.abs(ref).max()), key


@pytest.mark.parametrize('name', ['config1', 'config4', 'config5', 'config_holonomic3d',
                                  'config_dubins'])
def test_obstacle_motion_equals_the_references(name):
    """The reference's simulator (Environment.simulate -> ObstaclexD.simulate with the
    'trajectories' increments, rotating obstacles) over 5 s in 0.1 s updates, and the
    parameters every obstacle reports after each update (x, v, a, theta, checkpoints,
    rad) -- from /root/reference via tests/golden/make_model_golden.py -- against this
    framework's Obstacle.simulate / set_parameters.  (The reference integrates with
    scipy's odeint, hence 1e-6.)"""
    import os
    M = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'model_golden.npz'))
    pr = getattr(sc, name)(build_solver=False)
    env = pr.environment
    rows, t = [], 0.
    for _ in range(50):
        env.simulate(0.1, 0.01)
        t = np.round(t + 0.1, 6)
        row = []
        for o in env.obstacles:
            row += list(o.signals['position'][:, -1]) + list(o.signals['velocity'][:, -1])
            pars = o.set_parameters(t)[o]
            pars = {k: v for k, v in pars.items() if k in o._parameters}
            if 'theta' in pars:
                row += [o.signals['orientation'][0, -1]]
            for key in sorted(pars):
                row += list(np.atleast_1d(np.asarray(pars[key], float)).reshape(-1))
        rows.append(row)
    mine, ref = np.array(rows), M[name + '_obst']
    assert mine.shape == ref.shape
    assert np.abs(mine - ref).max() < 1e-6


def test_shapes_equal_the_references():
    """basics/shape.py: checkpoints and radii, canvas limits and (2D polyhedra) the
    half-planes used for non-rectangular rooms, for every shape class, against the
    reference's classes run from /root/reference (tests/golden/make_model_golden.py)."""
    import os
    import omg_tools_b200 as og
    M = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'model_golden.npz'))
    zoo = {
        'circle': og.Circle(0.4), 'rectangle': og.Rectangle(width=3., height=0.2),
        'rectangle_rot': og.Rectangle(width=0.5, height=1.2, orientation=0.3),
        'square': og.Square(0.7), 'beam': og.Beam(width=1.4, height=0.2),
        'beam_rot': og.Beam(width=2.2, height=0.2, orientation=0.5 * np.pi),
        'regpoly8': og.RegularPolyhedron(2.5, 8),
        'regpoly5_rot': og.RegularPolyhedron(0.6, 5, np.pi / 7.),
        'sphere': og.Sphere(0.5), 'cuboid': og.Cuboid(width=0.5, depth=4., height=2.),
        'cuboid_rot': og.Cuboid(width=0.5, depth=1., height=2., orientation=[0.1, 0.4, -0.3]),
        'cube': og.Cube(5.),
        'plate': og.Plate(og.Rectangle(5., 8.), 0.1, orientation=[0., np.pi / 2, 0.]),
        'prisma': og.RegularPrisma(0.25, 0.25, 6)}
    for key, shape in zoo.items():
        chck, rad = shape.get_checkpoints()
        assert np.array_equal(np.array(chck, float), M['shape_%s_chck' % key]), key
        assert np.array_equal(np.array(rad, float), M['shape_%s_rad' % key]), key
        assert np.array_equal(np.array(shape.get_canvas_limits(), float), M['shape_%s_lims' % key]), key
        if 'shape_%s_hyp' % key in M.files:
            hyp = shape.get_hyperplanes(position=[0.3, -0.2])
            mine = np.array([np.r_[np.asarray(h['a'], float).reshape(-1),
                                   float(np.asarray(h['b']).reshape(-1)[0])]
                             for _, h in sorted(hyp.items())])
            assert np.abs(mine - M['shape_%s_hyp' % key]).max() < 1e-14, key


class _RecordingOracleSolver(_OracleSolver):
    def __init__(self, tb):
        _OracleSolver.__init__(self, tb)
        self.calls = []

    def __call__(self, x0, p, lbg, ubg, lam_g0=None, **kw):
        args = [np.asarray(v, float).reshape(-1).copy() for v in (x0, p, lbg, ubg)]
        res = _OracleSolver.__call__(self, x0, p, lbg, ubg)
        self.calls.append(args + [np.asarray(res['x'], float).copy()])
        return res


@pytest.mark.parametrize('name,n_steps', [('config1', 12), ('config5', 12), ('config4', 3),
                                          ('config_dubins_plain', 6),
                                          ('config_quadrotor3d_simple', 6)])
def test_host_loop_equals_the_references_problem_solve_loop(name, n_steps):
    """tests/golden/loop_golden.npz: the REFERENCE's Deployer.update / Simulator.update /
    Problem.solve / OptiFather loop, run from /root/reference around this repository's
    solver (make_loop_golden.py), recorded what it hands to the solver at every MPC
    step.  This framework's loop must hand over the same x0, p, lbg, ubg -- through the
    first knot crossing (config 1 and 5 at t = 1.0) -- and unpack the same x.

    The default Dubins formulation and SimpleQuadrotor3D (loop_golden_ext.npz) run six 0.5 s
    updates, through their first knot crossing.

    Config 4: identical until the first knot crossing; there the reference leaves the
    acceleration slacks ddx/ddy/ddz unshifted (and relies on IPOPT's restoration phase,
    see vehicles/quadrotor3d.py) while this framework shifts them with the other splines."""
    import os
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    L = np.load(os.path.join(os.path.dirname(__file__), 'golden',
                             'loop_golden.npz' if name in ('config1', 'config4', 'config5')
                             else 'loop_golden_ext.npz'))   # make_loop_golden.py --ext
    pr = getattr(sc, name)(build_solver=False)
    tb = pr.father.tables
    pr.problem = _RecordingOracleSolver(tb)
    dt = float(L[name + '_dt'])
    pr.initialize(0.)
    t = 0.
    for k in range(n_steps):
        pr.predict(t, dt, 0.01)
        pr.solve(t, dt)
        pr.store(t, dt, 0.01)
        pr.simulate(t, dt, 0.01)
        t = np.round(t + dt, 6)
    calls = pr.problem.calls
    n_same = n_steps if name != 'config4' else 2
    for k in range(n_same):
        x0, p, lbg, ubg, x = calls[k]
        assert np.abs(x0 - L[name + '_x0'][k]).max() < 1e-6, k
        assert np.abs(p - L[name + '_p'][k]).max() < 1e-7, k        # (reference: odeint obstacle motion)
        assert np.array_equal(lbg, L[name + '_lbg'][k]) and np.array_equal(ubg, L[name + '_ubg'][k])
        assert np.abs(x - L[name + '_x'][k]).max() < 1e-5, k
    if name in ('config_dubins_plain', 'config_quadrotor3d_simple'):
        # non-convex models, 60+ iterations per solve: last-bit differences of the host
        # arithmetic (integrated positions, product splines) reach 1e-7 in the solutions
        assert max(np.abs(calls[k][1] - L[name + '_p'][k]).max() for k in range(n_steps)) < 1e-6
    elif name != 'config4':
        # tight: the two host paths are numerically the same computation
        assert max(np.abs(calls[k][0] - L[name + '_x0'][k]).max() for k in range(n_steps)) < 1e-11
        assert max(np.abs(calls[k][1] - L[name + '_p'][k]).max() for k in range(n_steps)) < 1e-12
    else:
        from omg_tools_b200.basics.spline_extra import shiftoverknot_T
        ent = pr.father._var_struct.entries
        veh = pr.vehicles[0]
        mine, ref = calls[2][0], L[name + '_x0'][2]
        slack = np.zeros(tb.n, dtype=bool)
        for nm in ('ddx', 'ddy', 'ddz'):
            off, size, _ = ent[(veh.label, nm)]
            slack[off:off + size] = True
            T = shiftoverknot_T(veh._splines_prim[nm]['basis'])
            assert np.abs(mine[off:off + size] - T.dot(ref[off:off + size])).max() < 1e-5
        assert np.abs(mine - ref)[~slack].max() < 1e-5


def test_shutdown_of_an_equality_constraint_is_rejected():
    """ADVICE r1: switching an equality row off through the bounds changes the structure the
    solver factorises (the border of the condensed KKT system).  The modelling layer refuses it
    at definition time instead of failing inside the solve."""
    import pytest
    from omg_tools_b200.basics.optilayer import OptiChild
    child = OptiChild('shutdown_test')
    x = child.define_variable('x', 2)
    child.define_constraint(x[0] - 1., -np.inf, 0., shutdown='t > 1.')      # inequality: fine
    with pytest.raises(NotImplementedError):
        child.define_constraint(x[1] - 2., 0., 0., shutdown='t > 1.')


def test_predict_branches_follow_the_reference():
    """Vehicle.predict / Problem.predict (reference vehicle.py:302-337, problem.py:138-163;
    ADVICE r1): computation delay shifts the read-out index, measured states are enforced
    through set_initial_conditions (always on the first iteration), a state + input pair
    without the enforce flags does NOT override the ideal prediction."""
    import pytest
    pr = sc.config1(build_solver=False)
    veh = pr.vehicles[0]
    n = 40
    veh.trajectories = {'time': np.arange(n)[None] * 0.01,
                        'state': np.vstack([np.arange(n) * 1.0, np.arange(n) * -1.0]),
                        'input': np.vstack([np.arange(n) * 0.5, np.arange(n) * 0.25])}
    veh.signals = {'state': np.array([[7., 8.], [9., 10.]]), 'input': np.array([[1., 2.], [3., 4.]])}
    # ideal prediction, 0.1 s ahead at 0.01 s sampling, 3 samples of delay -> sample 13
    pr.start_time = 0.
    pr.predict(0.5, 0.1, 0.01, delay=3)
    assert np.allclose(veh.prediction['state'], [13., -13.]) and np.allclose(veh.prediction['input'], [6.5, 3.25])
    # a measurement without enforce flags does not replace the prediction
    pr.predict(0.5, 0.1, 0.01, states=[0.3, 0.4], inputs=[0.1, 0.2])
    assert np.allclose(veh.prediction['state'], [10., -10.])
    # enforce_states: the measurement, or the last simulated signal
    pr.predict(0.5, 0.1, 0.01, states=[0.3, 0.4], enforce_states=True)
    assert np.allclose(veh.prediction['state'], [0.3, 0.4])
    pr.predict(0.5, 0.1, 0.01, enforce_states=True)
    assert np.allclose(veh.prediction['state'], [8., 10.])
    pr.predict(0.5, 0.1, 0.01, states=[0.5, 0.6], inputs=[0.1, 0.2], enforce_states=True, enforce_inputs=True)
    assert np.allclose(veh.prediction['state'], [0.5, 0.6]) and np.allclose(veh.prediction['input'], [0.1, 0.2])
    # first iteration: the state is enforced whatever the flags say
    pr.start_time = 0.5
    pr.predict(0.5, 0.1, 0.01, states=[1.5, 1.6])
    assert np.allclose(veh.prediction['state'], [1.5, 1.6])
    veh.options['ideal_prediction'] = False
    pr.start_time = 0.
    with pytest.raises(NotImplementedError):
        pr.predict(0.7, 0.1, 0.01)
