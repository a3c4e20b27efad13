"""The sparse L D L^T kernel (omg_ipm_kernel_sp: csrc/omg_sp.cuh, csrc/omg_sp_host.cuh) step by
step, across the symbolic structures it accepts.

A whole solve is a weak test of the linear algebra: convergence is judged on residuals computed
from x, so a factorisation that drops an update term still reaches the same point, often in the
same number of iterations.  Here one structure family -- Holonomic Point2point with k knot
intervals and static Circle(0.3) obstacles -- spans what the kernel executes (root size 1 ... 40,
supernode levels with and without equality rows, 16 ... 2 blocks per SM by shared memory, the
largest factor the packed pair records accept, and both fallbacks to the envelope kernels), and
the kernel is compared with

  (a) the pinned host-side structure of every point;
  (b) the first three interior-point iterates of oracle/ipm_ref with its linear solve replaced by
      an extended-precision one (iterative refinement, residual in long double);
  (c) the oracle's iteration trace, the inertia-correction path included;
  (d) the same instances solved alone, inside mixed batches where one block solves many
      different instances in turn.

Every test runs on two backends: ``emu`` (the kernel source in the CPU emulation of
tools/cpu_emu) and ``gpu`` (the product library on a B200)."""
import contextlib
import os
import re
import sys

import numpy as np
import pytest

from omg_tools_b200 import scenarios as sc
from omg_tools_b200 import Holonomic, Environment, Obstacle, Square, Circle
from oracle import ipm_c, ipm_ref

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import emu_support                       # noqa: E402

# the first three are config 2's obstacles (whose structure the (10, 3) point reproduces)
OBSTACLES = list(sc.CONFIG2_OBSTACLES) + [(0.0, 1.3), (-1.2, 0.9), (1.6, 0.6)]

# (knot intervals, obstacles): N, nnz(L), supernode levels, early-reject levels, root, smem bytes
SPARSE = {
    (4, 0): (38, 242, 5, 1, 1, 6960),
    (16, 0): (86, 710, 8, 1, 1, 16976),
    (4, 3): (104, 1620, 6, 6, 24, 24896),
    (4, 6): (170, 2874, 6, 6, 24, 41680),
    (10, 3): (200, 3960, 8, 8, 36, 54832),
    (16, 3): (296, 6696, 12, 9, 40, 87792),
    (12, 5): (340, 7395, 9, 9, 40, 97456),
}
# blocks per SM.  emu: shared memory alone (the emulation has no register file).  gpu: the
# occupancy calculator with the kernel's real register count -- 128 registers x 128 threads cap
# the four smallest structures at 4 blocks per SM on a B200.
CTAS = {
    'emu': {(4, 0): 16, (16, 0): 12, (4, 3): 8, (4, 6): 5, (10, 3): 4, (16, 3): 2, (12, 5): 2},
    'gpu': {(4, 0): 4, (16, 0): 4, (4, 3): 4, (4, 6): 4, (10, 3): 4, (16, 3): 2, (12, 5): 2},
}
FALLBACK = {
    (14, 5): 'factor too large for the packed pairs',
    (16, 6): 'factor too large for the packed pairs',
    (24, 3): 'column structure too long for the packed pairs',
}
U = 2.0 ** -53


def _holonomic(ki, n_obstacles):
    """Holonomic Point2point with ``ki`` knot intervals and the first ``n_obstacles`` static
    Circle(0.3) obstacles; start, goal, room and safety distance as in config 2."""
    vehicle = Holonomic()
    vehicle.define_knots(knot_intervals=ki)
    vehicle.set_options({'safety_distance': 0.1})
    vehicle.set_initial_conditions([-1.5, -1.5])
    vehicle.set_terminal_conditions([2., 2.])
    environment = Environment(room={'shape': Square(5.)})
    for pos in OBSTACLES[:n_obstacles]:
        environment.add_obstacle(Obstacle({'position': list(pos)}, shape=Circle(0.3)))
    return sc._p2p(vehicle, environment, None, True)


class _Backend(object):
    def __init__(self, name):
        self.name = name
        self._problems = {}

    def problem(self, ki, n_obstacles):
        key = (ki, n_obstacles)
        if key not in self._problems:
            self._problems[key] = _holonomic(ki, n_obstacles)
        return self._problems[key]


@pytest.fixture(scope='module', params=['emu', pytest.param('gpu', marks=pytest.mark.gpu)])
def backend(request):
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    if request.param == 'emu':
        saved = emu_support.activate()        # the problems built below bind to it
        yield _Backend('emu')
        emu_support.restore(saved)
    else:
        yield _Backend('gpu')


@contextlib.contextmanager
def _options(pr, **opts):
    old = dict((k, getattr(pr.problem._opt, k)) for k in opts)
    pr.problem.set_options(opts)
    try:
        yield
    finally:
        pr.problem.set_options(old)


def _structure(info):
    m = re.search(r'N=(\d+) nnz\(L\)=(\d+) .*levels=(\d+) \(early-reject (\d+)\) root=(\d+) .*'
                  r'ctas/SM=(\d+) smem=(\d+)', info)
    assert m, info
    return tuple(int(v) for v in m.groups())


# ---------------------------------------------------------------------------------------------
# (a) the structure family
# ---------------------------------------------------------------------------------------------
def test_structure_family_is_pinned(backend):
    """N, nnz(L), levels, early-reject levels, root and shared memory come from host code only
    and are the same on both backends; blocks per SM differ (CTAS: the emulation counts shared
    memory only, the B200's register file caps the small structures at 4).  The three largest
    problems fall back to the envelope kernels for the stated reason."""
    seen = {}
    for (ki, no), (N, nnz, lev, early, root, smem) in SPARSE.items():
        info = backend.problem(ki, no).problem.structure
        got = _structure(info)
        assert got == (N, nnz, lev, early, root, CTAS[backend.name][(ki, no)], smem), ((ki, no), info)
        assert backend.problem(ki, no).problem.info()['ctas_per_sm'] == got[5]
        seen[(ki, no)] = got
    for (ki, no), why in FALLBACK.items():
        info = backend.problem(ki, no).problem.structure
        assert info == 'envelope kernels (%s)' % why, ((ki, no), info)
    # what the family covers
    assert {s[4] for s in seen.values()} >= {1, 40}                        # smallest / largest root
    assert len(set(CTAS['emu'].values())) >= 4                             # shared-memory layouts
    assert any(s[3] < s[2] for s in seen.values())                         # equality rows in a level
    assert max(s[1] for s in seen.values()) > 7000                         # near SP_MAXL
    assert set(FALLBACK.values()) == {'factor too large for the packed pairs',
                                      'column structure too long for the packed pairs'}


# ---------------------------------------------------------------------------------------------
# (b) Newton steps against an extended-precision KKT solve
# ---------------------------------------------------------------------------------------------
def _extended_precision(monkeypatch, conds=None):
    """ipm_ref's signed Cholesky keeps every inertia decision; the solve with the accepted
    factor gets 4 sweeps of iterative refinement with the residual b - K w in long double.
    ``conds`` collects kappa_inf of every K that was solved with."""
    cholesky, solve = ipm_ref._signed_cholesky, ipm_ref._signed_solve
    held = {}

    def keep_k(K, sign, piv_tol, mode=0):
        held['K'] = np.array(K, dtype=np.longdouble)
        return cholesky(K, sign, piv_tol, mode)

    def refined(L, S, rhs):
        if conds is not None:
            conds.append(np.linalg.cond(held['K'].astype(np.float64), np.inf))
        b = np.asarray(rhs, dtype=np.longdouble)
        w = solve(L, S, rhs).astype(np.longdouble)
        for _ in range(4):
            w += solve(L, S, (b - held['K'].dot(w)).astype(np.float64))
        return w.astype(np.float64)

    monkeypatch.setattr(ipm_ref, '_signed_cholesky', keep_k)
    monkeypatch.setattr(ipm_ref, '_signed_solve', refined)


@pytest.mark.parametrize('point', list(SPARSE))
@pytest.mark.parametrize('jittered', [False, True], ids=['nominal', 'jittered'])
def test_newton_steps_match_an_extended_precision_solve(backend, monkeypatch, point, jittered):
    """x_k after k = 1, 2, 3 iterations (max_iter = k) against the extended-precision reference,
    error  max|x - x_ref| / max(1, max|x_ref - x0|),  bounded by  c N u kappa_inf(K)  with c =
    0.01, kappa the largest over the K the reference solved with in those k iterations (1e4 ...
    2e15: non-unique separating hyperplanes, and jittered starts far from the path).

    Measured error / (N u kappa), largest over all points and k: emulation 1.5e-3, B200 2.6e-4,
    ipm_ref's own dense fp64 signed Cholesky 1.3e-3.  A bound relative to that dense error (16 x)
    holds in the emulation (largest ratio 14) but not on the B200: 20 at (4, 6) nominal, k = 2, 3
    (2.5e-9 against 1.2e-10) -- the dense error is one sample of rounding, not a scale.
    A dropped term of the supernode gather or a skipped panel task gives errors of 0.04 ... 1.6
    at k = 1, above the bound at every point."""
    pr = backend.problem(*point)
    tb = pr.father.tables
    N = tb.n + tb.kkt_n_eq
    X0, P = sc.instance_data(pr, 2, jitter=0.2, seed=1)
    row = 1 if jittered else 0
    x0, p = X0[row:row + 1], P[row:row + 1]
    for k in (1, 2, 3):
        with _options(pr, max_iter=k):
            res = pr.problem.solve_batch(x0, p)
        conds = []
        with monkeypatch.context() as mp:
            _extended_precision(mp, conds)
            ref = ipm_ref.solve(tb, x0[0], p[0], options={'max_iter': k})
        assert res['iters'][0] == k == ref.iters
        assert res['status'][0] == ref.status
        err = np.abs(res['x'][0] - ref.x).max() / max(1.0, np.abs(ref.x - x0[0]).max())
        assert err <= 0.01 * N * U * max(conds), (k, err, max(conds))


# ---------------------------------------------------------------------------------------------
# (c) the iteration trace and the inertia correction
# ---------------------------------------------------------------------------------------------
# (point, seed): row 1 of instance_data(jitter=0.2, seed) solved as a batch of one
TRACED = [((4, 0), 1), ((4, 3), 1), ((10, 3), 4), ((16, 3), 3)]
TRACE_ROWS = 10


def _climbs(delta_w):
    """Per row: how often delta_w was multiplied after its first trial value, and whether by
    KAPPA_W_PLUS (an earlier iteration had a delta_w) -- from the sequence alone, the update
    rule of IPOPT's inertia correction (ipm_ref: delta_w0 = 1e-4, x100 the first time, x8 after,
    /3 decay).  -1: no correction."""
    o = ipm_ref.DEFAULTS
    last, out = 0.0, []
    for d in delta_w:
        if d > 0.0:
            if last == 0.0:
                first, fac = o['delta_w0'], o['kappa_w_plus_first']
            else:
                first, fac = max(o['delta_w_min'], o['kappa_w_minus'] * last), o['kappa_w_plus']
            out.append((int(round(np.log(d / first) / np.log(fac))), last != 0.0))
            last = d
        else:
            out.append((-1, False))
    return out


def _trace_error(a, ref):
    """max |a - ref| / |ref| over the rows; entries under 1e-6 of the column's largest (residuals
    at rounding level) are measured against that floor instead of their own size."""
    den = np.maximum(np.abs(ref), 1e-6 * np.abs(ref).max())
    return float((np.abs(a - ref) / den).max()) if len(ref) else 0.0


def test_iteration_trace_follows_the_oracle(backend, monkeypatch):
    """The kernel's trace of instance 0 (omg_get_trace: iter, f, cinf, dinf, mu, E0, alpha,
    delta_w) against ipm_ref's log over the first 10 iterations.  delta_w and mu are discrete
    decisions: delta_w exactly equal, mu to 4 ulp (on the B200 mu^1.5 comes from the device's
    pow, which is not correctly rounded: 1 ulp apart from numpy at (4, 0)).  The kernel writes row k at the top of iteration k, so its alpha
    and delta_w are those of step k - 1; the oracle's row k holds those of step k.

    f, cinf, dinf, E0 within 1e-8 and alpha within 1e-9 (relative) of the extended-precision
    oracle of test (b) -- or within 16 x the distance of the plain dense fp64 oracle from it.
    The allowance is needed: once a step is taken with a tiny alpha from an ill-conditioned K
    the trajectory itself amplifies rounding; at (4, 3) seed 1 the dense fp64 oracle differs from
    the extended-precision one by 1.6e-6 in cinf, at (16, 3) seed 3 by 2.2e-6 in alpha (the
    kernel in the emulation: 1.1e-6 and 1.6e-7).

    The seeds are chosen so that the inertia correction happens, climbs twice by KAPPA_W_PLUS
    within one iteration (three re-stagings of K through the bulk copy) and runs on the
    structure with equality rows inside the levels (16, 3)."""
    climbs = []
    for point, seed in TRACED:
        pr = backend.problem(*point)
        tb = pr.father.tables
        X0, P = sc.instance_data(pr, 2, jitter=0.2, seed=seed)
        with _options(pr, trace=1, max_iter=TRACE_ROWS):
            res = pr.problem.solve_batch(X0[1:2], P[1:2])
            tr = pr.problem.trace()
        opts = {'max_iter': TRACE_ROWS}
        dense = np.array(ipm_ref.solve(tb, X0[1], P[1], options=opts, trace=True).log)
        with monkeypatch.context() as mp:
            _extended_precision(mp)
            ref = ipm_ref.solve(tb, X0[1], P[1], options=opts, trace=True)
        assert res['iters'][0] == ref.iters and res['status'][0] == ref.status, point
        k = ref.iters + 1
        log = np.array(ref.log)
        assert log.shape == (k, 8) == dense.shape
        assert np.array_equal(tr[:k, 0], log[:, 0])
        # (mu^1.5 of the barrier update: the device's pow is not correctly rounded)
        assert np.allclose(tr[:k, 4], log[:, 4], rtol=4 * U, atol=0.0), (point, tr[:k, 4], log[:, 4])
        assert np.array_equal(tr[1:k, 7], log[:-1, 7]), (point, tr[1:k, 7], log[:-1, 7])
        assert np.array_equal(dense[:, [4, 7]], log[:, [4, 7]])        # the same decisions
        for c, tol in ((1, 1e-8), (2, 1e-8), (3, 1e-8), (5, 1e-8), (6, 1e-9)):
            mine, want, other = (tr[1:k, c], log[:-1, c], dense[:-1, c]) if c == 6 else \
                (tr[:k, c], log[:, c], dense[:, c])
            err, err_dense = _trace_error(mine, want), _trace_error(other, want)
            assert err <= max(tol, 16.0 * err_dense), (point, c, err, err_dense)
        climbs += [(point, c, plus) for c, plus in _climbs(log[:-1, 7])]
    assert any(c >= 0 for _, c, _ in climbs)                               # delta_w > 0
    assert any(c >= 2 and plus for _, c, plus in climbs)                   # two KAPPA_W_PLUS climbs
    assert any(c >= 0 for point, c, _ in climbs if SPARSE[point][3] < SPARSE[point][2])


# ---------------------------------------------------------------------------------------------
# (d) the result does not depend on the batch
# ---------------------------------------------------------------------------------------------
def test_mixed_batch_equals_instances_solved_alone(backend):
    """Different jittered instances in a shuffled batch, each compared bit for bit with the same
    instance solved alone: state a block carries from one instance to the next (the mbarrier
    phase, rd, the never-written fill positions of the assembly scratch) must not leak.  emu:
    (10, 3), 7 instances -- blocks run one after another, so one block solves all of them in
    turn.  gpu: (4, 0) with 3 x (SMs x blocks per SM) instances, so every block takes several;
    32 fixed positions are re-solved alone.  Statuses and iteration counts equal the C oracle."""
    rng = np.random.default_rng(11)
    if backend.name == 'emu':
        pr = backend.problem(10, 3)
        X0, P = sc.instance_data(pr, 8, jitter=0.1, seed=3)
        X0, P = X0[1:], P[1:]                       # row 0 is the nominal instance
        order = rng.permutation(len(X0))
        check = np.arange(len(order))
    else:
        pr = backend.problem(4, 0)
        info = pr.problem.info()
        X0, P = sc.instance_data(pr, 65, jitter=0.1, seed=3)
        X0, P = X0[1:], P[1:]
        B = 3 * info['n_sm'] * info['ctas_per_sm']
        order = rng.permutation(np.arange(B) % len(X0))
        check = np.sort(rng.choice(B, 32, replace=False))
    ref = ipm_c.solve_batch_full(pr.father.tables, X0, P, threads=4)
    assert len(set(ref['iters'])) > 1
    res = pr.problem.solve_batch(X0[order], P[order])
    assert np.array_equal(res['status'], ref['status'][order])
    assert np.array_equal(res['iters'], ref['iters'][order])
    for b in check:
        alone = pr.problem.solve_batch(X0[order[b]][None], P[order[b]][None])
        for key in ('x', 'lam_g', 'f', 'status', 'iters'):
            assert np.array_equal(res[key][b], alone[key][0]), (b, key)
