"""omg_tools_b200/basics/lower_casadi.py: the CasADi-graph -> tables binding that lets the
REFERENCE's own model reach the B200 solver (INTEGRATION.md, create_nlp branch).

CasADi is not installed here, so the interpreter is driven through the same instruction-level
interface (n_instructions / instruction_id / instruction_input / instruction_output /
instruction_constant) by a recording of the graph that the reference's modelling code
(/root/reference/omgtools: Holonomic, Environment, Obstacle, Point2point.construct, spline
algebra, evalspline with the symbolic abscissa t/T) builds for BASELINE configs 1 and 2 --
tests/golden/make_casadi_graph_golden.py, 80 k / 212 k scalar operations.  The tables it
produces must describe the same NLP as this framework's own lowering of the same scenario."""
import os

import numpy as np
import pytest

from omg_tools_b200 import scenarios as sc
from omg_tools_b200.basics import lower_casadi as lc
from oracle import nlp_eval

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'casadi_graph_golden.npz')


class RecordedSXFunction(object):
    """The instruction-level view of casadi.Function (expanded to SX), replayed from the file."""

    def __init__(self, G, name):
        self.ops, self.ins = G[name + '_ops'], G[name + '_ins']
        # the file keeps the constants of OP_CONST and the slots of OP_OUTPUT only; every other
        # instruction writes the next entry of the work vector and has the constant 0
        code = {str(nm): int(c) for nm, c in zip(G['op_names'], G['op_codes'])}
        is_const, is_out = self.ops == code['OP_CONST'], self.ops == code['OP_OUTPUT']
        self.consts = np.zeros(len(self.ops))
        self.consts[is_const] = G[name + '_const_values']
        self.outs = np.zeros((len(self.ops), 2), np.int32)
        self.outs[~is_out, 0] = np.arange(np.count_nonzero(~is_out))
        self.outs[is_out] = G[name + '_output_slots']
        self.n, self.n_par, self.m, self.w = [int(v) for v in G[name + '_sizes']]

    def n_instructions(self): return len(self.ops)
    def instruction_id(self, k): return int(self.ops[k])
    def instruction_input(self, k): return tuple(int(v) for v in self.ins[k])
    def instruction_output(self, k): return tuple(int(v) for v in self.outs[k])
    def instruction_constant(self, k): return float(self.consts[k])
    def sz_w(self): return self.w
    def nnz_in(self, i): return (self.n, self.n_par)[i]
    def nnz_out(self, i): return (1, self.m)[i]


@pytest.fixture(scope='module')
def gold():
    return np.load(GOLD)


@pytest.mark.parametrize('name', ['config1', 'config2'])
def test_reference_graph_lowers_to_the_same_nlp(gold, name):
    f = RecordedSXFunction(gold, name)
    ops = {int(c): str(nm) for nm, c in zip(gold['op_names'], gold['op_codes'])}
    tb_ref = lc.lower_sx_function(f, gold[name + '_lb'], gold[name + '_ub'], ops, names=name)
    pr = getattr(sc, name)(build_solver=False)
    tb = pr.father.tables
    assert (tb_ref.n, tb_ref.m, tb_ref.n_par) == (tb.n, tb.m, tb.n_par)
    assert np.array_equal(tb_ref.lbg, tb.lbg) and np.array_equal(tb_ref.ubg, tb.ubg)
    rng = np.random.default_rng(3)
    _, P0 = sc.instance_data(pr, 1)
    for k in range(3):
        x = rng.uniform(-1., 1., tb.n)
        p = P0[0] + 0.05 * rng.uniform(-1., 1., tb.n_par)
        a, b = nlp_eval.TableEval(tb_ref), nlp_eval.TableEval(tb)
        Va, Vb = a.tape(p), b.tape(p)
        ga, gb = a.g(x, Va), b.g(x, Vb)
        assert np.abs(ga - gb).max() < 1e-11 * max(1., np.abs(gb).max())
        assert abs(a.f(x, Va) - b.f(x, Vb)) < 1e-11
        Ja, Jb = a.jac_dense(x, Va), b.jac_dense(x, Vb)
        assert np.abs(Ja - Jb).max() < 1e-10 * max(1., np.abs(Jb).max())
        lam = rng.uniform(-1., 1., tb.m)
        Ha, Hb = a.hess_dense(x, Va, lam), b.hess_dense(x, Vb, lam)
        assert np.abs(Ha - Hb).max() < 1e-10 * max(1., np.abs(Hb).max())


def test_reference_graph_solves_like_the_repo_model(gold):
    """The tables lowered from the reference's graph through the CPU oracle: same optimum as the
    tables of this framework's own model (config 1, cold start)."""
    from oracle import ipm_c
    if not ipm_c.available():
        pytest.skip('C oracle not built')
    f = RecordedSXFunction(gold, 'config1')
    ops = {int(c): str(nm) for nm, c in zip(gold['op_names'], gold['op_codes'])}
    tb_ref = lc.lower_sx_function(f, gold['config1_lb'], gold['config1_ub'], ops, names='config1s')
    pr = sc.config1(build_solver=False)
    X0, P = sc.instance_data(pr, 2, jitter=0.1, seed=5)
    r1 = ipm_c.solve_batch_full(tb_ref, X0, P, threads=2)
    r2 = ipm_c.solve_batch_full(pr.father.tables, X0, P, threads=2)
    assert (r1['status'] == 0).all() and (r2['status'] == 0).all()
    assert np.abs(r1['x'] - r2['x'])[:, :26].max() < 1e-6
    assert np.abs(r1['f'] - r2['f']).max() < 1e-8


@pytest.mark.gpu
def test_reference_graph_on_the_gpu(gold):
    """The drop-in: the reference's own model (its recorded graph) solved by B200Solver."""
    from omg_tools_b200.solver.b200 import B200Solver
    from oracle import ipm_c
    f = RecordedSXFunction(gold, 'config1')
    ops = {int(c): str(nm) for nm, c in zip(gold['op_names'], gold['op_codes'])}
    tb_ref = lc.lower_sx_function(f, gold['config1_lb'], gold['config1_ub'], ops, names='config1g')
    pr = sc.config1(build_solver=False)
    X0, P = sc.instance_data(pr, 4, jitter=0.1, seed=6)
    res = B200Solver(tb_ref, {}).solve_batch(X0, P)
    ref = ipm_c.solve_batch_full(pr.father.tables, X0, P, threads=4)
    assert (res['status'] == 0).all() and np.array_equal(res['status'], ref['status'])
    assert np.abs(res['x'] - ref['x'])[:, :26].max() < 1e-4
    assert np.abs(res['f'] - ref['f']).max() < 1e-6
