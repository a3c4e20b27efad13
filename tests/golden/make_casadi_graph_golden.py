"""Record the expression GRAPH that the REFERENCE's modelling code builds, in the form CasADi
exposes it (the instruction list of an expanded SX Function), for the test of
omg_tools_b200/basics/lower_casadi.py.  Authoring container only (needs /root/reference):

    python tests/golden/make_casadi_graph_golden.py      ->  tests/golden/casadi_graph_golden.npz

CasADi is not installed, so nothing here is CasADi -- but the reference's modelling layer only
needs a scalar type with arithmetic, comparisons and sin / cos.  make_model_golden.py runs it
with a stand-in ``MX`` that carries NUMBERS; this script runs the same code with the same
stand-in carrying recording NODES: every scalar operation the reference performs on its symbols
(spline products, derivatives, evalspline's Cox-de Boor recursion with the symbolic abscissa
t/T, the obstacle models ...) appends a node.  The nodes reachable from the objective and the
constraint rows are then written as a straight-line program

    OP_INPUT (x | p, index) / OP_CONST (value) / OP_ADD, SUB, MUL, DIV, NEG, SIN, COS, LT, LE /
    OP_OUTPUT (f | g, index)

with a work-vector index per instruction -- exactly the data
``Function('nlp', [x, p], [f, g]).expand()`` offers through ``instruction_id / _input / _output /
_constant`` (CasADi example "accessing_sx_algorithm").  tests/test_lower_casadi.py replays the
program through ``lower_sx_function`` and checks the resulting tables against this framework's
own lowering of the same scenario.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_model_golden as mg          # noqa: E402  (the stand-in casadi module + scenario builders)

OUT = os.path.join(HERE, 'casadi_graph_golden.npz')

# operation codes of the recording (any distinct integers: the interpreter is handed the table)
OPS = {'OP_CONST': 1, 'OP_INPUT': 2, 'OP_OUTPUT': 3, 'OP_ADD': 10, 'OP_SUB': 11, 'OP_MUL': 12,
       'OP_DIV': 13, 'OP_NEG': 14, 'OP_SIN': 15, 'OP_COS': 16, 'OP_LT': 17, 'OP_LE': 18, 'OP_SQ': 19}


class Node(object):
    """One scalar operation of the recorded graph."""
    __slots__ = ('op', 'a', 'b', 'val', 'which', 'index', 'w')
    __array_priority__ = 2000
    __array_ufunc__ = None
    count = 0

    def __init__(self, op, a=None, b=None, val=0.0):
        self.op, self.a, self.b, self.val = op, a, b, val
        self.which, self.index, self.w = -1, -1, -1
        Node.count += 1

    @staticmethod
    def wrap(x):
        if isinstance(x, Node):
            return x
        if isinstance(x, mg.MX):
            return Node.wrap(x.a.reshape(-1)[0])
        return Node('OP_CONST', val=float(x))

    def _bin(self, other, op, swap=False):
        try:
            o = Node.wrap(other)
        except (TypeError, ValueError):
            return NotImplemented
        return Node(op, o, self) if swap else Node(op, self, o)

    def __add__(self, o): return self._bin(o, 'OP_ADD')
    def __radd__(self, o): return self._bin(o, 'OP_ADD', True)
    def __sub__(self, o): return self._bin(o, 'OP_SUB')
    def __rsub__(self, o): return self._bin(o, 'OP_SUB', True)
    def __mul__(self, o): return self._bin(o, 'OP_MUL')
    def __rmul__(self, o): return self._bin(o, 'OP_MUL', True)
    def __truediv__(self, o): return self._bin(o, 'OP_DIV')
    def __rtruediv__(self, o): return self._bin(o, 'OP_DIV', True)
    def __neg__(self): return Node('OP_NEG', self)
    def __pos__(self): return self

    def __pow__(self, k):
        k = int(k)
        if k == 0:
            return Node('OP_CONST', val=1.0)
        out = self
        for _ in range(k - 1):
            out = out * self
        return out

    # CasADi has only LT / LE: a >= b is b <= a
    def __lt__(self, o): return self._bin(o, 'OP_LT')
    def __le__(self, o): return self._bin(o, 'OP_LE')
    def __gt__(self, o): return self._bin(o, 'OP_LT', True)
    def __ge__(self, o): return self._bin(o, 'OP_LE', True)
    def sin(self): return Node('OP_SIN', self)
    def cos(self): return Node('OP_COS', self)
    __hash__ = object.__hash__


def _obj_array(arr):
    out = np.empty(arr.shape, dtype=object)
    for idx, v in np.ndenumerate(arr):
        out[idx] = v
    return out


def install():
    """Make the stand-in MX of make_model_golden carry Nodes."""
    def new_values(self, name, n, m):
        base = name.rsplit('_', 1)[0]
        if base in self.pending and self.pending[base].shape == (n, m):
            return self.pending.pop(base)
        out = np.empty((n, m), dtype=object)
        for idx in np.ndindex(n, m):
            out[idx] = Node('OP_INPUT')
        return out

    def placeholder(self, base, n, m):
        for full, val in self.values.items():
            if full.rsplit('_', 1)[0] == base and val.shape == (n, m):
                return val
        if base not in self.pending:
            self.pending[base] = new_values(self, base + '_x', n, m)
        return self.pending[base]
    mg.Registry.new_values = new_values
    mg.Registry.placeholder = placeholder

    old_num = mg._num

    def _num(a):
        if isinstance(a, (mg.MX, mg.DM)):
            return a.a
        if isinstance(a, Node):
            out = np.empty((1, 1), dtype=object)
            out[0, 0] = a
            return out
        arr = np.asarray(a)
        if arr.dtype == object:
            arr = _obj_array(arr)
            if arr.ndim == 0:
                arr = arr.reshape(1, 1)
            elif arr.ndim == 1:
                arr = arr.reshape(-1, 1)
            return arr
        return old_num(a)
    mg._num = _num
    cmp = lambda f: (lambda self, o: self._bin(o, lambda x, y: np.frompyfunc(f, 2, 1)(x, y)))
    mg.MX.__ge__ = cmp(lambda x, y: Node.wrap(x) >= y)
    mg.MX.__gt__ = cmp(lambda x, y: Node.wrap(x) > y)
    mg.MX.__le__ = cmp(lambda x, y: Node.wrap(x) <= y)
    mg.MX.__lt__ = cmp(lambda x, y: Node.wrap(x) < y)
    mg.MX.__float__ = lambda self: (_ for _ in ()).throw(TypeError('symbolic'))


def record(name):
    mg.REG = mg.Registry(seed=1)
    opt = mg.ref_import('basics.optilayer')
    for cls in list(opt.OptiChild.__subclasses__()) + [opt.OptiChild]:
        if hasattr(cls, '_labels'):
            cls._labels = []
    problem = mg.build_reference(name)
    children = list(problem.father.children.values())
    n = n_par = 0
    rows, lb, ub = [], [], []
    obj = Node('OP_CONST', val=0.0)
    for ch in children:                                  # flat order of optilayer.py:225-272
        for nm, v in ch._variables.items():
            for node in v.a.reshape(-1, order='F'):
                node.which, node.index = 0, n
                n += 1
        for nm, v in ch._parameters.items():
            for node in v.a.reshape(-1, order='F'):
                node.which, node.index = 1, n_par
                n_par += 1
    # named placeholders (OptiChild.define_symbol: 't', 'T') are resolved BY NAME to the variable
    # or parameter of that name (OptiFather.translate_symbols, optilayer.py:204-223)
    named = {}
    for ch in children:
        for nm, v in list(ch._variables.items()) + list(ch._parameters.items()):
            named.setdefault(nm, []).append(v)
    for ch in children:
        for nm, v in getattr(ch, '_symbols', {}).items():
            if len(named.get(nm, [])) != 1:
                raise RuntimeError('placeholder %s defined %d times' % (nm, len(named.get(nm, []))))
            for node, tgt in zip(v.a.reshape(-1, order='F'), named[nm][0].a.reshape(-1, order='F')):
                node.which, node.index = tgt.which, tgt.index
    for ch in children:
        for nm, con in ch._constraints.items():
            expr = con[0]
            vals = expr.a.reshape(-1, order='F') if isinstance(expr, mg.MX) else np.atleast_1d(np.asarray(expr, float))
            rows += [Node.wrap(v) for v in vals]
            lb += list(np.ones(len(vals)) * con[1])
            ub += list(np.ones(len(vals)) * con[2])
        o = ch._objective
        obj = obj + (Node.wrap(o) if not isinstance(o, (int, float)) else float(o))
    # straight-line program over the nodes reachable from the outputs
    ops, ins, outs, consts = [], [], [], []
    counter = [0]

    def emit(root):
        stack = [(root, False)]
        while stack:
            node, done = stack.pop()
            if node.w >= 0:
                continue
            if not done:
                stack.append((node, True))
                for dep in (node.a, node.b):
                    if dep is not None and dep.w < 0:
                        stack.append((dep, False))
                continue
            node.w = counter[0]
            counter[0] += 1
            if node.op == 'OP_INPUT':
                if node.which < 0:
                    raise RuntimeError('symbol used by the model but not a variable / parameter')
                ops.append(OPS['OP_INPUT']); ins.append((node.which, node.index)); outs.append((node.w, 0)); consts.append(0.0)
            elif node.op == 'OP_CONST':
                ops.append(OPS['OP_CONST']); ins.append((0, 0)); outs.append((node.w, 0)); consts.append(node.val)
            else:
                ops.append(OPS[node.op]); outs.append((node.w, 0)); consts.append(0.0)
                ins.append((node.a.w, node.b.w if node.b is not None else 0))
    emit(obj)
    ops.append(OPS['OP_OUTPUT']); ins.append((obj.w, 0)); outs.append((0, 0)); consts.append(0.0)
    for i, r in enumerate(rows):
        emit(r)
        ops.append(OPS['OP_OUTPUT']); ins.append((r.w, 0)); outs.append((1, i)); consts.append(0.0)
    print(name, 'n', n, 'n_par', n_par, 'm', len(rows), 'nodes created', Node.count, 'instructions', len(ops))
    # stored compactly to keep the file small: the constant of the OP_CONST rows and the output
    # slot of the OP_OUTPUT rows only (every other row writes its own work index and has no
    # constant); tests/test_lower_casadi.py restores the full lists
    ops = np.array(ops, np.int16)
    return {'ops': ops, 'ins': np.array(ins, np.int32),
            'output_slots': np.array(outs, np.int32)[ops == OPS['OP_OUTPUT']],
            'const_values': np.array(consts)[ops == OPS['OP_CONST']],
            'sizes': np.array([n, n_par, len(rows), counter[0]]),
            'lb': np.array(lb), 'ub': np.array(ub)}


def main():
    mg.install_stubs()
    install()
    out = {'op_names': np.array(sorted(OPS)), 'op_codes': np.array([OPS[k] for k in sorted(OPS)])}
    # (config5 -- rotating obstacles, sin / cos atoms -- records 730 k instructions, 3 MB: pass
    #  its name on the command line to include it)
    for name in ['config1', 'config2'] + sys.argv[1:]:
        Node.count = 0
        for key, val in record(name).items():
            out['%s_%s' % (name, key)] = val
    np.savez_compressed(OUT, **out)
    print('wrote', OUT, os.path.getsize(OUT), 'bytes')


if __name__ == '__main__':
    main()
