"""Generate tests/golden/model_golden.npz from the REFERENCE's own modelling code.

Run in the authoring container only (needs /root/reference):

    python tests/golden/make_model_golden.py

CasADi is not installed, so the reference's NLP cannot be *solved* here -- but its
modelling layer (omgtools/vehicles, environment, problems, basics/optilayer.OptiChild,
basics/spline*) only needs a scalar type with arithmetic and comparisons.  A stand-in
``casadi`` module is registered whose ``MX`` is a 2-D float array that carries one seeded
random VALUE per symbol (``MX.sym`` draws it; named placeholders take the value of their
definition), plotting and export modules are stubbed, and the reference's files are loaded
straight from /root/reference (nothing is copied).  ``Point2point(...).construct()`` then
runs the reference's own code -- ``define_trajectory_constraints``,
``define_collision_constraints``, the obstacle models, ``integrate_twice`` of Quadrotor3D,
the initial/terminal constraints and the objective -- and every constraint row and the
objective come out as NUMBERS: g_ref(x, p), f_ref(x, p) at that random point.  They are
stored with the flat layout (children order, entry names, shapes), the values of x and p
and the bounds; tests/test_model.py evaluates this framework's lowered tables at the same
points.  That pins the NLP *definition* (every row, its order, its bounds, the objective)
to the reference for BASELINE configs 1, 2, 4 and 5 and for the Holonomic3D, planar
Quadrotor and Dubins examples.
"""
import importlib.util
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

REF = '/root/reference/omgtools'
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'model_golden.npz')


# --------------------------------------------------------------------------
# stand-in for casadi.MX: a 2-D float array carrying one seeded random VALUE per symbol
# --------------------------------------------------------------------------
class Registry(object):
    """Values of every symbol, keyed by its full name ('splines_seg0_vehicle0').  Named
    placeholders (OptiChild.define_symbol: 'T', 't', ...) take the value of the variable or
    parameter with the same base name (optilayer.py:204-223 translate_symbols)."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.values = {}          # full name -> array
        self.pending = {}         # base name -> array (placeholder asked before definition)
        self.fixed = {}           # base name -> value forced by the generator (T, t)

    def new_values(self, name, n, m):
        base = name.rsplit('_', 1)[0]
        if base in self.fixed and n * m == 1:
            return np.full((n, m), self.fixed[base])
        if base in self.pending and self.pending[base].shape == (n, m):
            return self.pending.pop(base)
        return self.rng.uniform(-1., 1., (n, m))

    def define(self, name, n, m):
        if name not in self.values:
            self.values[name] = self.new_values(name, n, m)
        return self.values[name]

    def placeholder(self, base, n, m):
        for full, val in self.values.items():
            if full.rsplit('_', 1)[0] == base and val.shape == (n, m):
                return val
        if base not in self.pending:
            self.pending[base] = (np.full((n, m), self.fixed[base]) if base in self.fixed
                                  else self.rng.uniform(-1., 1., (n, m)))
        return self.pending[base]


REG = None


def _num(a):
    if isinstance(a, (MX, DM)):
        return a.a
    arr = np.asarray(a, dtype=float)
    if arr.ndim == 0:
        arr = arr.reshape(1, 1)
    elif arr.ndim == 1:
        arr = arr.reshape(-1, 1)
    return arr


class MX(object):
    __array_priority__ = 1000
    __array_ufunc__ = None

    def __init__(self, a=0.):
        self.a = _num(a)

    @staticmethod
    def sym(name, n=1, m=1):
        return MX(REG.define(name, n, m))

    @property
    def shape(self):
        return self.a.shape

    def size(self):
        return self.a.shape

    def size1(self):
        return self.a.shape[0]

    def size2(self):
        return self.a.shape[1]

    def __len__(self):
        return self.a.shape[0]

    @property
    def T(self):
        return MX(self.a.T)

    def __getitem__(self, key):
        if not isinstance(key, tuple) and self.a.shape[1] == 1:
            key = (key, slice(None))
        out = self.a[key]
        return MX(out)

    def __iter__(self):
        for i in range(self.a.shape[0]):
            yield self[i]

    def __float__(self):
        return float(self.a.reshape(-1)[0])

    def _bin(self, other, fun):
        if not isinstance(other, (MX, DM, int, float, np.number, np.ndarray, list)):
            return NotImplemented        # e.g. a reference BSpline: let its __r*__ handle it
        a, b = self.a, _num(other)
        if a.shape != b.shape and a.size != 1 and b.size != 1:
            raise ValueError('shape mismatch %s %s' % (a.shape, b.shape))
        return MX(fun(a, b))

    def __add__(self, o): return self._bin(o, lambda x, y: x + y)
    def __radd__(self, o): return self._bin(o, lambda x, y: y + x)
    def __sub__(self, o): return self._bin(o, lambda x, y: x - y)
    def __rsub__(self, o): return self._bin(o, lambda x, y: y - x)
    def __mul__(self, o): return self._bin(o, lambda x, y: x * y)
    def __rmul__(self, o): return self._bin(o, lambda x, y: y * x)
    def __truediv__(self, o): return self._bin(o, lambda x, y: x / y)
    def __rtruediv__(self, o): return self._bin(o, lambda x, y: y / x)
    __div__, __rdiv__ = __truediv__, __rtruediv__
    def __neg__(self): return MX(-self.a)
    def __pos__(self): return self
    def __pow__(self, k): return MX(self.a ** int(k))
    def __ge__(self, o): return self._bin(o, lambda x, y: (x >= y).astype(float))
    def __gt__(self, o): return self._bin(o, lambda x, y: (x > y).astype(float))
    def __le__(self, o): return self._bin(o, lambda x, y: (x <= y).astype(float))
    def __lt__(self, o): return self._bin(o, lambda x, y: (x < y).astype(float))

    def column(self):
        return self.a.reshape(-1, order='F')


class DM(object):
    def __init__(self, a=0.):
        self.a = _num(a.toarray() if hasattr(a, 'toarray') else a)


def mtimes(a, b):
    A, B = _num(a), _num(b)
    if A.size == 1 or B.size == 1:
        return MX(A * B)
    return MX(A.dot(B))


def vertcat(*items):
    return MX(np.vstack([_num(it) for it in items]))


def _unary(fun):
    return lambda x: MX(fun(x.a)) if isinstance(x, MX) else fun(x)


def install_stubs():
    cas = types.ModuleType('casadi')
    cas.MX, cas.SX, cas.DM = MX, type('SX', (), {}), DM
    cas.inf = np.inf
    cas.mtimes, cas.vertcat = mtimes, vertcat
    cas.cos, cas.sin = _unary(np.cos), _unary(np.sin)
    cas.symvar = lambda x: []          # only feeds a bookkeeping dict (optilayer.py:529-533)
    cas.vertsplit = lambda x: [x[i] for i in range(x.shape[0])]
    for name in ('Function', 'nlpsol', 'external', 'substitute',
                 'Compiler', 'Importer'):
        setattr(cas, name, lambda *a, **k: None)
    tools = types.ModuleType('casadi.tools')
    for name in ('struct', 'struct_MX', 'struct_symMX', 'entry'):
        setattr(tools, name, lambda *a, **k: None)
    cas.tools = tools
    sys.modules['casadi'], sys.modules['casadi.tools'] = cas, tools
    # package skeleton: sub-packages resolve to the reference's directories, none of the
    # reference's __init__.py files (which import plotting, GUI, export ...) is executed
    for pkg in ('', '.basics', '.vehicles', '.environment', '.problems', '.execution', '.export'):
        m = types.ModuleType('omgtools' + pkg)
        m.__path__ = [REF + pkg.replace('.', '/')]
        sys.modules['omgtools' + pkg] = m
    plot = types.ModuleType('omgtools.execution.plotlayer')

    class PlotLayer(object):
        def __init__(self, *a, **k):
            pass

        def update_plots(self, *a, **k):
            pass

    plot.PlotLayer = PlotLayer
    plot.mix_with_white = lambda *a, **k: None
    sys.modules['omgtools.execution.plotlayer'] = plot
    exp = types.ModuleType('omgtools.export.export_p2p')
    exp.ExportP2P = type('ExportP2P', (), {})
    sys.modules['omgtools.export.export_p2p'] = exp


def ref_import(name):
    return importlib.import_module('omgtools.' + name)


# --------------------------------------------------------------------------
# scenarios, written against the reference's API (same values as scenarios.py)
# --------------------------------------------------------------------------
def build_reference(name):
    hol = ref_import('vehicles.holonomic')
    env = ref_import('environment.environment')
    obs = ref_import('environment.obstacle')
    shp = ref_import('basics.shape')
    p2p = ref_import('problems.point2point')
    from omg_tools_b200.scenarios import CONFIG2_OBSTACLES
    if name == 'config1':
        vehicle = hol.Holonomic()
        vehicle.set_options({'safety_distance': 0.1})
        vehicle.set_initial_conditions([-1.5, -1.5])
        vehicle.set_terminal_conditions([2., 2.])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        trajectories = {'velocity': {'time': [0., 40.], 'values': [[-0.35, 0.35], [0., 0.15]]}}
        environment.add_obstacle(obs.Obstacle(
            {'position': [1.5, -1]}, shape=shp.Circle(0.5), options={'bounce': False},
            simulation={'trajectories': trajectories}))
        options = {}
    elif name == 'config2':
        vehicle = hol.Holonomic()
        vehicle.set_options({'safety_distance': 0.1})
        vehicle.set_initial_conditions([-1.5, -1.5])
        vehicle.set_terminal_conditions([2., 2.])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        for pos in CONFIG2_OBSTACLES:
            environment.add_obstacle(obs.Obstacle({'position': list(pos)}, shape=shp.Circle(0.4)))
        options = {}
    elif name == 'config5':
        vehicle = hol.Holonomic()
        vehicle.set_initial_conditions([0., -2.0])
        vehicle.set_terminal_conditions([0., 2.0])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        beam1 = shp.Beam(width=2.2, height=0.2)
        environment.add_obstacle(obs.Obstacle({'position': [-2., 0.]}, shape=beam1))
        environment.add_obstacle(obs.Obstacle({'position': [2., 0.]}, shape=beam1))
        beam2 = shp.Beam(width=1.4, height=0.2)
        horizon_time = 10.
        omega = 1.5 * 1. * 2 * np.pi / horizon_time
        environment.add_obstacle(obs.Obstacle(
            {'position': [0., 0.], 'velocity': [0., 0.], 'angular_velocity': omega},
            shape=beam2, simulation={}, options={'horizon_time': horizon_time}))
        environment.add_obstacle(obs.Obstacle(
            {'position': [0., 0.], 'velocity': [0., 0.], 'orientation': 0.5 * np.pi,
             'angular_velocity': omega},
            shape=beam2, simulation={}, options={'horizon_time': horizon_time}))
        options = {'horizon_time': horizon_time}
    elif name == 'config4':
        quad = ref_import('vehicles.quadrotor3d')
        vehicle = quad.Quadrotor3D(0.5)
        vehicle.set_initial_conditions([-3, -2, -0.5, 0, 0, 0, 0, 0])
        vehicle.set_terminal_conditions([3, 2, 0.5])
        vehicle.set_options({'safety_distance': 0.1, 'safety_weight': 10})
        environment = env.Environment(room={'shape': shp.Cuboid(8, 6, 8)})
        plate = lambda: shp.Plate(shp.Rectangle(5., 8.), 0.1, orientation=[0., np.pi / 2, 0.])
        trajectory = {'velocity': {'time': [1.5], 'values': [[0, 0, -0.6]]}}
        environment.add_obstacle(obs.Obstacle({'position': [-2, 0, -2]}, shape=plate()))
        environment.add_obstacle(obs.Obstacle({'position': [2, 0, 3.5]}, shape=plate(),
                                              simulation={'trajectories': trajectory}))
        options = {'horizon_time': 5.}
    elif name == 'config_holonomic3d':
        h3 = ref_import('vehicles.holonomic3d')
        vehicle = h3.Holonomic3D(shp.Plate(shp.Rectangle(0.5, 1.), height=0.1))
        vehicle.set_initial_conditions([-2., -2., -2])
        vehicle.set_terminal_conditions([2., 2., -2])
        environment = env.Environment(room={'shape': shp.Cube(5.)})
        environment.add_obstacle(obs.Obstacle(
            {'position': [0., 0., -1.5]}, shape=shp.Cuboid(width=0.5, depth=4., height=2.)))
        trajectories = {'velocity': {'time': [4.], 'values': [[0.0, 0.0, 1.]]}}
        environment.add_obstacle(obs.Obstacle(
            {'position': [1., 1., -2.25]}, shape=shp.RegularPrisma(0.25, 0.25, 6),
            simulation={'trajectories': trajectories}))
        options = {'hard_term_con': True, 'horizon_time': 12}
    elif name == 'config_quadrotor2d':
        q2 = ref_import('vehicles.quadrotor')
        vehicle = q2.Quadrotor()
        vehicle.set_options({'safety_distance': 0.1})
        vehicle.set_initial_conditions([-4., -4., 0., 0., 0.])
        vehicle.set_terminal_conditions([4., 4.])
        environment = env.Environment(room={'shape': shp.Square(10.)})
        environment.add_obstacle(obs.Obstacle({'position': [-0.6, -5.4]},
                                              shape=shp.Rectangle(width=0.2, height=12.)))
        options = {'horizon_time': 5}
    elif name in ('config_dubins', 'config_dubins_plain', 'config_dubins_rect',
                  'config_dubins_exact'):
        db = ref_import('vehicles.dubins')
        bounds = {'vmax': 0.7, 'wmax': np.pi / 3., 'wmin': -np.pi / 3.}
        if name == 'config_dubins':
            vehicle = db.Dubins(bounds=bounds, options={'substitution': True})
        elif name == 'config_dubins_plain':
            vehicle = db.Dubins(bounds=bounds, options={'substitution': False})
        elif name == 'config_dubins_rect':
            vehicle = db.Dubins(shapes=shp.Rectangle(width=0.4, height=0.2), bounds=bounds,
                                options={'substitution': False})
            vehicle.define_knots(knot_intervals=5)
        else:
            vehicle = db.Dubins(bounds=bounds, options={'substitution': True,
                                                        'exact_substitution': True})
            vehicle.define_knots(knot_intervals=5)
        vehicle.set_initial_conditions([0., 0., 0.])
        vehicle.set_terminal_conditions([3., 3., 0.])
        environment = env.Environment(room={'shape': shp.Square(5.), 'position': [1.5, 1.5]})
        trajectories = {'velocity': {'time': [0.5], 'values': [[0.25, 0.0]]}}
        environment.add_obstacle(obs.Obstacle({'position': [1., 1.]}, shape=shp.Circle(0.5),
                                              simulation={'trajectories': trajectories}))
        options = {}
    elif name == 'config_bicycle':
        bi = ref_import('vehicles.bicycle')
        vehicle = bi.Bicycle(length=0.4, options={'plot_type': 'car', 'substitution': False})
        vehicle.define_knots(knot_intervals=5)
        vehicle.set_initial_conditions([0., 0., 0., 0.])
        vehicle.set_terminal_conditions([3., 3., 0.])
        environment = env.Environment(room={'shape': shp.Square(5.), 'position': [1.5, 1.5]})
        trajectories = {'velocity': {'time': [0.5], 'values': [[0.3, 0.0]]}}
        environment.add_obstacle(obs.Obstacle({'position': [1., 1.]}, shape=shp.Circle(0.5),
                                              simulation={'trajectories': trajectories}))
        options = {}
    elif name == 'config_agv':
        ag = ref_import('vehicles.agv')
        vehicle = ag.AGV(length=0.8, options={'plot_type': 'agv'})
        vehicle.define_knots(knot_intervals=5)
        vehicle.set_initial_conditions([0.8, -0.05, 0., 0.])
        vehicle.set_terminal_conditions([2.45, -0.35, 0.])
        environment = env.Environment(room={'shape': shp.Rectangle(width=4, height=1),
                                            'position': [2, 0.]})
        rectangle = shp.Rectangle(width=0.8, height=0.2)
        environment.add_obstacle(obs.Obstacle({'position': [1., -0.35]}, shape=rectangle))
        environment.add_obstacle(obs.Obstacle({'position': [3.4, -0.35]}, shape=rectangle))
        options = {}
    elif name == 'config_quadrotor3d_simple':
        qs = ref_import('vehicles.quadrotor3d_simple')
        vehicle = qs.SimpleQuadrotor3D(0.5)
        vehicle.set_initial_conditions(np.array([-3, -2, -0.5, 0, 0, 0, 0, 0], float))
        vehicle.set_terminal_conditions([3, 2, 0.5])
        vehicle.set_options({'safety_distance': 0.1, 'safety_weight': 10})
        environment = env.Environment(room={'shape': shp.Cuboid(8, 6, 8)})
        plate = lambda: shp.Plate(shp.Rectangle(5., 8.), 0.1, orientation=[0., np.pi / 2, 0.])
        trajectory = {'velocity': {'time': [1.5], 'values': [[0, 0, -0.6]]}}
        environment.add_obstacle(obs.Obstacle({'position': [-2, 0, -2]}, shape=plate()))
        environment.add_obstacle(obs.Obstacle({'position': [2, 0, 3.5]}, shape=plate(),
                                              simulation={'trajectories': trajectory}))
        options = {}
    elif name in ('config_freeT', 'config_freeT_moving', 'config_freeT_safety', 'config_dubins_freeT'):
        # free end time: the reference defines T twice under one name, as a parameter (handed
        # to the vehicle / environment rows) and as the variable of the objective
        # (point2point.py:53-62, 281-284); both carry the same registry value here
        if name == 'config_dubins_freeT':
            db = ref_import('vehicles.dubins')
            vehicle = db.Dubins(bounds={'vmax': 0.7, 'wmax': np.pi / 3., 'wmin': -np.pi / 3.},
                                options={'substitution': True})
            vehicle.define_knots(knot_intervals=5)
            vehicle.set_initial_conditions([0., 0., 0.])
            vehicle.set_terminal_conditions([3., 3., 0.])
            environment = env.Environment(room={'shape': shp.Square(5.), 'position': [1.5, 1.5]})
            trajectories = {'velocity': {'time': [0.5], 'values': [[0.25, 0.0]]}}
            environment.add_obstacle(obs.Obstacle({'position': [1., 1.]}, shape=shp.Circle(0.5),
                                                  simulation={'trajectories': trajectories}))
        elif name == 'config_freeT_safety':
            vehicle = hol.Holonomic()
            vehicle.set_options({'safety_distance': 0.1})
            vehicle.set_initial_conditions([-1.5, -1.5])
            vehicle.set_terminal_conditions([2., 2.])
            environment = env.Environment(room={'shape': shp.Square(5.)})
            environment.add_obstacle(obs.Obstacle({'position': [0.3, 0.2]}, shape=shp.Circle(0.5)))
        else:
            vehicle = hol.Holonomic()
            vehicle.set_initial_conditions([-1.5, -1.5])
            vehicle.set_terminal_conditions([2., 2.])
            environment = env.Environment(room={'shape': shp.Square(5.)})
            rectangle = shp.Rectangle(width=3., height=0.2)
            environment.add_obstacle(obs.Obstacle({'position': [-2.1, -0.5]}, shape=rectangle))
            environment.add_obstacle(obs.Obstacle({'position': [1.7, -0.5]}, shape=rectangle))
            trajectories = {'velocity': {'time': [3., 4.], 'values': [[-0.15, 0.0], [0., 0.15]]}}
            environment.add_obstacle(obs.Obstacle(
                {'position': [1.5, 0.5]}, shape=shp.Circle(0.4),
                simulation={'trajectories': trajectories} if name == 'config_freeT_moving' else None))
        problem = p2p.Point2point(vehicle, environment, options={'verbose': 0}, freeT=True)
        problem.father.reset()
        problem.construct()
        return problem
    elif name == 'config_trailer':
        db, tr = ref_import('vehicles.dubins'), ref_import('vehicles.trailer')
        vehicle = db.Dubins(shapes=shp.Circle(0.2),
                            bounds={'vmax': 0.8, 'wmax': np.pi / 3., 'wmin': -np.pi / 3.})
        vehicle.define_knots(knot_intervals=9)
        vehicle.set_initial_conditions([0., 0., 0.])
        vehicle.set_terminal_conditions([3.4, 3., 0.])
        trailer = tr.Trailer(lead_veh=vehicle, shapes=shp.Rectangle(0.2, 0.2), l_hitch=0.6,
                             bounds={'tmax': np.pi / 4., 'tmin': -np.pi / 4.})
        trailer.define_knots(knot_intervals=9)
        trailer.set_initial_conditions(0.)
        trailer.set_terminal_conditions(0.)
        environment = env.Environment(room={'shape': shp.Square(5.), 'position': [1.5, 1.5]})
        problem = p2p.Point2point(trailer, environment, options={'verbose': 0}, freeT=True)
        problem.father.add(vehicle)            # examples/p2p_trailer.py:43-47
        problem.vehicles.append(vehicle)
        vehicle.to_simulate = False
        problem.father.reset()
        problem.construct()
        return problem
    elif name == 'config_warehouse':
        vehicle = hol.Holonomic(options={'syslimit': 'norm_2', 'safety_distance': 0.1})
        vehicle.define_knots(knot_intervals=10)
        vehicle.set_initial_conditions([0., 0.])
        vehicle.set_terminal_conditions([6., 3.5])
        environment = env.Environment(room={'shape': shp.Rectangle(width=7., height=4.5),
                                            'position': [3., 1.75]})
        rectangle = shp.Rectangle(width=1., height=1.)
        for pos in ([1., 1.], [3., 1.], [5., 1.], [1., 2.5], [3., 2.5], [5., 2.5]):
            environment.add_obstacle(obs.Obstacle({'position': pos}, shape=rectangle))
        trajectories1 = {'velocity': {'time': [0, 2], 'values': [[0., 0.0], [0., 0.15]]}}
        trajectories2 = {'velocity': {'time': [0, 2], 'values': [[0., 0.0], [0., -0.1]]}}
        environment.add_obstacle(obs.Obstacle({'position': [4., 2.5]}, shape=shp.Circle(0.5),
                                              simulation={'trajectories': trajectories2}))
        environment.add_obstacle(obs.Obstacle({'position': [2., 1.]}, shape=shp.Circle(0.5),
                                              simulation={'trajectories': trajectories1}))
        problem = p2p.Point2point(vehicle, environment, options={'verbose': 0}, freeT=True)
        problem.father.reset()
        problem.construct()
        return problem
    elif name == 'config_revolving_door_diffdrive':
        db = ref_import('vehicles.dubins')
        vehicle = db.Dubins(bounds={'vmax': 0.7, 'wmin': -30., 'wmax': 30.})
        vehicle.define_knots(knot_intervals=6)
        vehicle.set_initial_conditions([0., -2.0, np.pi / 2])
        vehicle.set_terminal_conditions([-1.5, 2.0, np.pi / 2])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        beam1 = shp.Beam(width=2.2, height=0.2)
        environment.add_obstacle(obs.Obstacle({'position': [-2., 0.]}, shape=beam1))
        environment.add_obstacle(obs.Obstacle({'position': [2., 0.]}, shape=beam1))
        beam2 = shp.Beam(width=1.4, height=0.2)
        horizon_time = 15.
        omega = 0.1 * 1. * (2 * np.pi / horizon_time)
        for orient in (0. + np.pi / 4., 0.5 * np.pi + np.pi / 4.):
            environment.add_obstacle(obs.Obstacle(
                {'position': [0., 0.], 'velocity': [0., 0.], 'orientation': orient,
                 'angular_velocity': omega}, shape=beam2, simulation={},
                options={'horizon_time': horizon_time}))
        options = {'horizon_time': horizon_time, 'hard_term_con': True}
    elif name == 'config_revolving_door_quadrotor':
        q2 = ref_import('vehicles.quadrotor')
        vehicle = q2.Quadrotor(radius=0.1, bounds={'u1max': 10, 'u2max': 8})
        vehicle.define_knots(knot_intervals=10)
        vehicle.set_initial_conditions([0., -2.0])
        vehicle.set_terminal_conditions([-0.5, 2.0])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        beam1 = shp.Beam(width=2.2, height=0.2)
        environment.add_obstacle(obs.Obstacle({'position': [-2., 0.]}, shape=beam1))
        environment.add_obstacle(obs.Obstacle({'position': [2., 0.]}, shape=beam1))
        beam2 = shp.Beam(width=1.4, height=0.2)
        horizon_time = 10.
        omega = 0.45 * 1. * (2 * np.pi / horizon_time)
        for orient in (0. + np.pi / 4, 0.5 * np.pi + np.pi / 4):
            environment.add_obstacle(obs.Obstacle(
                {'position': [0., 0.], 'velocity': [0., 0.], 'orientation': orient,
                 'angular_velocity': omega}, shape=beam2, simulation={},
                options={'horizon_time': horizon_time}))
        options = {'horizon_time': horizon_time}
    elif name == 'config_free_end':
        vehicle = hol.Holonomic()
        vehicle.set_options({'safety_distance': 0.1})
        vehicle.set_initial_conditions([-1.5, -1.5])
        vehicle.set_terminal_conditions([2., 2.])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        environment.add_obstacle(obs.Obstacle({'position': [1.5, -1]}, shape=shp.Circle(0.5)))
        problem = p2p.FreeEndPoint2point(vehicle, environment, {'verbose': 0}, {vehicle: [0, 1]})
        problem.father.reset()
        problem.construct()
        return problem
    elif name == 'config_interveh':
        N = 2
        vehicles = [hol.Holonomic() for _ in range(N)]
        for k, vehicle in enumerate(vehicles):
            vehicle.set_initial_conditions([1.5 * np.cos((k * 2. * np.pi) / N),
                                            1.5 * np.sin((k * 2. * np.pi) / N)])
            vehicle.set_terminal_conditions([-1.5 * np.cos((k * 2. * np.pi) / N),
                                             -1.5 * np.sin((k * 2. * np.pi) / N)])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        problem = p2p.Point2point(vehicles, environment, options={'verbose': 0}, freeT=False)
        problem.set_options({'inter_vehicle_avoidance': True})
        problem.father.reset()
        problem.construct()
        return problem
    elif name in ('config_formation_central', 'config_formation_central_example'):
        fl = ref_import('vehicles.fleet')
        fc = ref_import('problems.formation_central')
        N = 4
        vehicles = [hol.Holonomic() for _ in range(N)]
        for k, vehicle in enumerate(vehicles):
            vehicle.set_initial_conditions([-1. - 0.5 * N * 0.5 + 0.5 * k, -1.5])
        fleet = fl.Fleet(vehicles)
        configuration = shp.RegularPolyhedron(0.2, N, np.pi / 4.).vertices.T
        fleet.set_configuration(configuration.tolist())
        fleet.set_terminal_conditions((np.array([2., 2.]) + configuration).tolist())
        environment = env.Environment(room={'shape': shp.Square(5.)})
        rectangle = shp.Rectangle(width=3., height=0.2)
        environment.add_obstacle(obs.Obstacle({'position': [-1.8, 0.5]}, shape=rectangle))
        environment.add_obstacle(obs.Obstacle({'position': [1.7, 0.5]}, shape=rectangle))
        problem = fc.FormationPoint2pointCentral(
            fleet, environment, options={'verbose': 0, 'horizon_time': 15, 'soft_formation': True,
                                         'soft_formation_weight': 100})
        if name.endswith('_example'):
            problem.set_options({'inter_vehicle_avoidance': True})
        problem.father.reset()
        problem.construct()
        return problem
    elif name == 'config_holonomic_orient':
        ho = ref_import('vehicles.holonomicorient')
        vehicle = ho.HolonomicOrient()
        vehicle.set_options({'reg_type': 'norm_1', 'reg_weight': 10})
        vehicle.set_initial_conditions([-1.5, -1.5, np.pi / 4.])
        vehicle.set_terminal_conditions([2., 2., np.pi / 2.])
        environment = env.Environment(room={'shape': shp.Square(5.)})
        rectangle = shp.Rectangle(width=3., height=0.2)
        environment.add_obstacle(obs.Obstacle({'position': [-1.8, -0.5]}, shape=rectangle))
        environment.add_obstacle(obs.Obstacle({'position': [1.7, -0.5]}, shape=rectangle))
        trajectories = {'velocity': {'time': [3., 4.], 'values': [[-0.15, 0.0], [0., 0.15]]}}
        environment.add_obstacle(obs.Obstacle({'position': [1.5, 0.5]}, shape=shp.Circle(0.4),
                                              simulation={'trajectories': trajectories}))
        options = {}
    else:
        raise ValueError(name)
    opts = {'verbose': 0}
    opts.update(options)
    problem = p2p.Point2point(vehicle, environment, options=opts, freeT=False)
    problem.father.reset()
    problem.construct()
    return problem


def flatten(problem):
    """Flat layout, values and rows of the reference problem (optilayer.py:225-272 order)."""
    children = list(problem.father.children.values())
    var, par, rows, lb, ub = [], [], [], [], []
    obj = 0.
    for ch in children:
        for nm, v in ch._variables.items():
            var.append((ch.label, nm, v))
        for nm, v in ch._parameters.items():
            par.append((ch.label, nm, v))
        for nm, con in ch._constraints.items():
            expr = con[0]
            vals = expr.column() if isinstance(expr, MX) else np.atleast_1d(np.asarray(expr, float))
            rows += list(vals)
            lb += list(np.ones(len(vals)) * con[1])
            ub += list(np.ones(len(vals)) * con[2])
        o = ch._objective
        obj = obj + (float(o) if isinstance(o, MX) else o)
    return var, par, np.array(rows, float), np.array(lb, float), np.array(ub, float), float(obj)


def host_values(problem, par, var, current_time):
    """What the reference's host code feeds the solver: the parameter vector of
    OptiFather.set_parameters (optilayer.py:427-445, values from every child's
    set_parameters) and the initial guess of the vehicle splines
    (Point2pointProblem.reinitialize -> vehicle.get_init_spline_value)."""
    children = list(problem.father.children.values())
    merged = {}
    for ch in children:
        for owner, dic in ch.set_parameters(current_time).items():
            merged.setdefault(owner, {}).update(dic)
    P = []
    for ch in children:
        for nm, v in ch._parameters.items():
            val = merged.get(ch, {}).get(nm, ch._values[nm])
            P.append(np.broadcast_to(np.asarray(val, float).reshape(-1, order='F') if np.ndim(val) else
                                     np.asarray(val, float), (v.a.size,)).reshape(-1))
    X0 = []
    for ch in children:
        for nm, v in ch._variables.items():
            val = np.zeros(v.a.shape)
            init = ch._values.get(nm)            # define_variable(..., value=...): T = 10
            if init is not None and np.size(init) == v.a.size:
                val = np.asarray(init, float).reshape(v.a.shape)
            if nm == 'splines_seg0':
                val = np.asarray(ch.get_init_spline_value()[0], float).reshape(v.a.shape)
            X0.append(val.reshape(-1, order='F'))
    return np.concatenate(P), np.concatenate(X0)


def trajectories(problem, horizon, seed):
    """Post-solve extraction by the reference (Vehicle.store -> concat_splines,
    splines2signals, sample_splines; vehicle.py:250-300): state / input trajectories of
    a perturbed initial-guess spline, sampled from a time inside the first knot interval."""
    spl = ref_import('basics.spline')
    vehicle = problem.vehicles[0]
    rng = np.random.default_rng(seed)
    C = np.asarray(vehicle.get_init_spline_value()[0], float)
    C = C + 0.05 * rng.standard_normal(C.shape)
    if type(vehicle).__name__ in ('Quadrotor3D',):
        C[:, 0] += 9.81                      # thrust spline around hover
    if type(vehicle).__name__ == 'Dubins':
        C[:, 0] = np.abs(C[:, 0]) + 0.2      # forward speed
    splines = [spl.BSpline(vehicle.basis, C[:, k]) for k in range(C.shape[1])]
    sample_time, t_rel = 0.01, 0.17
    n_samp = int(round((horizon - t_rel) / sample_time, 6)) + 1
    time_axis = np.linspace(t_rel, t_rel + (n_samp - 1) * sample_time, n_samp)
    # (the reference's err_* plot signals need a solved problem: switch them off for this call)
    subst = vehicle.options.get('substitution')
    if subst is not None:
        vehicle.options['substitution'] = False
    vehicle.store(1.3, sample_time, [splines], horizon, time_axis)
    if subst is not None:
        vehicle.options['substitution'] = subst
    tr = vehicle.trajectories
    keys = sorted(k for k in tr if k not in ('time', 'pose', 'splines', 'fleet_center')
                  and not k.startswith('err_'))
    return C, time_axis, {k: np.atleast_2d(np.asarray(tr[k], float)) for k in keys}


def obstacle_motion(problem, total_time, update_time=0.1, sample_time=0.01):
    """Obstacle states after every update of the reference's simulator
    (Environment.simulate -> ObstaclexD.simulate, obstacle.py:246-264, 375-386) and the
    parameters the obstacles report then (set_parameters, obstacle.py:142-155, 345-348)."""
    env = problem.environment
    rows = []
    t = 0.
    for _ in range(int(round(total_time / update_time))):
        env.simulate(update_time, sample_time)
        t = np.round(t + update_time, 6)
        row = []
        for o in env.obstacles:
            row += list(o.signals['position'][:, -1]) + list(o.signals['velocity'][:, -1])
            pars = o.set_parameters(t)[o]
            pars = {k: v for k, v in pars.items() if k in o._parameters}   # what the NLP receives
            if 'theta' in pars:
                row += [o.signals['orientation'][0, -1]]
            for key in sorted(pars):
                row += list(np.atleast_1d(np.asarray(pars[key], float)).reshape(-1))
        rows.append(row)
    return np.array(rows, float)


def shape_zoo(shp):
    """One instance of every shape class both code bases provide (same arguments)."""
    return {
        'circle': shp.Circle(0.4),
        'rectangle': shp.Rectangle(width=3., height=0.2),
        'rectangle_rot': shp.Rectangle(width=0.5, height=1.2, orientation=0.3),
        'square': shp.Square(0.7),
        'beam': shp.Beam(width=1.4, height=0.2),
        'beam_rot': shp.Beam(width=2.2, height=0.2, orientation=0.5 * np.pi),
        'regpoly8': shp.RegularPolyhedron(2.5, 8),
        'regpoly5_rot': shp.RegularPolyhedron(0.6, 5, np.pi / 7.),
        'sphere': shp.Sphere(0.5),
        'cuboid': shp.Cuboid(width=0.5, depth=4., height=2.),
        'cuboid_rot': shp.Cuboid(width=0.5, depth=1., height=2., orientation=[0.1, 0.4, -0.3]),
        'cube': shp.Cube(5.),
        'plate': shp.Plate(shp.Rectangle(5., 8.), 0.1, orientation=[0., np.pi / 2, 0.]),
        'prisma': shp.RegularPrisma(0.25, 0.25, 6),
    }


BASE_NAMES = ('config1', 'config2', 'config4', 'config5', 'config_holonomic3d',
              'config_quadrotor2d', 'config_dubins')
# second set of fixture files (model_golden_ext1..3.npz, `--ext`): formulations whose rows multiply the
# intermediates by decision variables
EXT_NAMES = ('config_dubins_plain', 'config_dubins_rect', 'config_dubins_exact',
             'config_holonomic_orient', 'config_bicycle', 'config_agv',
             'config_quadrotor3d_simple', 'config_formation_central', 'config_interveh', 'config_free_end',
             'config_freeT', 'config_freeT_moving', 'config_freeT_safety', 'config_dubins_freeT',
             'config_trailer', 'config_formation_central_example', 'config_warehouse',
             'config_revolving_door_diffdrive', 'config_revolving_door_quadrotor')


def main(ext=False):
    global REG
    install_stubs()
    out, owner = {}, {}
    n_samples = 3
    for name in (EXT_NAMES if ext else BASE_NAMES):
        Xs, Ps, Gs, Fs = [], [], [], []
        for k in range(n_samples):
            REG = Registry(seed=1000 * k + 7)
            horizon = {'config4': 5., 'config_quadrotor2d': 5., 'config_holonomic3d': 12.,
                       'config_formation_central': 15.,
                       'config_formation_central_example': 15.,
                       'config_revolving_door_diffdrive': 15.}.get(name, 10.)
            # T is the horizon of the scenario, t a time inside the first knot interval
            REG.fixed = {'T': horizon, 't': 0.037 * horizon * (k + 1)}
            if 'freeT' in name or name in ('config_trailer', 'config_warehouse'):
                # t is 0 (point2point.py:300-306); T -- parameter, variable and the vehicles'
                # placeholders of that name -- one value per sample
                REG.fixed = {'t': 0., 'T': 6.3 + 1.7 * k}
            # labels restart for every build so that the layout strings are comparable
            opt = ref_import('basics.optilayer')
            for cls in list(opt.OptiChild.__subclasses__()) + [opt.OptiChild]:
                if hasattr(cls, '_labels'):
                    cls._labels = []
            problem = build_reference(name)
            var, par, g, lb, ub, f = flatten(problem)
            Xs.append(np.concatenate([v.column() for _, _, v in var]))
            Ps.append(np.concatenate([v.column() for _, _, v in par]))
            Gs.append(g)
            Fs.append(f)
        C, tax, tr = trajectories(problem, horizon, 11)
        out[name + '_traj_C'], out[name + '_traj_time'] = C, tax
        for key, val in tr.items():
            out[name + '_traj_' + key] = val
        out[name + '_traj_keys'] = np.array(sorted(tr))
        t_host = 0.37
        if name in ('config1', 'config4', 'config5', 'config_holonomic3d', 'config_dubins') + EXT_NAMES:
            host = host_values(problem, par, var, t_host)
            out[name + '_obst'] = obstacle_motion(problem, 5.0)
            out[name + '_host_P'], out[name + '_host_X0'] = host
            print(name, 'reference layout: n', len(Xs[0]), 'm', len(Gs[0]), 'n_par', len(Ps[0]))
            continue_flag = True
        else:
            continue_flag = False
        if not continue_flag:
            out[name + '_host_P'], out[name + '_host_X0'] = host_values(problem, par, var, t_host)
            print(name, 'reference layout: n', len(Xs[0]), 'm', len(Gs[0]), 'n_par', len(Ps[0]))
        out[name + '_X'], out[name + '_P'] = np.array(Xs), np.array(Ps)
        out[name + '_G'], out[name + '_F'] = np.array(Gs), np.array(Fs)
        out[name + '_lb'], out[name + '_ub'] = lb, ub
        out[name + '_var_layout'] = np.array(['%s|%s|%dx%d' % ((lab, nm) + v.a.shape) for lab, nm, v in var])
        out[name + '_par_layout'] = np.array(['%s|%s|%dx%d' % ((lab, nm) + v.a.shape) for lab, nm, v in par])
        owner.update((k, name) for k in out if k not in owner)
    if ext:
        # three files of whole models, each below 1 MB
        for part, names in enumerate((EXT_NAMES[:7], EXT_NAMES[7:15], EXT_NAMES[15:])):
            path = OUT.replace('model_golden.npz', 'model_golden_ext%d.npz' % (part + 1))
            np.savez_compressed(path, **{k: v for k, v in out.items() if owner[k] in names})
            print('wrote', path, os.path.getsize(path), 'bytes')
        return
    # Fleet of the formation examples (vehicles/fleet.py: set_configuration, neighbours)
    hol, fl = ref_import('vehicles.holonomic'), ref_import('vehicles.fleet')
    shp = ref_import('basics.shape')
    for n_agents in (4, 6):
        conf = shp.RegularPolyhedron(0.2, n_agents, np.pi / 4.).vertices.T
        fleet = fl.Fleet([hol.Holonomic() for _ in range(n_agents)])
        fleet.set_configuration(conf.tolist())
        out['fleet%d_rel_pos_c' % n_agents] = np.array([v.rel_pos_c for v in fleet.vehicles], float)
        out['fleet%d_nghb' % n_agents] = np.array(
            [[fleet.vehicles.index(w) for w in fleet.get_neighbors(v)] for v in fleet.vehicles])
    # shapes (basics/shape.py): checkpoints + radii, canvas limits, room half-planes
    for key, shape in shape_zoo(shp).items():
        chck, rad = shape.get_checkpoints()
        out['shape_%s_chck' % key] = np.array(chck, float)
        out['shape_%s_rad' % key] = np.array(rad, float)
        out['shape_%s_lims' % key] = np.array(shape.get_canvas_limits(), float)
        if hasattr(shape, 'get_hyperplanes') and shape.n_dim == 2 and hasattr(shape, 'vertices'):
            hyp = shape.get_hyperplanes(position=[0.3, -0.2])
            out['shape_%s_hyp' % key] = np.array(
                [np.r_[np.asarray(h['a'], float).reshape(-1), float(np.asarray(h['b']).reshape(-1)[0])]
                 for _, h in sorted(hyp.items())])
    np.savez_compressed(OUT, **out)
    print('wrote', OUT)


if __name__ == '__main__':
    main(ext='--ext' in sys.argv)
