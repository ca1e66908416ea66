"""ctypes loader for the CPU oracle (oracle/liboracle_strict.so) — test infrastructure only."""
import ctypes as C
import os
import subprocess

import numpy as np

from bio_ik_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")


def build_oracle():
    subprocess.run(["make", "-C", ORACLE_DIR, "-s"], check=True)


class Oracle:
    def __init__(self, variant="strict"):
        path = os.path.join(ORACLE_DIR, f"liboracle_{variant}.so")
        if not os.path.exists(path):
            build_oracle()
        self.lib = lib = C.CDLL(path)
        dp, ip, up = _abi.c_double_p, _abi.c_int32_p, _abi.c_uint32_p
        lib.oracle_last_error.restype = C.c_char_p
        lib.oracle_tables_create.argtypes = [C.c_uint32]
        lib.oracle_tables_create.restype = C.c_void_p
        lib.oracle_tables_destroy.argtypes = [C.c_void_p]
        lib.oracle_tables_uniform.argtypes = [C.c_void_p]
        lib.oracle_tables_uniform.restype = dp
        lib.oracle_tables_gauss.argtypes = [C.c_void_p]
        lib.oracle_tables_gauss.restype = dp
        lib.oracle_xorshift.argtypes = [C.c_int, C.POINTER(C.c_uint64)]
        lib.oracle_minstd_uniform.argtypes = [C.c_uint32, C.c_int, dp]
        lib.oracle_minstd_normal.argtypes = [C.c_uint32, C.c_int, dp]
        lib.oracle_minstd_index.argtypes = [C.c_uint32, C.c_uint64, C.c_int, C.POINTER(C.c_uint64)]
        lib.oracle_sincos.argtypes = [C.c_int, dp, dp, dp]
        lib.oracle_acos.argtypes = [C.c_int, dp, dp]
        lib.oracle_concat.argtypes = [dp, dp, dp]
        lib.oracle_invert.argtypes = [dp, dp]
        lib.oracle_change.argtypes = [dp, dp, dp, dp]
        lib.oracle_fk_batch.argtypes = [C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem), C.c_int, C.c_int, dp, dp, dp]
        lib.oracle_approx_batch.argtypes = [C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem), C.c_int, dp, dp, ip, dp]
        lib.oracle_approx_fitness_batch.argtypes = [C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem), C.c_int, C.c_int, dp, dp, dp, dp, dp, dp]
        lib.oracle_approx_frames_batch.argtypes = [C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem), C.c_int, C.c_int, dp, dp, dp]
        lib.oracle_set_component_flags.argtypes = [C.c_int]
        lib.oracle_solve_batch.argtypes = [C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem), C.POINTER(_abi.BioikSolverCfg), C.c_void_p, C.c_int, dp, dp, up,
                                           C.c_int, C.c_int, C.c_int, C.c_int, dp, dp, ip, ip, dp, dp, dp]
        lib.oracle_select_islands.argtypes = [C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem), C.c_int, C.c_int, dp, dp, dp, dp, ip, ip, C.c_int, dp, dp, ip, ip, ip]
        lib.oracle_solve_islands.argtypes = [C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem), C.POINTER(_abi.BioikSolverCfg), C.c_void_p, C.c_int, C.c_int, dp, dp, up, C.c_int,
                                             C.c_int, C.c_int, C.c_int, C.c_int, dp, dp, ip, ip, ip, dp, dp, ip, ip]
        lib.oracle_hardware_threads.restype = C.c_int
        self._tables = {}

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("oracle: " + self.lib.oracle_last_error().decode())

    def tables(self, seed):
        if seed not in self._tables:
            self._tables[seed] = self.lib.oracle_tables_create(seed)
        return self._tables[seed]

    def table_arrays(self, seed, n=None):
        t = self.tables(seed)
        n = n or (1 << 23)
        u = np.ctypeslib.as_array(self.lib.oracle_tables_uniform(t), shape=(1 << 23,))[:n]
        g = np.ctypeslib.as_array(self.lib.oracle_tables_gauss(t), shape=(1 << 23,))[:n]
        return u, g

    def sincos(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        s, c = np.empty_like(x), np.empty_like(x)
        self.lib.oracle_sincos(len(x), _abi.dptr(x), _abi.dptr(s), _abi.dptr(c))
        return s, c

    def acos(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty_like(x)
        self.lib.oracle_acos(len(x), _abi.dptr(x), _abi.dptr(out))
        return out

    def fk(self, robot, problem, variables, libm=False, links=False):
        v = np.ascontiguousarray(variables, dtype=np.float64).reshape(-1, robot.n_vars)
        B, T = v.shape[0], len(problem.tip_link_indices)
        out = np.zeros((B, T, 7))
        lf = np.zeros((B, len(robot.links), 7)) if links else None
        r, p = robot.to_abi(), problem.to_abi()
        self._check(self.lib.oracle_fk_batch(C.byref(r), C.byref(p), int(libm), B, _abi.dptr(v), _abi.dptr(out), _abi.dptr(lf)))
        return (out, lf) if links else out

    def approx(self, robot, problem, variables, jacobian=False):
        v = np.ascontiguousarray(variables, dtype=np.float64).reshape(-1, robot.n_vars)
        B, T, n = v.shape[0], len(problem.tip_link_indices), len(problem.active_variables)
        delta = np.zeros((B, T, n, 7))
        mask = np.zeros((B, T, n), dtype=np.int32)
        jac = np.zeros((B, 6 * T, n))
        r, p = robot.to_abi(), problem.to_abi()
        self._check(self.lib.oracle_approx_batch(C.byref(r), C.byref(p), B, _abi.dptr(v), _abi.dptr(delta), _abi.iptr(mask), _abi.dptr(jac)))
        return (delta, mask, jac) if jacobian else (delta, mask)

    def approx_fitness(self, robot, problem, goal_params, seeds, base, genotypes):
        base = np.ascontiguousarray(base, dtype=np.float64).reshape(-1, robot.n_vars)
        B, n = base.shape[0], len(problem.active_variables)
        g = np.ascontiguousarray(genotypes, dtype=np.float64).reshape(B, -1, n)
        M = g.shape[1]
        seeds = np.ascontiguousarray(seeds, dtype=np.float64).reshape(B, robot.n_vars)
        gp = None if goal_params is None else np.ascontiguousarray(goal_params, dtype=np.float64).reshape(B, problem.n_goals, _abi.GOAL_NPARAM)
        prim, sec = np.zeros((B, M)), np.zeros((B, M))
        r, p = robot.to_abi(), problem.to_abi()
        self._check(self.lib.oracle_approx_fitness_batch(C.byref(r), C.byref(p), B, M, _abi.dptr(gp), _abi.dptr(seeds), _abi.dptr(base), _abi.dptr(g), _abi.dptr(prim), _abi.dptr(sec)))
        return prim, sec

    def approx_frames(self, robot, problem, base, genotypes):
        base = np.ascontiguousarray(base, dtype=np.float64).reshape(-1, robot.n_vars)
        B, n, T = base.shape[0], len(problem.active_variables), len(problem.tip_link_indices)
        g = np.ascontiguousarray(genotypes, dtype=np.float64).reshape(B, -1, n)
        out = np.zeros((B, g.shape[1], T, 7))
        r, p = robot.to_abi(), problem.to_abi()
        self._check(self.lib.oracle_approx_frames_batch(C.byref(r), C.byref(p), B, g.shape[1], _abi.dptr(base), _abi.dptr(g), _abi.dptr(out)))
        return out

    def component_flags(self, flags):
        """bit0: libm sin/cos (as the reference calls) in fk / approx / approx_fitness / approx_frames"""
        self.lib.oracle_set_component_flags(int(flags))

    def solve(self, robot, problem, cfg, goal_params, seeds, rng_seeds, steps, early_exit=False, flags=0, nthreads=0, table_seed=None):
        seeds = np.ascontiguousarray(seeds, dtype=np.float64).reshape(-1, robot.n_vars)
        B, n = seeds.shape[0], len(problem.active_variables)
        gp = None if goal_params is None else np.ascontiguousarray(goal_params, dtype=np.float64).reshape(B, problem.n_goals, _abi.GOAL_NPARAM)
        rs = np.ascontiguousarray(rng_seeds, dtype=np.uint32)
        res = dict(solutions=np.zeros((B, robot.n_vars)), fitness=np.zeros(B), success=np.zeros(B, dtype=np.int32), steps=np.zeros(B, dtype=np.int32),
                   genes=np.zeros((B, 2, 2, n)), gradients=np.zeros((B, 2, 2, n)), species_fitness=np.zeros((B, 2)))
        r, p = robot.to_abi(), problem.to_abi()
        t = self.tables(cfg.table_seed if table_seed is None else table_seed)
        nthreads = nthreads or min(B, os.cpu_count() or 1)
        self._check(self.lib.oracle_solve_batch(C.byref(r), C.byref(p), C.byref(cfg), t, B, _abi.dptr(gp), _abi.dptr(seeds), _abi.uptr(rs), steps, int(early_exit), flags, nthreads,
                                                _abi.dptr(res["solutions"]), _abi.dptr(res["fitness"]), _abi.iptr(res["success"]), _abi.iptr(res["steps"]),
                                                _abi.dptr(res["genes"]), _abi.dptr(res["gradients"]), _abi.dptr(res["species_fitness"])))
        return res


def oracle_solve_islands(o, robot, problem, cfg, goal_params, seeds, islands, steps, rng_seeds=None, early_exit=0, wrap=True, flags=0, nthreads=0, island_stride=0):
    """the oracle's statement of bioik_solve_islands (lock-step islands, IKParallel's selection, the plugin's wrap);
    early_exit: 0 none, 1 per island, 2 per query (the reference's `finished` flag).  res["runs"] holds the per-island results."""
    seeds = np.ascontiguousarray(seeds, dtype=np.float64).reshape(-1, robot.n_vars)
    Q = seeds.shape[0]
    B = Q * islands
    gp = None if goal_params is None else np.ascontiguousarray(goal_params, dtype=np.float64).reshape(Q, problem.n_goals, _abi.GOAL_NPARAM)
    rs = (1 + np.arange(B)).astype(np.uint32) if rng_seeds is None else np.ascontiguousarray(rng_seeds, dtype=np.uint32).reshape(B)
    res = dict(solutions=np.zeros((Q, robot.n_vars)), fitness=np.zeros(Q), success=np.zeros(Q, dtype=np.int32), island=np.zeros(Q, dtype=np.int32), steps=np.zeros(Q, dtype=np.int32))
    runs = dict(solutions=np.zeros((B, robot.n_vars)), fitness=np.zeros(B), success=np.zeros(B, dtype=np.int32), steps=np.zeros(B, dtype=np.int32))
    r, p = robot.to_abi(), problem.to_abi()
    nthreads = nthreads or min(Q, os.cpu_count() or 1)
    flags = int(flags) | (int(island_stride) << 8)  # bits 8..15: the product's BIOIK_OPT_ISLAND_STREAM_STRIDE
    o._check(o.lib.oracle_solve_islands(C.byref(r), C.byref(p), C.byref(cfg), o.tables(cfg.table_seed), Q, islands, _abi.dptr(gp), _abi.dptr(seeds), _abi.uptr(rs), steps, int(early_exit), int(wrap), flags, nthreads,
                                        _abi.dptr(res["solutions"]), _abi.dptr(res["fitness"]), _abi.iptr(res["success"]), _abi.iptr(res["island"]), _abi.iptr(res["steps"]),
                                        _abi.dptr(runs["solutions"]), _abi.dptr(runs["fitness"]), _abi.iptr(runs["success"]), _abi.iptr(runs["steps"])))
    res["runs"] = runs
    return res


def make_cfg(population=18, generations=8, memetic="q", memetic_iters=8, table_seed=1, device=0):
    c = _abi.BioikSolverCfg()
    c.population, c.generations = population, generations
    c.memetic = ord(memetic) if isinstance(memetic, str) and memetic else int(memetic or 0)
    c.memetic_iters, c.table_seed, c.device = memetic_iters, table_seed, device
    return c


# ---------------------------------------------------------------------------------------------
# the REFERENCE's own code (oracle/_ref/, built by `make -C oracle ref` where /root/reference exists)
# ---------------------------------------------------------------------------------------------
REF_DIR = os.path.join(ORACLE_DIR, "_ref")
REFERENCE_ROOT = "/root/reference"


def ref_lib_path(variant="strict"):
    return os.path.join(REF_DIR, f"libbioik_ref_{variant}.so")


def build_ref():
    """Compile the reference's bio2 solver sources in place (never copied); False when they are not on this machine."""
    if not os.path.exists(os.path.join(REFERENCE_ROOT, "src", "ik_evolution_2.cpp")):
        return os.path.exists(ref_lib_path("strict")) and os.path.exists(ref_lib_path("fast"))
    return subprocess.run(["make", "-C", ORACLE_DIR, "-s", "ref"]).returncode == 0


class Reference:
    """ctypes front of oracle/ref_harness.cpp: same batch contract as Oracle.solve / approx_fitness, executed by
    the reference's IKEvolution2 / RobotFK_Fast / Problem classes."""

    def __init__(self, variant="strict"):
        path = ref_lib_path(variant)
        if not os.path.exists(path) and not build_ref():
            raise FileNotFoundError(path)
        self.lib = lib = C.CDLL(path)
        dp, ip, up = _abi.c_double_p, _abi.c_int32_p, _abi.c_uint32_p
        RP, PP = C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem)
        lib.ref_last_error.restype = C.c_char_p
        lib.ref_solve_batch.argtypes = [RP, PP, C.POINTER(_abi.BioikSolverCfg), C.c_void_p, C.c_int, dp, dp, up, C.c_int, C.c_int, C.c_int, C.c_int, dp, dp, ip, ip, dp, dp, dp]
        lib.ref_approx_fitness_batch.argtypes = [RP, PP, C.c_int, C.c_int, dp, dp, dp, dp, dp, dp, dp, dp, dp]
        lib.ref_effective_goal_params.argtypes = [RP, PP, C.c_int, dp, dp]
        lib.ref_effective_link_origins.argtypes = [RP, dp]
        lib.ref_set_contract_math.argtypes = [C.c_int]
        lib.ref_table.argtypes = [C.c_int, C.c_uint32]
        lib.ref_table.restype = dp

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("reference: " + self.lib.ref_last_error().decode())

    def _gp(self, problem, goal_params, B):
        gp = np.repeat(problem.default_goal_params()[None], B, 0) if goal_params is None else goal_params
        return np.ascontiguousarray(gp, dtype=np.float64).reshape(B, problem.n_goals, _abi.GOAL_NPARAM)

    def contract_math(self, on):
        """True: the reference's sin / cos (forward_kinematics.h:103-104) and ConeGoal's acos use the arithmetic contract's
        det_sincos / det_acos instead of libm; everything else of the reference runs unchanged"""
        self.lib.ref_set_contract_math(int(bool(on)))

    def table(self, which, seed, n=1 << 23):
        return np.ctypeslib.as_array(self.lib.ref_table(which, seed), shape=(1 << 23,))[:n].copy()

    def effective_link_origins(self, robot):
        """[n_links][7]: the link origins as the reference stores them (its Isometry3d -> quaternion conversion, forward_kinematics.h:203)"""
        out = np.zeros((len(robot.links), 7))
        r = robot.to_abi()
        self._check(self.lib.ref_effective_link_origins(C.byref(r), _abi.dptr(out)))
        return out

    def effective_robot(self, robot):
        """copy of `robot` whose link origins are the frames the reference derives from the same robot (its
        Isometry3d -> quaternion conversion, forward_kinematics.h:203); differs from the input by at most an ulp"""
        import copy
        out = self.effective_link_origins(robot)
        src = robot.arrays["link_origin"].reshape(-1, 7)
        sign = np.where((out[:, 3:] * src[:, 3:]).sum(axis=1) < 0, -1.0, 1.0)[:, None]  # q and -q are the same rotation
        assert np.allclose(out[:, :3], src[:, :3], rtol=0, atol=0) and np.allclose(out[:, 3:] * sign, src[:, 3:], rtol=0, atol=1e-14)
        eff = copy.copy(robot)
        eff.arrays = dict(robot.arrays)
        eff.arrays["link_origin"] = np.ascontiguousarray(out.reshape(robot.arrays["link_origin"].shape))
        return eff

    def effective_goal_params(self, robot, problem, goal_params, B):
        """the goal parameters as the reference's goal objects store them (normalising constructors applied)"""
        gp = self._gp(problem, goal_params, B)
        out = np.zeros_like(gp)
        r, p = robot.to_abi(), problem.to_abi()
        self._check(self.lib.ref_effective_goal_params(C.byref(r), C.byref(p), B, _abi.dptr(gp), _abi.dptr(out)))
        return out

    def solve(self, robot, problem, cfg, goal_params, seeds, rng_seeds, steps, early_exit=False, nthreads=0):
        seeds = np.ascontiguousarray(seeds, dtype=np.float64).reshape(-1, robot.n_vars)
        B, n = seeds.shape[0], len(problem.active_variables)
        gp = self._gp(problem, goal_params, B)
        rs = np.ascontiguousarray(rng_seeds, dtype=np.uint32)
        res = dict(solutions=np.zeros((B, robot.n_vars)), fitness=np.zeros(B), success=np.zeros(B, dtype=np.int32), steps=np.zeros(B, dtype=np.int32),
                   genes=np.zeros((B, 2, 2, n)), gradients=np.zeros((B, 2, 2, n)), species_fitness=np.zeros((B, 2)))
        r, p = robot.to_abi(), problem.to_abi()
        nthreads = nthreads or min(B, os.cpu_count() or 1)
        self._check(self.lib.ref_solve_batch(C.byref(r), C.byref(p), C.byref(cfg), None, B, _abi.dptr(gp), _abi.dptr(seeds), _abi.uptr(rs), steps, int(early_exit), 0, nthreads,
                                             _abi.dptr(res["solutions"]), _abi.dptr(res["fitness"]), _abi.iptr(res["success"]), _abi.iptr(res["steps"]),
                                             _abi.dptr(res["genes"]), _abi.dptr(res["gradients"]), _abi.dptr(res["species_fitness"])))
        return res

    def approx_fitness(self, robot, problem, goal_params, seeds, base, genotypes):
        """primary, secondary [B][M]; tip frames [B][T][7]; delta frames [B][T][n][7]; approximated frames [B][M][T][7]"""
        base = np.ascontiguousarray(base, dtype=np.float64).reshape(-1, robot.n_vars)
        B, n, T = base.shape[0], len(problem.active_variables), len(problem.tip_link_indices)
        g = np.ascontiguousarray(genotypes, dtype=np.float64).reshape(B, -1, n)
        M = g.shape[1]
        seeds = np.ascontiguousarray(seeds, dtype=np.float64).reshape(B, robot.n_vars)
        gp = self._gp(problem, goal_params, B)
        out = dict(primary=np.zeros((B, M)), secondary=np.zeros((B, M)), tips=np.zeros((B, T, 7)), delta=np.zeros((B, T, n, 7)), frames=np.zeros((B, M, T, 7)))
        r, p = robot.to_abi(), problem.to_abi()
        self._check(self.lib.ref_approx_fitness_batch(C.byref(r), C.byref(p), B, M, _abi.dptr(gp), _abi.dptr(seeds), _abi.dptr(base), _abi.dptr(g), _abi.dptr(out["primary"]), _abi.dptr(out["secondary"]),
                                                      _abi.dptr(out["tips"]), _abi.dptr(out["delta"]), _abi.dptr(out["frames"])))
        return out
