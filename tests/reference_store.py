"""Answers of the reference's own code, stored, so that the tests that compare with it run from the repository alone.

oracle/_ref/ holds the reference's solver sources compiled in place (oracle/Makefile, targets `ref` and `adapter`); it can only
be built where those sources are.  Every call a test makes to it is answered here from tests/golden/reference/<store>.npz, keyed by
a digest of the call's inputs: a test whose inputs no longer match a recorded call fails instead of comparing with stale numbers.
What the tests compare bit for bit is stored as a Digest (compare with same()); the arrays a test reads as numbers (tolerance
checks, statistics) are named with StoredReference.keep_values and stored whole.

To record the stores again, build oracle/_ref/ and run the tests with BIOIK_RECORD_REFERENCE=<dir>: every call then goes to the
live build and its answers are written to <dir>/<store>.npz (copy them to tests/golden/reference/).  The adapter's calls drive the
GPU, so the stores of the GPU tests are recorded on a GPU machine.
"""
import ctypes as C
import hashlib
import os

import numpy as np

import oracle_lib
from bio_ik_b200 import _abi

STORE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RECORD_ENV = "BIOIK_RECORD_REFERENCE"
_recorded = {}  # store name -> answers recorded by this process


def _feed(h, x):
    if isinstance(x, np.ndarray):
        h.update(f"{x.dtype.str}{x.shape}".encode())
        h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(b"[")
        for y in x:
            _feed(h, y)
        h.update(b"]")
    elif isinstance(x, bytes):
        h.update(x)
    else:
        h.update(repr(x).encode())
    h.update(b";")


def _robot(robot):
    return [robot.arrays[k] for k in sorted(robot.arrays)]


def _problem(problem):
    return [np.asarray(problem._tips), np.asarray(problem._active), bytes(problem._goals), (problem.dpos, problem.drot, problem.dtwist)]


def recording():
    return bool(os.environ.get(RECORD_ENV))


class Digest(str):
    """sha256 (first 128 bits) of an array's dtype, shape and bytes: stands in for a stored array that is only ever compared bit for bit"""

    @classmethod
    def of(cls, a):
        a = np.ascontiguousarray(a)
        h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
        return cls(h.hexdigest()[:32])


def same(candidate, stored):
    """np.array_equal(candidate, stored) for a stored array or its Digest"""
    if isinstance(stored, Digest):
        return Digest.of(candidate) == stored
    return np.array_equal(candidate, stored)


def _xor(a, b):
    """bitwise difference of two float64 arrays of one shape (the effective inputs differ from the given ones by an ulp at most)"""
    return (np.ascontiguousarray(a, dtype=np.float64).view(np.uint64) ^ np.ascontiguousarray(b, dtype=np.float64).view(np.uint64)).view(np.float64)


class _Store:
    def __init__(self, name):
        self.name = name
        if recording():
            self.data = _recorded.setdefault(name, {})
        else:
            path = os.path.join(STORE_DIR, name + ".npz")
            if not os.path.exists(path):
                raise FileNotFoundError(f"{path}: no stored reference answers (record them with {RECORD_ENV}=<dir>)")
            with np.load(path) as f:
                self.data = {k: f[k] for k in f.files if k != "digests"}
                if "digests" in f.files:  # one "<field> <digest>" line per digest
                    self.data.update(dict((k, Digest(d)) for k, d in (line.decode().split() for line in f["digests"])))

    def answer(self, what, inputs, compute, values=None):
        """the recorded answer (dict of arrays or Digests) to call `what` with `inputs`; in record mode `compute()` gives it,
        and only the fields in `values` (all when None) are stored as arrays"""
        h = hashlib.sha256()
        _feed(h, inputs)
        key = f"{what}-{h.hexdigest()[:20]}"
        if recording():
            out = {k: np.asarray(v) for k, v in compute().items()}
            out = {k: v if values is None or k in values else Digest.of(v) for k, v in out.items()}
            for k, v in out.items():
                self.data[f"{key}.{k}"] = v
            return out
        out = {k[len(key) + 1:]: v for k, v in self.data.items() if k.startswith(key + ".")}
        if not out:
            raise KeyError(f"store {self.name}: no recorded answer of {what} for these inputs; record it again with {RECORD_ENV}=<dir>")
        return out

    def close(self):
        if recording():
            out = os.environ[RECORD_ENV]
            os.makedirs(out, exist_ok=True)
            arrays = {k: v for k, v in self.data.items() if not isinstance(v, Digest)}
            digests = [f"{k} {v}".encode() for k, v in self.data.items() if isinstance(v, Digest)]
            if digests:
                arrays["digests"] = np.array(digests)
            np.savez_compressed(os.path.join(out, self.name + ".npz"), **arrays)


_live = {}


def _live_reference():
    if "ref" not in _live:
        _live["ref"] = oracle_lib.Reference("strict")
    return _live["ref"]


class StoredReference(oracle_lib.Reference):
    """oracle_lib.Reference (the strict build) answered from a store: same methods; the outputs of solve and approx_fitness are
    Digests except the fields named with keep_values"""

    def __init__(self, name):
        self.store = _Store(name)
        self.live = _live_reference() if recording() else None
        self.math = False
        self.values = set()

    def close(self):
        self.contract_math(False)
        self.store.close()

    def keep_values(self, *fields):
        """store these output fields as arrays: the test reads them as numbers"""
        self.values |= set(fields)

    def _answer(self, what, inputs, compute, values=None):
        return self.store.answer(what, [self.math, inputs], lambda: compute(self.live), values=self.values if values is None else values)

    def contract_math(self, on):
        self.math = bool(on)
        if self.live is not None:
            self.live.contract_math(on)

    def table(self, which, seed, n=1 << 23):
        return self._answer("table", [which, seed, n], lambda r: {"table": r.table(which, seed, n)})["table"]

    def effective_link_origins(self, robot):
        src = robot.arrays["link_origin"].reshape(-1, 7)
        xor = self._answer("origins", _robot(robot), lambda r: {"xor": _xor(r.effective_link_origins(robot), src)}, values={"xor"})["xor"]
        return _xor(xor, src)

    def effective_goal_params(self, robot, problem, goal_params, B):
        gp = self._gp(problem, goal_params, B)
        xor = self._answer("goal_params", [_robot(robot), _problem(problem), gp], lambda r: {"xor": _xor(r.effective_goal_params(robot, problem, gp, B), gp)}, values={"xor"})["xor"]
        return _xor(xor, gp)

    def solve(self, robot, problem, cfg, goal_params, seeds, rng_seeds, steps, early_exit=False, nthreads=0):
        seeds = np.ascontiguousarray(seeds, dtype=np.float64).reshape(-1, robot.n_vars)
        gp = self._gp(problem, goal_params, seeds.shape[0])
        rs = np.ascontiguousarray(rng_seeds, dtype=np.uint32)
        inputs = [_robot(robot), _problem(problem), bytes(cfg), gp, seeds, rs, steps, bool(early_exit)]
        return self._answer("solve", inputs, lambda r: r.solve(robot, problem, cfg, gp, seeds, rs, steps, early_exit=early_exit, nthreads=nthreads))

    def approx_fitness(self, robot, problem, goal_params, seeds, base, genotypes):
        base = np.ascontiguousarray(base, dtype=np.float64).reshape(-1, robot.n_vars)
        B = base.shape[0]
        seeds = np.ascontiguousarray(seeds, dtype=np.float64).reshape(B, robot.n_vars)
        g = np.ascontiguousarray(genotypes, dtype=np.float64).reshape(B, -1, len(problem.active_variables))
        gp = self._gp(problem, goal_params, B)
        inputs = [_robot(robot), _problem(problem), gp, seeds, base, g]
        return self._answer("approx_fitness", inputs, lambda r: r.approx_fitness(robot, problem, gp, seeds, base, g))


def store_name(prefix, request):
    return f"{prefix}.{request.node.name.replace('[', '.').replace(']', '')}"


def reference_fixture(prefix):
    """a pytest fixture `ref`: the StoredReference of the test case (store <prefix>.<test name>[.<parameters>])"""
    import pytest

    @pytest.fixture
    def ref(request):
        r = StoredReference(store_name(prefix, request))
        yield r
        r.close()
    return ref


class StoredAdapter:
    """The adapter library (adapter/ik_evolution_2_b200.cpp inside the reference's IKFactory / IKParallel, oracle/_ref/libbioik_adapter.so)
    answered from a store.  Its answers depend on BIOIK_B200_ISLANDS, which is part of every key."""

    def __init__(self, name, load_live):
        self.store = _Store(name)
        self.lib = load_live() if recording() else None

    def close(self):
        self.store.close()

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("adapter: " + self.lib.ref_last_error().decode())

    def steps(self, robot, problem, solver, random_seed, goal_params, seeds, steps, use_clone):
        """IKFactory::create(solver) -> initialize -> step() x steps -> getSolution() per query: solutions [Q][n_vars]"""
        gp, sd = np.ascontiguousarray(goal_params, dtype=np.float64), np.ascontiguousarray(seeds, dtype=np.float64)
        Q = sd.shape[0]

        def run():
            r, p = robot.to_abi(), problem.to_abi()
            got = np.zeros((Q, robot.n_vars))
            self._check(self.lib.adapter_steps(C.byref(r), C.byref(p), solver.encode(), random_seed, Q, _abi.dptr(gp), _abi.dptr(sd), steps, use_clone, _abi.dptr(got)))
            return {"solutions": got}
        inputs = [os.environ.get("BIOIK_B200_ISLANDS"), _robot(robot), _problem(problem), solver, random_seed, gp, sd, steps, use_clone]
        return self.store.answer("steps", inputs, run)["solutions"]

    def parallel(self, robot, problem, solver, random_seed, threads, goal_params, seed, timeout):
        """IKParallel(params).solve() of one query: (solution, success, fitness, bursts)"""
        gp, sd = np.ascontiguousarray(goal_params, dtype=np.float64), np.ascontiguousarray(seed, dtype=np.float64)

        def run():
            r, p = robot.to_abi(), problem.to_abi()
            sol, succ, fit, iters = np.zeros(robot.n_vars), C.c_int32(), C.c_double(), C.c_int32()
            self._check(self.lib.adapter_parallel(C.byref(r), C.byref(p), solver.encode(), random_seed, threads, _abi.dptr(gp), _abi.dptr(sd), timeout, _abi.dptr(sol),
                                                  C.byref(succ), C.byref(fit), C.byref(iters)))
            return {"solution": sol, "success": succ.value, "fitness": fit.value, "bursts": iters.value}
        inputs = [os.environ.get("BIOIK_B200_ISLANDS"), _robot(robot), _problem(problem), solver, random_seed, threads, gp, sd, timeout]
        out = self.store.answer("parallel", inputs, run)
        return out["solution"], int(out["success"]), float(out["fitness"]), int(out["bursts"])
