"""SURVEY.md §8(b): the drop-in boundary, compiled.  adapter/ik_evolution_2_b200.cpp (the translation unit a bio_ik maintainer adds)
is built INSIDE the reference's own solver framework - IKBase, IKFactory, Problem, the goal classes, IKParallel where they lie under
the reference's sources, third-party headers from oracle/shims (oracle/adapter_harness.cpp -> oracle/_ref/libbioik_adapter.so) - and
driven through the reference's types:
    IKFactory::create("bio2_memetic_b200") -> initialize(problem) -> step() x k -> getSolution()      (src/ik_base.h:138-154)
    IKParallel(params).solve()                                                                     (src/ik_parallel.h:148-269)
The GPU tests demand the same solution BITS as the C ABI called directly (bioik_begin / bioik_step / bioik_get_solution and
bioik_solve_islands); they read the adapter's and the reference's answers from tests/golden/reference/ (tests/reference_store.py),
recorded from that library on a B200, so only the test of the library itself needs the reference's sources."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib
import reference_store
from bio_ik_b200 import _abi, goals as G, robots, workloads
from bio_ik_b200.problem import Problem

ADAPTER_LIB = os.path.join(oracle_lib.REF_DIR, "libbioik_adapter.so")


def load_adapter():
    if os.path.exists(os.path.join(oracle_lib.REFERENCE_ROOT, "src", "ik_parallel.h")):
        import __graft_entry__ as ge
        ge.build_cuda()
        subprocess.run(["make", "-C", oracle_lib.ORACLE_DIR, "-s", "adapter"], check=True)
    if not os.path.exists(ADAPTER_LIB):
        pytest.skip("oracle/_ref/libbioik_adapter.so is not built (it needs the reference's sources at build time)")
    lib = C.CDLL(ADAPTER_LIB)
    dp, ip = _abi.c_double_p, _abi.c_int32_p
    RP, PP = C.POINTER(_abi.BioikRobot), C.POINTER(_abi.BioikProblem)
    lib.ref_last_error.restype = C.c_char_p
    lib.adapter_can_create.argtypes = [RP, PP, C.c_char_p, dp]
    lib.adapter_steps.argtypes = [RP, PP, C.c_char_p, C.c_int, C.c_int, dp, dp, C.c_int, C.c_int, dp]
    lib.adapter_parallel.argtypes = [RP, PP, C.c_char_p, C.c_int, C.c_int, dp, dp, C.c_double, dp, ip, dp, ip]
    return lib


def arm_problem():
    rm, groups = robots.pr2_like()
    g = groups["right_arm"]
    pr = Problem().initialize(rm, g, [G.PoseGoal("r_wrist_roll_link")])
    return rm, pr


def has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


# ---------------------------------------------------------------------------------------------- CPU
def test_adapter_registers_with_the_reference_factory_and_has_no_cpu_fallback():
    """The adapter library loads, the reference's IKFactory still builds its own CPU class through the same harness, and the
    *_b200 classes are registered: without a CUDA device creating one fails loudly with the library's message (no CPU fallback)."""
    lib = load_adapter()
    rm, pr = arm_problem()
    r, p = rm.to_abi(), pr.to_abi()
    seed = np.zeros(rm.n_vars)
    assert lib.adapter_can_create(C.byref(r), C.byref(p), b"bio2_memetic", _abi.dptr(seed)) == 1
    assert lib.adapter_can_create(C.byref(r), C.byref(p), b"no_such_solver", _abi.dptr(seed)) == 0
    assert "class not found" in lib.ref_last_error().decode()
    for name in (b"bio2_b200", b"bio2_memetic_b200", b"bio2_memetic_l_b200"):
        ok = lib.adapter_can_create(C.byref(r), C.byref(p), name, _abi.dptr(seed))
        if has_cuda():
            assert ok == 1, lib.ref_last_error().decode()
        else:
            msg = lib.ref_last_error().decode()
            assert ok == 0 and "bioik_create" in msg and "no CPU fallback" in msg, msg


# ---------------------------------------------------------------------------------------------- GPU
ref = reference_store.reference_fixture("adapter")


@pytest.fixture
def adapter(request):
    a = reference_store.StoredAdapter(reference_store.store_name("adapter", request), load_adapter)
    yield a
    a.close()


def effective(ref, w, B):
    return ref.effective_robot(w.robot), ref.effective_goal_params(w.robot, w.problem, w.goal_params, B)


@pytest.mark.gpu
@pytest.mark.parametrize("solver,mode", [("bio2_memetic_b200", "bio2_memetic"), ("bio2_b200", "bio2"), ("bio2_memetic_l_b200", "bio2_memetic_l")])
@pytest.mark.parametrize("use_clone", [0, 1])
def test_factory_initialize_step_get_solution_equals_the_c_abi(oracle, adapter, ref, solver, mode, use_clone, monkeypatch):
    """IKFactory::create -> initialize -> step() x k -> getSolution() through the reference's types (optionally on an
    IKFactory::clone copy, re-initialised for three queries in a row) returns the solution bits of bioik_begin / bioik_step /
    bioik_get_solution and of bioik_solve_islands called directly."""
    from bio_ik_b200.solver import IKSolver
    islands, steps, Q, random_seed = 16, 7, 3, 5
    monkeypatch.setenv("BIOIK_B200_ISLANDS", str(islands))
    w = workloads.make("cfg2", lambda rm, pr, v: oracle.fk(rm, pr, v), batch=Q)
    robot, gp = effective(ref, w, Q)
    got = adapter.steps(w.robot, w.problem, solver, random_seed, w.goal_params, w.seeds, steps, use_clone)
    direct = IKSolver(robot, mode=mode, population=18, random_seed=random_seed, device=0).initialize(w.problem)
    rs = (random_seed + np.arange(islands)).astype(np.uint32)
    for q in range(Q):
        direct.begin(gp[q], w.seeds[q], islands=islands, rng_seeds=rs, max_steps=0, early_exit=2)
        for _ in range(steps):
            direct.step(1)
        a = direct.get_solution(wrap=False)
        assert np.array_equal(got[q], a["solutions"][0]), (q, "begin/step/get_solution")
        b = direct.solve_islands(gp[q], w.seeds[q], islands, steps, rng_seeds=rs, early_exit=2, wrap=False)
        assert np.array_equal(got[q], b["solutions"][0]), (q, "solve_islands")
    assert not np.array_equal(got[0], w.seeds[0])


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [1, 2])
def test_ikparallel_drives_the_gpu_solver_unchanged(oracle, adapter, ref, threads, monkeypatch):
    """The reference's driver - IKParallel::solve with its thread pool, 4-step bursts, its own exact FK + checkSolution on what the
    solver returns (src/ik_parallel.h:148-269) - around the adapter.  It stops at the first burst after which the returned vector
    passes the reference's success test; the same loop written against the C ABI gives the same bits and the same burst count."""
    from bio_ik_b200.solver import IKSolver
    islands, random_seed, Q = 32, 3, 4
    monkeypatch.setenv("BIOIK_B200_ISLANDS", str(islands))
    w = workloads.make("cfg2", lambda rm, pr, v: oracle.fk(rm, pr, v), batch=Q)
    robot, gp = effective(ref, w, Q)
    direct = IKSolver(robot, mode="bio2_memetic", population=18, random_seed=random_seed, device=0).initialize(w.problem)
    solved = 0
    for q in range(Q):
        sol, succ, fit, iters = adapter.parallel(w.robot, w.problem, "bio2_memetic_b200", random_seed, threads, w.goal_params[q], w.seeds[q], 20.0)
        assert succ == 1  # reachable PR2-arm poses, 32+ islands: the reference's own test accepts the GPU's answer
        solved += succ
        # the reference's exact FK of the returned vector really is at the goal
        tip = oracle.fk(w.robot, w.problem, sol[None])[0, 0]
        assert np.abs(tip[:3] - w.goal_params[q, 0, :3]).max() < 1e-4
        if threads == 1:
            # the same driver loop against the C ABI: bursts of 4 steps until the best island passes the success test
            direct.begin(gp[q], w.seeds[q], islands=islands, rng_seeds=(random_seed + np.arange(islands)).astype(np.uint32), max_steps=0, early_exit=2)
            bursts = 0
            while True:
                direct.step(4)
                bursts += 1
                a = direct.get_solution(wrap=False)
                if a["success"][0] or bursts > 200:
                    break
            assert bursts == iters and np.array_equal(sol, a["solutions"][0]), (q, bursts, iters)
    assert solved == Q


@pytest.mark.gpu
def test_resumable_steps_cost_no_restart(oracle):
    """k calls of bioik_step(1) leave the device in the state of one bioik_step(k) (and of bioik_solve_islands with k steps):
    the solver state is resident, nothing is re-solved from the seed."""
    from bio_ik_b200.solver import IKSolver
    w = workloads.make("cfg2", lambda rm, pr, v: oracle.fk(rm, pr, v), batch=8)
    s = IKSolver(w.robot, mode="bio2_memetic", population=32, random_seed=1, device=0).initialize(w.problem)
    islands, k = 4, 9
    l0 = s.launch_count()
    s.begin(w.goal_params, w.seeds, islands=islands, early_exit=0)
    for _ in range(k):
        s.step(1)
    one = s.get_solution()
    l1 = s.launch_count()
    s.begin(w.goal_params, w.seeds, islands=islands, early_exit=0)
    s.step(k)
    many = s.get_solution()
    l2 = s.launch_count()
    whole = s.solve_islands(w.goal_params, w.seeds, islands, k, early_exit=0, wrap=False)
    for key in ("solutions", "fitness", "success", "island", "steps"):
        assert np.array_equal(one[key], many[key]) and np.array_equal(one[key], whole[key]), key
    assert np.all(one["steps"] == k)
    assert l1 - l0 <= (l2 - l1) + 4 * k  # O(k) launches either way (queue set-up, solve kernel and the active-run count per call)


@pytest.mark.gpu
def test_adapter_flattens_a_balance_goal_from_the_urdf_inertials(oracle, adapter, ref, monkeypatch):
    """BalanceGoal through the reference's types: the adapter reads the link inertials from RobotModel::getURDF() like
    BalanceGoal::describe does, the reference's Problem::initialize makes every link with mass a tip link, and the device answer equals
    the C ABI called with the same flattened problem."""
    from bio_ik_b200.solver import IKSolver
    islands, steps, random_seed = 8, 5, 2
    monkeypatch.setenv("BIOIK_B200_ISLANDS", str(islands))
    rm, groups = robots.balancing_tree()
    g = groups["all"]
    pr = Problem().initialize(rm, g, [G.PoseGoal(g.tip_links[0]), G.BalanceGoal((0.05, -0.02, 0.3), 0.8, axis=(0.1, 0.2, 0.97))])
    rng = np.random.default_rng(4)
    seeds = workloads.sample_configurations(rm, pr.active_variables, 1, rng)
    gp = pr.default_goal_params()[None]
    got = adapter.steps(rm, pr, "bio2_memetic_b200", random_seed, gp, seeds, steps, 0)
    direct = IKSolver(ref.effective_robot(rm), mode="bio2_memetic", population=18, random_seed=random_seed, device=0).initialize(pr)
    rs = (random_seed + np.arange(islands)).astype(np.uint32)
    want = direct.solve_islands(ref.effective_goal_params(rm, pr, gp, 1), seeds, islands, steps, rng_seeds=rs, early_exit=2, wrap=False)
    assert np.array_equal(got[0], want["solutions"][0]) and not np.array_equal(got[0], seeds[0])
