"""Parity of the CUDA path with the CPU oracle, through the C ABI, on a real B200 (-m gpu).
Bar: BIT-IDENTICAL joint angles and fitness (far inside BASELINE.json's 1e-5), because oracle and
kernels share one arithmetic contract (DESIGN.md §3).  The only tolerance-based comparisons are the
libm-class functions of the success test."""
import ctypes as C

import numpy as np
import pytest

import gpu_util
import oracle_lib
import reference_store
from bio_ik_b200 import _abi, goals as G, robots, workloads
from bio_ik_b200.problem import Problem
from bio_ik_b200.solver import BioIKError, IKSolver

pytestmark = pytest.mark.gpu
ref = reference_store.reference_fixture("gpu_parity")


def ofk(oracle):
    return lambda rm, pr, v: oracle.fk(rm, pr, v)


# ---------------------------------------------------------------------------------------------
# rows a9-a11, a6, a7 of SURVEY.md §8(a): exact FK, Jacobian/approximator, approximate fitness
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("maker,group", [(robots.pr2_like, "all"), (robots.pr2_like, "right_arm"), (robots.snake, "all"), (robots.shadow_like_hand, "hand"),
                                         (lambda: robots.random_tree(1), "all"), (lambda: robots.random_tree(2, n_joints=12, branch_at=7), "all"), (robots.mimic_gripper_arm, "all"),
                                         (robots.floating_base_arm, "all"), (robots.planar_base_arm, "all")])
def test_exact_fk_and_delta_frames(oracle, maker, group):
    rm, groups = maker()
    g = groups[group]
    pr = Problem().initialize(rm, g, [G.PoseGoal(t) for t in g.tip_links])
    solver = IKSolver(rm).initialize(pr)
    rng = np.random.default_rng(3)
    v = workloads.sample_configurations(rm, range(rm.n_vars), 500, rng)
    v[:8] *= 50.0  # far outside the limits: exercises the large-argument path of the contract sin/cos
    assert np.array_equal(solver.fk(v), oracle.fk(rm, pr, v))
    d, mask = oracle.approx(rm, pr, v[:200])
    d = d.copy()
    d[mask == 0, 6] = 0.0
    assert np.array_equal(solver.approx(v[:200]), d)


def test_approximate_fitness_all_device_goals(oracle):
    rm, groups = robots.pr2_like()
    g = groups["all"]
    r, l = "r_wrist_roll_link", "l_wrist_roll_link"
    gl = [G.PoseGoal(r, (0.6, -0.2, 0.9), (0.1, 0.2, 0.3, 0.9)), G.PositionGoal(l, (0.5, 0.3, 1.0), 0.7), G.OrientationGoal(l, (0, 0.5, 0, 1), 1.3),
          G.LookAtGoal(r, (1, 0, 0), (2, 0.5, 1)), G.MaxDistanceGoal(l, (0.5, 0, 1), 0.3), G.MinDistanceGoal(r, (0.5, 0, 1), 0.6), G.LineGoal(r, (0.5, 0, 1), (1, 1, 0)),
          G.PlaneGoal(l, (0.5, 0, 1), (0, 1, 1)), G.SideGoal(r, (0, 0, 1), (0, 1, 0)), G.DirectionGoal(l, (1, 0, 0), (0, 0, 1)), G.JointVariableGoal("torso_lift_joint", 0.2, 2.0),
          G.AvoidJointLimitsGoal(1.5), G.CenterJointsGoal(0.5, secondary=False), G.RegularizationGoal(0.25), G.MinimalDisplacementGoal(2.0),
          G.ConeGoal(r, (1, 0, 0), (0, 0.6, 0.8), 0.3, weight=0.5, position=(0.5, 0, 1), position_weight=0.7), G.ConeGoal(l, (0, 0, 1), (1, 0, 0), 1.2)]
    pr = Problem().initialize(rm, g, gl)
    solver = IKSolver(rm).initialize(pr)
    rng = np.random.default_rng(4)
    B, M, n = 40, 16, len(pr.active_variables)
    base = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    genes = base[:, pr.active_variables][:, None, :] + rng.normal(0, 0.2, (B, M, n))
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    gp[:, 0, 0:3] += rng.normal(0, 0.1, (B, 3))
    p_ref, s_ref = oracle.approx_fitness(rm, pr, gp, seeds, base, genes)
    p_gpu, s_gpu = solver.approx_fitness(gp, seeds, base, genes)
    assert np.array_equal(p_gpu, p_ref) and np.array_equal(s_gpu, s_ref)
    # NULL goal_params -> BioikGoal::p defaults
    p_ref, s_ref = oracle.approx_fitness(rm, pr, None, seeds, base, genes)
    p_gpu, s_gpu = solver.approx_fitness(None, seeds, base, genes)
    assert np.array_equal(p_gpu, p_ref) and np.array_equal(s_gpu, s_ref)


# ---------------------------------------------------------------------------------------------
# the whole step(): trajectory-level parity (rows a1-a8, a12-a15)
# ---------------------------------------------------------------------------------------------
TRACE_CASES = [
    ("cfg2", 16, 18, "q", 8, 10), ("cfg2", 16, 64, "q", 8, 25), ("cfg2", 24, 128, "q", 8, 25), ("cfg2", 8, 35, "q", 8, 7), ("cfg2", 8, 4, "q", 8, 5), ("cfg2", 4, 256, "q", 8, 3),
    ("cfg2", 16, 18, 0, 16, 10), ("cfg2", 16, 40, "l", 8, 10), ("cfg3", 12, 128, "q", 8, 12), ("cfg4", 8, 128, "q", 8, 10), ("cfg4", 8, 37, "l", 8, 6), ("cfg5", 12, 128, "q", 8, 10),
]


@pytest.mark.parametrize("name,B,pop,mode,gens,steps", TRACE_CASES)
def test_solver_state_is_bit_identical_to_the_oracle(oracle, name, B, pop, mode, gens, steps):
    w = workloads.make(name, ofk(oracle), batch=B)
    cfg = oracle_lib.make_cfg(population=pop, memetic=mode, generations=gens)
    ref = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, steps)
    solver = gpu_util.make_solver(w, pop, mode, gens)
    got = solver.trace(w.goal_params, w.seeds, w.rng_seeds, steps)
    gpu_util.assert_bit_equal(got, ref, what=f"{name} pop={pop}")
    res = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, steps)
    gpu_util.assert_bit_equal(res, ref, keys=("solutions", "fitness", "success", "steps"), what=f"{name} pop={pop}")


def test_table_seed_and_query_seed_are_honoured(oracle):
    w = workloads.make("cfg2", ofk(oracle), batch=8)
    cfg = oracle_lib.make_cfg(population=18, table_seed=77)
    rs = np.array([5, 5, 9, 1 << 31, 0, 2147483647, 3, 3], dtype=np.uint32)
    ref = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, rs, 8)
    solver = gpu_util.make_solver(w, 18, random_seed=77)
    gpu_util.assert_bit_equal(solver.trace(w.goal_params, w.seeds, rs, 8), ref)


def test_early_exit_matches_the_driver_contract(oracle):
    w = workloads.make("cfg2", ofk(oracle), batch=64)
    cfg = oracle_lib.make_cfg(population=32)
    ref = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 22, early_exit=True)
    solver = gpu_util.make_solver(w, 32)
    got = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 22, early_exit=True)
    gpu_util.assert_bit_equal(got, ref, keys=("solutions", "fitness", "success", "steps"))
    assert set(got["steps"].tolist()) <= {4, 8, 12, 16, 20, 22} and got["steps"].min() < 22


def test_batch_composition_does_not_matter(oracle):
    """Queries are independent: a query's answer does not depend on its batch neighbours or position."""
    w = workloads.make("cfg2", ofk(oracle), batch=300)
    solver = gpu_util.make_solver(w, 64)
    full = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 9)
    idx = np.array([299, 0, 17, 150, 151, 33, 32, 31])
    part = solver.solve_batch(w.goal_params[idx], w.seeds[idx], w.rng_seeds[idx], 9)
    for k in ("solutions", "fitness", "success"):
        assert np.array_equal(part[k], full[k][idx])
    one = solver.solve_batch(w.goal_params[5:6], w.seeds[5:6], w.rng_seeds[5:6], 9)
    assert np.array_equal(one["solutions"][0], full["solutions"][5])


def test_zero_steps_returns_the_seed(oracle):
    w = workloads.make("cfg2", ofk(oracle), batch=5)
    solver = gpu_util.make_solver(w, 18)
    res = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 0)
    assert np.array_equal(res["solutions"], w.seeds) and np.all(res["steps"] == 0)
    cfg = oracle_lib.make_cfg(population=18)
    ref = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 0)
    assert np.array_equal(res["fitness"], ref["fitness"])


# ---------------------------------------------------------------------------------------------
# BASELINE.json full sizes: size-independent properties + a bounded oracle sample
# ---------------------------------------------------------------------------------------------
def test_cfg2_full_size_10k_queries(oracle):
    w = workloads.make("cfg2", ofk(oracle), batch=10000)
    solver = gpu_util.make_solver(w, 128)
    res = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 25)
    again = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 25)
    for k in res:
        assert np.array_equal(res[k], again[k])  # deterministic
    assert res["success"].mean() >= 0.93
    ok = res["success"] == 1
    # FK -> IK -> FK round trip: solved queries reach their goal pose (dtwist = 1e-5 on every twist component)
    tips = solver.fk(res["solutions"])
    assert np.abs(tips[ok, 0, :3] - w.goal_params[ok, 0, :3]).max() < 2e-5
    qerr = np.minimum(np.abs(tips[ok, 0, 3:] - w.goal_params[ok, 0, 3:7]).max(1), np.abs(tips[ok, 0, 3:] + w.goal_params[ok, 0, 3:7]).max(1))
    assert qerr.max() < 2e-5
    # the reported fitness IS the goal error of the returned solution (idempotent re-evaluation)
    p = w.goal_params[:, 0]
    e = ((p[:, :3] - tips[:, 0, :3]) ** 2).sum(1) + np.minimum(((p[:, 3:7] - tips[:, 0, 3:]) ** 2).sum(1), ((p[:, 3:7] + tips[:, 0, 3:]) ** 2).sum(1)) * 0.25
    assert np.allclose(res["fitness"], e, rtol=1e-9, atol=1e-30)
    # clip limits hold
    a = w.robot.arrays
    for ivar in w.problem.active_variables:
        if a["var_bounded"][ivar] and a["var_max"][ivar] - a["var_min"][ivar] < 6.28:
            assert res["solutions"][:, ivar].min() >= a["var_min"][ivar] and res["solutions"][:, ivar].max() <= a["var_max"][ivar]
    # inactive variables pass through
    inactive = [v for v in range(w.robot.n_vars) if v not in w.problem.active_variables]
    assert np.array_equal(res["solutions"][:, inactive], w.seeds[:, inactive])
    # bounded oracle sample of the same batch: bit-identical
    idx = np.r_[0:96, 9990:10000]
    cfg = oracle_lib.make_cfg(population=128)
    ref = oracle.solve(w.robot, w.problem, cfg, w.goal_params[idx], w.seeds[idx], w.rng_seeds[idx], 25)
    for k in ("solutions", "fitness", "success", "steps"):
        assert np.array_equal(res[k][idx], ref[k]), k


@pytest.mark.parametrize("name,B,sample", [("cfg3", 4096, 24), ("cfg4", 2048, 16), ("cfg5", 8192, 16)])
def test_other_configs_full_size(oracle, name, B, sample):
    w = workloads.make(name, ofk(oracle), batch=B)
    solver = gpu_util.make_solver(w, 128)
    res = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 25)
    assert np.all(np.isfinite(res["fitness"])) and np.all(res["steps"] == 25)
    assert np.median(res["fitness"]) < 1e-6
    idx = np.arange(sample)
    cfg = oracle_lib.make_cfg(population=128)
    ref = oracle.solve(w.robot, w.problem, cfg, w.goal_params[idx], w.seeds[idx], w.rng_seeds[idx], 25)
    for k in ("solutions", "fitness", "success", "steps"):
        assert np.array_equal(res[k][idx], ref[k]), k


# ---------------------------------------------------------------------------------------------
# error behaviour of the boundary (status codes instead of ERROR(...) exceptions)
# ---------------------------------------------------------------------------------------------
def test_error_paths():
    rm, groups = robots.pr2_like()
    g = groups["right_arm"]
    pr = Problem().initialize(rm, g, [G.PoseGoal("r_wrist_roll_link")])
    solver = IKSolver(rm)
    with pytest.raises(BioIKError) as e:
        solver.solve_batch(None, np.zeros((1, rm.n_vars)), np.ones(1, dtype=np.uint32), 1)
    assert e.value.code == _abi.E_NO_PROBLEM
    p = pr.to_abi()
    p.goals[0].type = 99
    assert solver.lib.bioik_set_problem(solver._ctx, C.byref(p)) == _abi.E_UNSUPPORTED_GOAL
    p.goals[0].type = _abi.GOAL_POSE
    assert solver.lib.bioik_set_problem(solver._ctx, C.byref(p)) == _abi.OK
    with pytest.raises(BioIKError) as e:
        IKSolver(rm, population=3)
    assert e.value.code == _abi.E_LIMIT
    with pytest.raises(BioIKError):
        IKSolver(rm, mode="bio1")
    # a floating joint whose rotation variables are not consecutive genes is refused, not silently mis-solved
    links = [robots.Link("world", None), robots.Link("base", "world", _abi.JOINT_FLOATING, joint_name="virtual"), robots.Link("arm", "base", _abi.JOINT_REVOLUTE, lower=-1, upper=1, joint_name="j")]
    rm2 = robots.RobotModel("floating", links)
    g2 = robots.JointModelGroup(rm2, "all", ["virtual", "j"], ["arm"])
    pr2 = Problem().initialize(rm2, g2, [G.PositionGoal("arm")])
    pr2.active_variables = [0, 1, 2, 3, 7, 4, 5, 6]  # rot_x followed by the arm joint
    pr2._active = np.array(pr2.active_variables, dtype=np.int32)
    with pytest.raises(BioIKError) as e:
        IKSolver(rm2).initialize(pr2)
    assert e.value.code == _abi.E_UNSUPPORTED_JOINT


def test_device_pointer_entry_point(oracle):
    torch = pytest.importorskip("torch")
    w = workloads.make("cfg2", ofk(oracle), batch=128)
    solver = gpu_util.make_solver(w, 64)
    dev = torch.device("cuda:0")
    gp = torch.from_numpy(w.goal_params).to(dev)
    seeds = torch.from_numpy(w.seeds).to(dev)
    rs = torch.from_numpy(w.rng_seeds.astype(np.int64)).to(dev).to(torch.int32)  # same 32-bit pattern
    sol = torch.empty((128, w.robot.n_vars), dtype=torch.float64, device=dev)
    fit = torch.empty(128, dtype=torch.float64, device=dev)
    succ = torch.empty(128, dtype=torch.int32, device=dev)
    stp = torch.empty(128, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream()
    solver.kernel_time()  # switches per-launch timing on
    solver.solve_batch_device(128, gp.data_ptr(), seeds.data_ptr(), rs.data_ptr(), 6, False, sol.data_ptr(), fit.data_ptr(), succ.data_ptr(), stp.data_ptr(), stream=st.cuda_stream)
    st.synchronize()
    ref = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 6)
    assert np.array_equal(sol.cpu().numpy(), ref["solutions"]) and np.array_equal(fit.cpu().numpy(), ref["fitness"])
    ev, nev, se, nse = solver.kernel_time(disable=True)
    assert nev >= 1 and ev > 0 and solver.launch_count() > 0  # one launch per step in the stepped path, one per solve in the persistent one
    # with timing off, repeated host-API solves of one shape replay a CUDA graph: same answers
    for _ in range(3):
        again = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 6)
        assert np.array_equal(again["solutions"], ref["solutions"]) and np.array_equal(again["fitness"], ref["fitness"])
    other = solver.solve_batch(w.goal_params[:50], w.seeds[:50], w.rng_seeds[:50], 6)  # shape change drops the graph
    assert np.array_equal(other["solutions"], ref["solutions"][:50])


def test_generic_and_fast_generation_kernels_agree(oracle, monkeypatch):
    """The generic kernel (k_evolve, any problem shape) and the register-blocked k_evolve_fast are two schedules of
    the same arithmetic: identical results, both identical to the oracle."""
    for name, B, pop, steps in (("cfg2", 32, 128, 6), ("cfg3", 16, 100, 4), ("cfg4", 8, 128, 4), ("cfg5", 8, 64, 3)):
        w = workloads.make(name, ofk(oracle), batch=B)
        fast = gpu_util.make_solver(w, pop)
        monkeypatch.setenv("BIOIK_FORCE_GENERIC", "1")
        generic = gpu_util.make_solver(w, pop)
        monkeypatch.delenv("BIOIK_FORCE_GENERIC")
        a = fast.trace(w.goal_params, w.seeds, w.rng_seeds, steps)
        b = generic.trace(w.goal_params, w.seeds, w.rng_seeds, steps)
        gpu_util.assert_bit_equal(a, b, what=name + " fast vs generic")
        cfg = oracle_lib.make_cfg(population=pop)
        ref = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, steps)
        gpu_util.assert_bit_equal(a, ref, what=name)


def test_mixed_goal_problem_on_gpu(oracle):
    rm, groups = robots.pr2_like()
    g = groups["all"]
    r, l = "r_wrist_roll_link", "l_wrist_roll_link"
    gl = [G.PositionGoal(r, (0.6, -0.3, 0.9)), G.LookAtGoal(l, (1, 0, 0), (2, 0.5, 1), 0.3), G.JointVariableGoal("torso_lift_joint", 0.2, 2.0), G.CenterJointsGoal(0.5, secondary=False),
          G.LineGoal(l, (0.5, 0.2, 1), (1, 1, 0), 0.7), G.MinimalDisplacementGoal(1.5), G.AvoidJointLimitsGoal(0.8), G.DirectionGoal(r, (1, 0, 0), (0, 0, 1), 0.4),
          G.ConeGoal(l, (1, 0, 0), (0, 0.6, 0.8), 0.4, weight=0.3)]
    pr = Problem().initialize(rm, g, gl)
    rng = np.random.default_rng(5)
    seeds = workloads.sample_configurations(rm, pr.active_variables, 40, rng)
    rs = np.arange(40, dtype=np.uint32) + 3
    cfg = oracle_lib.make_cfg(population=45)
    ref = oracle.solve(rm, pr, cfg, None, seeds, rs, 8)
    solver = IKSolver(rm, population=45).initialize(pr)
    gpu_util.assert_bit_equal(solver.trace(None, seeds, rs, 8), ref)


@pytest.mark.parametrize("pop", [20, 128, 200])
def test_preselection_with_tied_secondary_fitness_on_gpu(oracle, pop):
    """AvoidJointLimitsGoal as the only secondary goal: most children score exactly 0.0, the pre-selection order (:366-378) is
    decided by the child slot - the fast rank pass of the generation kernel has to fall back to its exact pass."""
    w = workloads.cfg2(32)
    pr = Problem().initialize(w.robot, w.group, [G.PoseGoal("r_wrist_roll_link"), G.AvoidJointLimitsGoal(1.0)])
    w.problem = pr
    w.generate(lambda rm, p, v: oracle.fk(rm, p, v), B=32, cfg_id=2)
    cfg = oracle_lib.make_cfg(population=pop)
    ref = oracle.solve(w.robot, pr, cfg, w.goal_params, w.seeds, w.rng_seeds, 6)
    solver = IKSolver(w.robot, population=pop).initialize(pr)
    gpu_util.assert_bit_equal(solver.trace(w.goal_params, w.seeds, w.rng_seeds, 6), ref)


def test_mimic_joints_on_gpu(oracle):
    rm, groups = robots.mimic_gripper_arm()
    pr = Problem().initialize(rm, groups["all"], [G.PositionGoal("pad_a"), G.PoseGoal("pad_b")])
    rng = np.random.default_rng(1)
    B = 48
    tg = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    tips = oracle.fk(rm, pr, tg)
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    gp[:, 0, 0:3], gp[:, 1, 0:7] = tips[:, 0, 0:3], tips[:, 1, :]
    cfg = oracle_lib.make_cfg(population=64)
    rs = np.arange(B, dtype=np.uint32) + 1
    ref = oracle.solve(rm, pr, cfg, gp, seeds, rs, 12)
    solver = IKSolver(rm, population=64).initialize(pr)
    gpu_util.assert_bit_equal(solver.trace(gp, seeds, rs, 12), ref)


def test_virtual_joints_that_mimic_on_gpu(oracle):
    """a PLANAR joint mimicking a prismatic joint, a FLOATING joint mimicking a revolute one (forward_kinematics.h:230-246,698-699)"""
    rm, groups = robots.mimic_virtual_joint_arm()
    pr = Problem().initialize(rm, groups["all"], [G.PoseGoal("ee"), G.PositionGoal("probe")])
    rng = np.random.default_rng(2)
    B = 40
    base = robots.mimic_virtual_joint_base(rm)
    tg = workloads.sample_configurations(rm, pr.active_variables, B, rng, base=base)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng, base=base)
    tips = oracle.fk(rm, pr, tg)
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    gp[:, 0, 0:7], gp[:, 1, 0:3] = tips[:, 0, :], tips[:, 1, 0:3]
    cfg = oracle_lib.make_cfg(population=64)
    rs = np.arange(B, dtype=np.uint32) + 1
    ref = oracle.solve(rm, pr, cfg, gp, seeds, rs, 10)
    solver = IKSolver(rm, population=64).initialize(pr)
    assert np.array_equal(solver.fk(seeds), oracle.fk(rm, pr, seeds))
    gpu_util.assert_bit_equal(solver.trace(gp, seeds, rs, 10), ref)


# ---------------------------------------------------------------------------------------------
# SURVEY.md §8(f) rows 1 and 3: islands of one query, IKParallel's selection, the plugin's angle wrap
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,Q,islands,steps,early", [("cfg2", 24, 8, 12, 0), ("cfg2", 16, 5, 25, 1), ("cfg2", 16, 7, 25, 2), ("cfg4", 6, 4, 12, 2), ("cfg4", 6, 4, 6, 0), ("cfg3", 8, 3, 6, 0)])
def test_solve_islands_matches_the_oracle(oracle, name, Q, islands, steps, early):
    w = workloads.make(name, ofk(oracle), batch=Q)
    solver = IKSolver(w.robot, mode="bio2_memetic", population=40, random_seed=1, device=0).initialize(w.problem)
    cfg = oracle_lib.make_cfg(population=40)
    for wrap in (True, False):
        got = solver.solve_islands(w.goal_params, w.seeds, islands, steps, early_exit=early, wrap=wrap)
        ref = oracle_lib.oracle_solve_islands(oracle, w.robot, w.problem, cfg, w.goal_params, w.seeds, islands, steps, early_exit=early, wrap=wrap)
        for k in ("solutions", "fitness", "success", "island", "steps"):
            assert np.array_equal(got[k], ref[k]), (k, wrap)
    if steps >= 12:
        # islands share the table-driven mutation stream (fixed-seed XORShift64 index, src/ik_base.h:118-125); their own
        # minstd engine only enters through the wipeout of the second species, so they need a few steps to part ways
        assert len(set(ref["island"].tolist())) > 1
    # a batch solve afterwards still works (the staging buffers are shared)
    a = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 3)
    b = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 3)
    assert np.array_equal(a["solutions"], b["solutions"])


@pytest.mark.parametrize("name,Q,islands,steps,early,stride", [("cfg2", 16, 8, 12, 0, 1), ("cfg2", 12, 6, 25, 2, 2), ("cfg4", 6, 4, 8, 2, 1), ("cfg3", 8, 3, 6, 0, 1)])
def test_island_stream_stride_matches_the_oracle(oracle, name, Q, islands, steps, early, stride):
    """BIOIK_OPT_ISLAND_STREAM_STRIDE: island i starts i * stride steps into the shared random streams (the oracle restates the option)"""
    w = workloads.make(name, ofk(oracle), batch=Q)
    solver = IKSolver(w.robot, mode="bio2_memetic", population=40, random_seed=1, device=0, island_stream_stride=stride).initialize(w.problem)
    cfg = oracle_lib.make_cfg(population=40)
    got = solver.solve_islands(w.goal_params, w.seeds, islands, steps, early_exit=early)
    ref = oracle_lib.oracle_solve_islands(oracle, w.robot, w.problem, cfg, w.goal_params, w.seeds, islands, steps, early_exit=early, island_stride=stride)
    for k in ("solutions", "fitness", "success", "island", "steps"):
        assert np.array_equal(got[k], ref[k]), k
    # a plain batch on the same context is not affected by the option
    a = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 3)
    b = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 3)
    assert np.array_equal(a["solutions"], b["solutions"])
    # and switching it off gives the clone islands back
    solver.set_option(_abi.OPT_ISLAND_STREAM_STRIDE, 0)
    got = solver.solve_islands(w.goal_params, w.seeds, islands, steps, early_exit=early)
    ref = oracle_lib.oracle_solve_islands(oracle, w.robot, w.problem, cfg, w.goal_params, w.seeds, islands, steps, early_exit=early)
    for k in ("solutions", "fitness", "success", "island", "steps"):
        assert np.array_equal(got[k], ref[k]), k


def test_solve_islands_default_goal_parameters_and_seeds(oracle):
    rm, groups = robots.pr2_like()
    g = groups["right_arm"]
    pr = Problem().initialize(rm, g, [G.PoseGoal("r_wrist_roll_link", (0.55, -0.25, 0.95), (0.0, 0.0, 0.0, 1.0)), G.MinimalDisplacementGoal(0.3)])
    solver = IKSolver(rm, mode="bio2_memetic", population=32, random_seed=1, device=0).initialize(pr)
    rng = np.random.default_rng(2)
    seeds = workloads.sample_configurations(rm, pr.active_variables, 5, rng)
    rs = rng.integers(1, 2 ** 31 - 2, 5 * 7).astype(np.uint32)
    got = solver.solve_islands(None, seeds, 7, 10, rng_seeds=rs, early_exit=0)
    ref = oracle_lib.oracle_solve_islands(oracle, rm, pr, oracle_lib.make_cfg(population=32), None, seeds, 7, 10, rng_seeds=rs, early_exit=0)
    for k in ("solutions", "fitness", "success", "island", "steps"):
        assert np.array_equal(got[k], ref[k]), k


# ---------------------------------------------------------------------------------------------
# the CUDA path against the REFERENCE'S OWN CODE (its answers stored under tests/golden/reference/, see tests/reference_store.py)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B,pop,steps", [("cfg2", 256, 128, 25), ("cfg2", 64, 18, 25), ("cfg1", 1, 64, 25), ("cfg4", 16, 128, 10)])
def test_gpu_equals_the_reference_code_with_contract_math(ref, name, B, pop, steps):
    """No oracle in between: the reference's src/ik_evolution_2.cpp + src/problem.cpp + forward_kinematics.h, compiled in place
    (oracle/ref_harness.cpp), with its two libm calls sin / cos swapped for the arithmetic contract's det_sincos and its child pool
    re-sized to `pop` - against bioik_solve_batch on the GPU.  Bit-identical joint angles, fitness, success flags and every
    species' genes and gradients (single-tip problems: quirk Q2 does not apply)."""
    w = workloads.make(name, lambda rm, pr, v: oracle_lib.Oracle().fk(rm, pr, v), batch=B)
    B = len(w.rng_seeds)
    # the numbers the reference stores after its own normalising constructors / Isometry3d conversion (ulp-level changes)
    robot, gp = ref.effective_robot(w.robot), ref.effective_goal_params(w.robot, w.problem, w.goal_params, B)
    solver = IKSolver(robot, mode="bio2_memetic", population=pop, random_seed=1, device=0).initialize(w.problem)
    got = solver.trace(gp, w.seeds, w.rng_seeds, steps)
    res = solver.solve_batch(gp, w.seeds, w.rng_seeds, steps)
    ref.contract_math(True)
    try:
        want = ref.solve(w.robot, w.problem, oracle_lib.make_cfg(population=pop), w.goal_params, w.seeds, w.rng_seeds, steps)
    finally:
        ref.contract_math(False)
    for k in ("genes", "gradients", "species_fitness", "solutions", "fitness"):
        assert reference_store.same(got[k], want[k]), k
    assert reference_store.same(res["success"], want["success"]) and reference_store.same(res["solutions"], want["solutions"])


@pytest.mark.parametrize("name,B,pop,steps", [("cfg3", 64, 128, 25), ("cfg5", 48, 128, 12), ("cfg3", 32, 18, 25)])
def test_gpu_reference_stale_tip_mode_equals_the_reference_code(oracle, ref, name, B, pop, steps):
    """Multi-tip problems in the reference-quirk mode (BIOIK_OPT_REFERENCE_STALE_TIPS): bit-identical to the oracle's emulation
    of quirk Q2 and to the reference's own code (contract sin / cos, phenotypes3 pre-filled with identity frames by the
    harness), i.e. all five BASELINE configurations match the reference's code on the GPU."""
    w = workloads.make(name, ofk(oracle), batch=B)
    cfg = oracle_lib.make_cfg(population=pop)
    robot, gp = ref.effective_robot(w.robot), ref.effective_goal_params(w.robot, w.problem, w.goal_params, B)
    solver = IKSolver(robot, mode="bio2_memetic", population=pop, random_seed=1, device=0, reference_stale_tips=True).initialize(w.problem)
    got = solver.trace(gp, w.seeds, w.rng_seeds, steps)
    want = oracle.solve(robot, w.problem, cfg, gp, w.seeds, w.rng_seeds, steps, flags=8)
    for k in ("genes", "gradients", "species_fitness", "solutions", "fitness"):
        assert np.array_equal(got[k], want[k]), k
    ref.contract_math(True)
    try:
        r = ref.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, steps)
    finally:
        ref.contract_math(False)
    for k in ("genes", "gradients", "species_fitness", "solutions", "fitness"):
        assert reference_store.same(got[k], r[k]), ("reference", k)
    # and the default mode differs on these problems (documented deviation Q2)
    plain = IKSolver(robot, mode="bio2_memetic", population=pop, random_seed=1, device=0).initialize(w.problem).trace(gp, w.seeds, w.rng_seeds, steps)
    assert not np.array_equal(plain["genes"], got["genes"])


def floating_problem(oracle, group, B, seed=1, maker=None):
    rm, groups = (maker or robots.floating_base_arm)()
    g = groups[group]
    pr = Problem().initialize(rm, g, [G.PoseGoal(t) for t in g.tip_links])
    rng = np.random.default_rng(seed)
    targets = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    tips = oracle.fk(rm, pr, targets)
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    for gi, rec in enumerate(pr.goal_list):
        gp[:, gi, 0:7] = tips[:, rec["tip"], 0:7]
    return rm, pr, gp, seeds


@pytest.mark.parametrize("maker", [robots.floating_base_arm, robots.planar_base_arm])
@pytest.mark.parametrize("group,mode,gens", [("whole_arm", "q", 8), ("all", "q", 8), ("all", 0, 16), ("whole_arm", "l", 8)])
def test_floating_and_planar_base_joints(oracle, ref, group, mode, gens, maker):
    """SURVEY.md §8(f) row 4: a FLOATING joint on the chain (src/forward_kinematics.h:120-127 joint frame, :695-726 numeric
    Jacobian through frameTwist, src/ik_evolution_2.cpp:118-126,320-324 quaternion-gene normalisation) - bit-identical to the
    oracle and to the reference's own code (contract sin / cos / acos; quirk mode for the
    two-tip problem, where the base moves both tips but the arm joints only one).  PLANAR joints take the same numeric route;
    their joint frame is MoveIt's computeTransform + Eigen's matrix -> quaternion, restated (oracle/shims/README.md)."""
    B, pop, steps = 48, 64 if maker is robots.floating_base_arm else 128, 12
    rm, pr, gp, seeds = floating_problem(oracle, group, B, maker=maker)
    rs = 1 + np.arange(B, dtype=np.uint32)
    name = {0: "bio2", "q": "bio2_memetic", "l": "bio2_memetic_l"}[mode]
    cfg = oracle_lib.make_cfg(population=pop, memetic=mode, generations=gens)
    got = IKSolver(rm, mode=name, population=pop, random_seed=1, device=0).initialize(pr).trace(gp, seeds, rs, steps)
    want = oracle.solve(rm, pr, cfg, gp, seeds, rs, steps)
    for k in ("genes", "gradients", "species_fitness", "solutions", "fitness"):
        assert np.array_equal(got[k], want[k]), k
    robot, gpe = ref.effective_robot(rm), ref.effective_goal_params(rm, pr, gp, B)
    got = IKSolver(robot, mode=name, population=pop, random_seed=1, device=0, reference_stale_tips=True).initialize(pr).trace(gpe, seeds, rs, steps)
    ref.contract_math(True)
    try:
        r = ref.solve(rm, pr, cfg, gp, seeds, rs, steps)
    finally:
        ref.contract_math(False)
    for k in ("genes", "gradients", "species_fitness", "solutions", "fitness"):
        assert reference_store.same(got[k], r[k]), ("reference", k)


def test_cancel_from_another_thread(oracle):
    """bioik_cancel = the reference's `canceled` flag (src/ik_base.h:143, polled at ik_evolution_2.cpp:355,457): a solve in flight
    stops at the next kernel and returns what it had reached; the next solve starts with the flag cleared."""
    import threading
    import time
    w = workloads.make("cfg2", ofk(oracle), batch=4000)
    solver = IKSolver(w.robot, mode="bio2_memetic", population=128, random_seed=1, device=0).initialize(w.problem)
    solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 2)  # sizes the state
    out = {}
    t = threading.Thread(target=lambda: out.update(solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 400)))
    t0 = time.perf_counter()
    t.start()
    time.sleep(0.02)
    solver.cancel()
    t.join()
    dt = time.perf_counter() - t0
    assert out["steps"].max() < 400 and dt < 1.0  # 400 steps of 4000 queries take ~1.5 s uncancelled
    assert np.isfinite(out["fitness"]).all()
    # the flag is cleared by the next solve: same result as a fresh solver
    a = solver.solve_batch(w.goal_params[:64], w.seeds[:64], w.rng_seeds[:64], 5)
    b = oracle.solve(w.robot, w.problem, oracle_lib.make_cfg(population=128), w.goal_params[:64], w.seeds[:64], w.rng_seeds[:64], 5)
    assert np.array_equal(a["solutions"], b["solutions"]) and a["steps"].min() == 5


@pytest.mark.parametrize("first", [False, True])
def test_balance_goal_on_gpu(oracle, first):
    """BalanceGoal (src/goal_types.cpp:231-272): 12 links with mass = 12 tip links, centre of mass accumulated in link order.
    Problems with more than 8 tips run the generic kernels; approximate fitness, trajectories and the islands driver are
    bit-identical to the oracle (which is pinned against the reference's own BalanceGoal class in test_reference_pin.py)."""
    rm, groups = robots.balancing_tree()
    g = groups["all"]
    bal = G.BalanceGoal((0.05, -0.02, 0.3), 0.8, axis=(0.1, 0.2, 0.97))
    gl = ([bal] if first else []) + [G.PoseGoal(g.tip_links[0])] + ([] if first else [bal]) + [G.PositionGoal(g.tip_links[1], weight=0.5)]
    pr = Problem().initialize(rm, g, gl)
    assert len(pr.tip_link_indices) == 12
    rng = np.random.default_rng(3)
    B, M, n = 64, 8, len(pr.active_variables)
    base = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    genes = base[:, pr.active_variables][:, None, :] + rng.normal(0, 0.2, (B, M, n))
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    solver = IKSolver(rm, population=24).initialize(pr)
    prim, sec = solver.approx_fitness(gp, seeds, base, genes)
    oprim, osec = oracle.approx_fitness(rm, pr, gp, seeds, base, genes)
    assert np.array_equal(prim, oprim) and np.abs(prim).min() > 0
    rs = (1 + np.arange(B)).astype(np.uint32)
    got = solver.trace(gp, seeds, rs, 6)
    want = oracle.solve(rm, pr, oracle_lib.make_cfg(population=24), gp, seeds, rs, 6)
    gpu_util.assert_bit_equal(got, want, what="balance")
    # a robot without inertials has nothing to balance
    rm0, groups0 = robots.random_tree(5, n_joints=9, branch_at=4)
    with pytest.raises(BioIKError):
        IKSolver(rm0).initialize(Problem().initialize(rm0, groups0["all"], [G.PoseGoal(groups0["all"].tip_links[0]), G.BalanceGoal()]))


@pytest.mark.parametrize("name,B", [("cfg2", 512), ("cfg3", 128), ("cfg5", 64)])
def test_gpu_against_the_reference_as_shipped(oracle, ref, name, B):
    """The GPU against the reference's own code with NOTHING swapped (libm sin / cos, oracle/_ref/libbioik_ref_strict.so), in the
    tolerance BASELINE.json names:
      * per-component quantities - exact FK tip frames, delta frames, approximate fitness - agree to 1e-12 (measured <= 3e-15: the
        contract sin / cos is <= 2 ulp from libm's);
      * whole trajectories cannot: one step() is 8 generations of argmin selection on pop=128 plus a line search on second
        differences, and the reference's own IEEE and -ffast-math builds already disagree after ONE step on 997 of 1000 queries
        (profiles/tolerance_study.py -> profiles/r02_tolerance_study.json).  What is comparable is the distribution: success rate
        within sampling error and the same median fitness scale after 25 steps."""
    w = workloads.make(name, ofk(oracle), batch=B)
    ref.keep_values("success", "fitness")  # compared as a distribution
    robot, gp = ref.effective_robot(w.robot), ref.effective_goal_params(w.robot, w.problem, w.goal_params, B)
    solver = IKSolver(robot, mode="bio2_memetic", population=128, random_seed=1, device=0).initialize(w.problem)
    rng = np.random.default_rng(0)
    n = len(w.problem.active_variables)
    base = workloads.sample_configurations(w.robot, w.problem.active_variables, B, rng)
    genes = base[:, w.problem.active_variables][:, None, :] + rng.normal(0, 0.05, (B, 8, n))
    stored = ref.approx_fitness(w.robot, w.problem, w.goal_params, w.seeds, base, genes)  # libm: the reference exactly as it is
    # its numbers: the oracle with libm sin / cos on the reference's link frames reproduces them bit for bit (checked against the stored digests)
    oracle.component_flags(1)
    try:
        r = dict(tips=oracle.fk(robot, w.problem, base, libm=True), delta=oracle.approx(robot, w.problem, base)[0], primary=oracle.approx_fitness(robot, w.problem, gp, w.seeds, base, genes)[0])
    finally:
        oracle.component_flags(0)
    for k in ("tips", "delta", "primary"):
        assert reference_store.same(r[k], stored[k]), k
    assert np.allclose(solver.fk(base), r["tips"], rtol=1e-12, atol=1e-12)
    assert np.allclose(solver.approx(base), np.where(np.abs(r["delta"]) > 0, r["delta"], solver.approx(base)), rtol=1e-10, atol=1e-12)
    prim, _ = solver.approx_fitness(gp, w.seeds, base, genes)
    assert np.allclose(prim, r["primary"], rtol=1e-12, atol=0)
    if name != "cfg2":
        return
    got = solver.solve_batch(gp, w.seeds, w.rng_seeds, 25)
    want = ref.solve(w.robot, w.problem, oracle_lib.make_cfg(population=128), w.goal_params, w.seeds, w.rng_seeds, 25)
    p = want["success"].mean()
    assert abs(got["success"].mean() - p) < 4 * np.sqrt(max(p * (1 - p), 1e-3) / B) + 1e-9
    assert np.median(got["fitness"]) < 1e-12 and np.median(want["fitness"]) < 1e-12
    # every successful answer really is a solution in the reference's own exact FK (1e-5 on the pose)
    tips = oracle.fk(w.robot, w.problem, got["solutions"], libm=True)[:, 0]
    ok = got["success"] != 0
    assert ok.sum() > 0.9 * B and np.abs(tips[ok, :3] - w.goal_params[ok, 0, :3]).max() < 1e-4


def test_cached_graph_survives_reallocation_by_the_device_entry_point(oracle):
    """ADVICE r01: bioik_solve_batch caches a CUDA graph that bakes in the addresses of the state, schedule and staging buffers;
    bioik_solve_batch_device with a larger batch or more steps reallocates them.  The cached graph must be dropped, not replayed on
    freed memory: solve_batch x2 (eager, then captured), a bigger device-pointer solve, solve_batch again - same bits as before."""
    torch = pytest.importorskip("torch")
    w = workloads.make("cfg2", ofk(oracle), batch=96)
    solver = gpu_util.make_solver(w, 32)
    first = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 5)
    second = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 5)  # captures the graph
    third = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 5)   # replays it
    for k in ("solutions", "fitness", "success"):
        assert np.array_equal(first[k], second[k]) and np.array_equal(first[k], third[k])
    big = workloads.make("cfg2", ofk(oracle), batch=700)
    dev = torch.device("cuda:0")
    gp, seeds = torch.from_numpy(big.goal_params).to(dev), torch.from_numpy(big.seeds).to(dev)
    rs = torch.from_numpy(big.rng_seeds.astype(np.int64)).to(dev).to(torch.int32)
    sol = torch.empty((700, big.robot.n_vars), dtype=torch.float64, device=dev)
    fit, succ, stp = torch.empty(700, dtype=torch.float64, device=dev), torch.empty(700, dtype=torch.int32, device=dev), torch.empty(700, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream()
    solver.solve_batch_device(700, gp.data_ptr(), seeds.data_ptr(), rs.data_ptr(), 40, False, sol.data_ptr(), fit.data_ptr(), succ.data_ptr(), stp.data_ptr(), stream=st.cuda_stream)  # larger B and more steps
    st.synchronize()
    solver.synchronize()  # torch's default stream is handle 0 = "use the context's own stream" for the ABI
    want = oracle.solve(big.robot, big.problem, oracle_lib.make_cfg(population=32), big.goal_params, big.seeds, big.rng_seeds, 40)
    assert np.array_equal(sol.cpu().numpy(), want["solutions"])
    again = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 5)
    for k in ("solutions", "fitness", "success"):
        assert np.array_equal(first[k], again[k]), k


def test_cancel_does_not_stick_to_the_next_device_solve(oracle):
    """ADVICE r01: bioik_cancel sets the device flag every kernel reads; like IKParallel::solve (src/ik_parallel.h:211-212) every
    solve entry point - the device-pointer one included - clears it when it starts, so a cancel that lands after a solve has finished
    does not turn the next solve into a no-op."""
    torch = pytest.importorskip("torch")
    w = workloads.make("cfg2", ofk(oracle), batch=64)
    solver = gpu_util.make_solver(w, 32)
    want = solver.solve_batch(w.goal_params, w.seeds, w.rng_seeds, 6)
    solver.cancel()
    torch.cuda.synchronize()  # the cancel's copy (its own stream) has landed: the flag is set on the device
    dev = torch.device("cuda:0")
    gp, seeds = torch.from_numpy(w.goal_params).to(dev), torch.from_numpy(w.seeds).to(dev)
    rs = torch.from_numpy(w.rng_seeds.astype(np.int64)).to(dev).to(torch.int32)
    sol = torch.empty((64, w.robot.n_vars), dtype=torch.float64, device=dev)
    fit, succ, stp = torch.empty(64, dtype=torch.float64, device=dev), torch.empty(64, dtype=torch.int32, device=dev), torch.empty(64, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream()
    solver.solve_batch_device(64, gp.data_ptr(), seeds.data_ptr(), rs.data_ptr(), 6, False, sol.data_ptr(), fit.data_ptr(), succ.data_ptr(), stp.data_ptr(), stream=st.cuda_stream)
    st.synchronize()
    solver.synchronize()  # torch's default stream is handle 0 = "use the context's own stream" for the ABI
    assert np.array_equal(sol.cpu().numpy(), want["solutions"]) and int(stp.min().item()) == 6
