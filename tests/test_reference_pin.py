"""Pins the oracle restatement against the REFERENCE'S OWN CODE.

oracle/_ref/libbioik_ref_strict.so is the reference's src/ik_evolution_2.cpp + src/problem.cpp (with every bio_ik
header they include: forward_kinematics.h, ik_base.h, utils.h, goal_types.h ...) compiled where they lie under
/root/reference through oracle/ref_harness.cpp, against the stand-in third-party headers of oracle/shims/.
Every comparison below is BIT-EXACT.  The oracle runs with one switch flipped: libm sin/cos (what the reference
calls, forward_kinematics.h:95-109) instead of the arithmetic contract's det_sincos, which is the single
documented numeric deviation of the product path (DESIGN.md §3, <= 2 ulp, tested in test_oracle.py).

The reference's answers come from tests/golden/reference/ (tests/reference_store.py), recorded from that library, which is
built by `make -C oracle ref` (done by __graft_entry__.build()) where the reference's sources are available.
"""
import numpy as np
import pytest

import oracle_lib
import reference_store
from bio_ik_b200 import goals as G, robots, workloads
from bio_ik_b200.problem import Problem

LIBM = 1  # oracle flag: libm sin/cos like the reference
STALE = 8  # oracle flag: emulate quirk Q2 (see test_stale_tip_quirk_is_confined_to_multi_tip_problems)
KEYS = ("solutions", "fitness", "success", "steps", "genes", "gradients", "species_fitness")
MODES = {"bio2": (0, 16), "bio2_memetic": ("q", 8), "bio2_memetic_l": ("l", 8)}


ref = reference_store.reference_fixture("reference_pin")


@pytest.fixture(scope="module")
def oracle():
    return oracle_lib.Oracle("strict")


def libm_fk(oracle):
    return lambda rm, pr, v: oracle.fk(rm, pr, v, libm=True)


def compare(oracle, ref, rm, pr, cfg, gp, seeds, rs, steps, early_exit=False):
    B = len(rs)
    gpe = ref.effective_goal_params(rm, pr, gp, B)
    a = oracle.solve(ref.effective_robot(rm), pr, cfg, gpe, seeds, rs, steps, early_exit=early_exit, flags=LIBM | STALE)
    b = ref.solve(rm, pr, cfg, gp, seeds, rs, steps, early_exit=early_exit)
    for k in KEYS:
        assert reference_store.same(a[k], b[k]), k
    return a


def test_lookup_tables_are_the_references(ref, oracle):
    """Random::Random (utils.h) fills both 2^23 tables from the seed; the oracle's Tables (and through it the product's make_tables) match it."""
    for seed in (1, 7):
        u, g = oracle.table_arrays(seed)
        assert reference_store.same(u, ref.table(0, seed))
        assert reference_store.same(g, ref.table(1, seed))


@pytest.mark.parametrize("mode", list(MODES))
def test_cfg2_trajectories(ref, oracle, mode):
    """BASELINE configs[1] shape at the reference's fixed population (2 parents + 16 children): the whole 25-step solve,
    every species' genes, gradients and fitness, the extracted solution and the success test."""
    memetic, gens = MODES[mode]
    B = 96
    w = workloads.make("cfg2", libm_fk(oracle), batch=B)
    cfg = oracle_lib.make_cfg(population=18, memetic=memetic, generations=gens)
    for steps in (1, 7, 25):
        compare(oracle, ref, w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, steps)
    a = compare(oracle, ref, w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 25, early_exit=True)
    assert len(set(a["steps"].tolist())) > 1  # early exit really happened on some queries


@pytest.mark.parametrize("population", [128, 64, 35, 4])
def test_baseline_population_sizes(ref, oracle, population):
    """The reference sizes its child pool to 2 + 16 in initialize() and drives every loop by children.size(); the harness
    re-sizes that public vector (ref_harness.cpp: setPopulation) so the reference's own code runs BASELINE.json's
    pop=128 (configs[1]) and pop=64 (configs[0]) - and odd / minimal pools - for the full 200 generations."""
    B = 48
    w = workloads.make("cfg2", libm_fk(oracle), batch=B)
    for mode in MODES:
        memetic, gens = MODES[mode]
        cfg = oracle_lib.make_cfg(population=population, memetic=memetic, generations=gens)
        compare(oracle, ref, w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 25)
    for name in ("cfg3", "cfg4", "cfg5"):
        w = workloads.make(name, libm_fk(oracle), batch=8)
        compare(oracle, ref, w.robot, w.problem, oracle_lib.make_cfg(population=population), w.goal_params, w.seeds, w.rng_seeds, 6)


@pytest.mark.parametrize("name,B,steps", [("cfg1", 1, 25), ("cfg3", 24, 10), ("cfg4", 12, 8), ("cfg5", 24, 10)])
def test_other_configs(ref, oracle, name, B, steps):
    """multi-tip (cfg3), secondary goals on a 30-DOF chain (cfg4), five position tips on a branching hand (cfg5)"""
    w = workloads.make(name, libm_fk(oracle), batch=B)
    for mode in ("bio2_memetic", "bio2"):
        memetic, gens = MODES[mode]
        cfg = oracle_lib.make_cfg(population=18, memetic=memetic, generations=gens)
        compare(oracle, ref, w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, steps)


def test_stale_tip_quirk_is_confined_to_multi_tip_problems(oracle):
    """Quirk Q2: the reference's computeApproximateMutation1 (forward_kinematics.h:940) skips the tips a variable does
    not move, so the memetic gradient probe (ik_evolution_2.cpp:469-470) scores those tips on stale frames left by an
    earlier call (uninitialised heap memory the first time; the harness pre-fills the buffer to make runs reproducible).
    The product path and the oracle's default implement out[t] = in[t] instead.  The emulation switch used by every
    comparison in this file changes nothing when each variable moves every tip (cfg2), and does change multi-tip
    memetic runs (cfg3) - which is why DESIGN.md lists Q2 as a deliberate deviation."""
    for name, differs in (("cfg2", False), ("cfg3", True)):
        w = workloads.make(name, libm_fk(oracle), batch=8)
        cfg = oracle_lib.make_cfg(population=18)
        a = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 3, flags=LIBM)
        b = oracle.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 3, flags=LIBM | STALE)
        assert np.array_equal(a["genes"], b["genes"]) != differs
        # without memetic steps the probe never runs
        cfg0 = oracle_lib.make_cfg(population=18, memetic=0, generations=16)
        a = oracle.solve(w.robot, w.problem, cfg0, w.goal_params, w.seeds, w.rng_seeds, 3, flags=LIBM)
        b = oracle.solve(w.robot, w.problem, cfg0, w.goal_params, w.seeds, w.rng_seeds, 3, flags=LIBM | STALE)
        assert np.array_equal(a["genes"], b["genes"])


def goal_zoo():
    rm, groups = robots.pr2_like()
    g = groups["all"]
    r, l = "r_wrist_roll_link", "l_wrist_roll_link"
    gl = [G.PoseGoal(r, (0.6, -0.2, 0.9), (0.1, 0.2, 0.3, 0.9)), G.PositionGoal(l, (0.5, 0.3, 1.0), 0.7), G.OrientationGoal(l, (0, 0.5, 0, 1), 1.3),
          G.LookAtGoal(r, (1, 0, 0), (2, 0.5, 1)), G.MaxDistanceGoal(l, (0.5, 0, 1), 0.3), G.MinDistanceGoal(r, (0.5, 0, 1), 0.6), G.LineGoal(r, (0.5, 0, 1), (1, 1, 0)),
          G.PlaneGoal(l, (0.5, 0, 1), (0, 1, 1)), G.SideGoal(r, (0, 0, 1), (0, 1, 0)), G.DirectionGoal(l, (1, 0, 0), (0, 0, 1)), G.JointVariableGoal("torso_lift_joint", 0.2, 2.0),
          G.AvoidJointLimitsGoal(1.5), G.CenterJointsGoal(0.5, secondary=False), G.RegularizationGoal(0.25), G.MinimalDisplacementGoal(2.0)]
    return rm, g, gl


def test_goal_classes_and_problem_initialize(ref, oracle):
    """Every goal class the device path implements except ConeGoal, evaluated by the reference's own goal_types.h
    on the reference's approximated frames; Problem::initialize's active-variable and tip order is asserted inside
    the harness against the flattened problem of bio_ik_b200.problem.Problem."""
    rm, g, gl = goal_zoo()
    pr = Problem().initialize(rm, g, gl)
    rng = np.random.default_rng(4)
    B, M, n = 24, 12, len(pr.active_variables)
    base = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    genes = base[:, pr.active_variables][:, None, :] + rng.normal(0, 0.2, (B, M, n))
    genes[:, :4] = base[:, pr.active_variables][:, None, :] + rng.normal(0, 1e-7, (B, 4, n))  # the memetic probe scale
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    gp[:, 0, 0:3] += rng.normal(0, 0.1, (B, 3))
    gpe = ref.effective_goal_params(rm, pr, gp, B)
    ref.keep_values("delta")  # compared where the variable moves the tip
    b = ref.approx_fitness(rm, pr, gp, seeds, base, genes)
    oracle.component_flags(LIBM)
    try:
        assert reference_store.same(oracle.fk(rm, pr, base, libm=True), b["tips"])
        delta, mask = oracle.approx(rm, pr, base)
        assert np.array_equal(delta[mask != 0], b["delta"][mask != 0])
        assert reference_store.same(oracle.approx_frames(rm, pr, base, genes), b["frames"])
        prim, sec = oracle.approx_fitness(rm, pr, gpe, seeds, base, genes)
    finally:
        oracle.component_flags(0)
    assert reference_store.same(prim, b["primary"]) and reference_store.same(sec, b["secondary"])
    assert np.abs(sec).min() > 0  # the secondary goals really contribute
    # ...and the same problem through whole solver steps
    cfg = oracle_lib.make_cfg(population=18)
    compare(oracle, ref, rm, pr, cfg, gp, seeds, 1 + np.arange(B, dtype=np.uint32), 4)


def test_cone_goal_is_the_one_exception(ref, oracle):
    """ConeGoal calls libm acos (goal_types.h:705); the arithmetic contract replaces it by det_acos (fdlibm algorithm,
    <= 1 ulp from libm, test_oracle.py).  Against the reference's own ConeGoal the approximate fitness therefore
    agrees to rounding, not to the bit."""
    rm, groups = robots.pr2_like()
    g = groups["all"]
    r, l = "r_wrist_roll_link", "l_wrist_roll_link"
    gl = [G.ConeGoal(r, (1, 0, 0), (0, 0.6, 0.8), 0.3, weight=0.5, position=(0.5, 0, 1), position_weight=0.7), G.ConeGoal(l, (0, 0, 1), (1, 0, 0), 1.2)]
    pr = Problem().initialize(rm, g, gl)
    rng = np.random.default_rng(5)
    B, M, n = 16, 8, len(pr.active_variables)
    base = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    genes = base[:, pr.active_variables][:, None, :] + rng.normal(0, 0.2, (B, M, n))
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    ref.keep_values("primary")
    b = ref.approx_fitness(rm, pr, gp, base, base, genes)
    oracle.component_flags(LIBM)
    try:
        prim, _ = oracle.approx_fitness(rm, pr, ref.effective_goal_params(rm, pr, gp, B), base, base, genes)
    finally:
        oracle.component_flags(0)
    assert np.allclose(prim, b["primary"], rtol=1e-13, atol=0)


def test_reference_with_contract_math_equals_the_default_oracle(ref, oracle):
    """The other direction: instead of giving the oracle libm, give the REFERENCE the contract's sin / cos / acos
    (ref_harness.cpp: the two unqualified calls of forward_kinematics.h:103-104 resolve to bio_ik::sin / cos; ConeGoal's
    acos through a shim hook).  The reference's code then equals the oracle in its default - product - arithmetic,
    ConeGoal included, which is what the GPU path is tested against."""
    ref.contract_math(True)
    try:
        for name, B, pop in (("cfg2", 48, 128), ("cfg2", 32, 18), ("cfg4", 8, 64)):
            w = workloads.make(name, lambda rm, pr, v: oracle.fk(rm, pr, v), batch=B)
            cfg = oracle_lib.make_cfg(population=pop)
            gpe = ref.effective_goal_params(w.robot, w.problem, w.goal_params, B)
            a = oracle.solve(ref.effective_robot(w.robot), w.problem, cfg, gpe, w.seeds, w.rng_seeds, 25)  # default flags: the arithmetic contract
            b = ref.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, 25)
            for k in KEYS:
                assert reference_store.same(a[k], b[k]), (name, k)
        # ConeGoal, now to the bit
        rm, groups = robots.pr2_like()
        g = groups["all"]
        gl = [G.ConeGoal("r_wrist_roll_link", (1, 0, 0), (0, 0.6, 0.8), 0.3, weight=0.5, position=(0.5, 0, 1), position_weight=0.7), G.ConeGoal("l_wrist_roll_link", (0, 0, 1), (1, 0, 0), 1.2)]
        pr = Problem().initialize(rm, g, gl)
        rng = np.random.default_rng(5)
        B, M, n = 16, 8, len(pr.active_variables)
        base = workloads.sample_configurations(rm, pr.active_variables, B, rng)
        genes = base[:, pr.active_variables][:, None, :] + rng.normal(0, 0.2, (B, M, n))
        gp = np.repeat(pr.default_goal_params()[None], B, 0)
        b = ref.approx_fitness(rm, pr, gp, base, base, genes)
        prim, _ = oracle.approx_fitness(ref.effective_robot(rm), pr, ref.effective_goal_params(rm, pr, gp, B), base, base, genes)
        assert reference_store.same(prim, b["primary"])
    finally:
        ref.contract_math(False)


def test_mimic_joints_and_prismatic(ref, oracle):
    """updateMimic, the mimic branches of the Jacobian and prismatic joints (forward_kinematics.h:640-760) in the reference's code"""
    rm, groups = robots.mimic_gripper_arm()
    g = groups[sorted(groups)[0]] if "all" not in groups else groups["all"]
    gl = [G.PositionGoal(t) for t in g.tip_links]
    pr = Problem().initialize(rm, g, gl)
    rng = np.random.default_rng(6)
    B = 16
    targets = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    tips = oracle.fk(rm, pr, targets, libm=True)
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    for gi, rec in enumerate(pr.goal_list):
        gp[:, gi, 0:3] = tips[:, rec["tip"], 0:3]
    for mode in ("bio2_memetic", "bio2_memetic_l", "bio2"):
        memetic, gens = MODES[mode]
        cfg = oracle_lib.make_cfg(population=18, memetic=memetic, generations=gens)
        compare(oracle, ref, rm, pr, cfg, gp, seeds, 11 + np.arange(B, dtype=np.uint32), 6)


def test_virtual_joints_that_mimic(ref, oracle):
    """a PLANAR joint mimicking a prismatic joint and a FLOATING joint mimicking a revolute one in the reference's code: updateMimic
    copies the first variable (forward_kinematics.h:230-246), the Jacobian reaches them through the numeric branch with ivar2 (:698-699)"""
    rm, groups = robots.mimic_virtual_joint_arm()
    g = groups["all"]
    pr = Problem().initialize(rm, g, [G.PoseGoal("ee"), G.PositionGoal("probe")])
    rng = np.random.default_rng(8)
    B = 12
    base = robots.mimic_virtual_joint_base(rm)
    targets = workloads.sample_configurations(rm, pr.active_variables, B, rng, base=base)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng, base=base)
    tips = oracle.fk(rm, pr, targets, libm=True)
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    gp[:, 0, 0:7], gp[:, 1, 0:3] = tips[:, 0, :], tips[:, 1, 0:3]
    for mode in ("bio2_memetic", "bio2_memetic_l", "bio2"):
        memetic, gens = MODES[mode]
        cfg = oracle_lib.make_cfg(population=18, memetic=memetic, generations=gens)
        compare(oracle, ref, rm, pr, cfg, gp, seeds, 11 + np.arange(B, dtype=np.uint32), 6)


@pytest.mark.parametrize("maker", ["floating_base_arm", "planar_base_arm"])
@pytest.mark.parametrize("group", ["whole_arm", "all"])
def test_floating_and_planar_joints(ref, oracle, group, maker):
    """a FLOATING base joint: the reference's own floating branch of getJointFrame (forward_kinematics.h:120-127), its numeric
    Jacobian (:695-726, frameTwist) and the quaternion-gene normalisation of reproduce() (ik_evolution_2.cpp:118-126,320-324)"""
    rm, groups = robots.floating_base_arm()
    g = groups[group]
    pr = Problem().initialize(rm, g, [G.PoseGoal(t) for t in g.tip_links])
    rng = np.random.default_rng(1)
    B = 12
    targets = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    tips = oracle.fk(rm, pr, targets, libm=True)
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    for gi, rec in enumerate(pr.goal_list):
        gp[:, gi, 0:7] = tips[:, rec["tip"], 0:7]
    for mode in MODES:
        memetic, gens = MODES[mode]
        for pop in (18, 64):
            compare(oracle, ref, rm, pr, oracle_lib.make_cfg(population=pop, memetic=memetic, generations=gens), gp, seeds, 1 + np.arange(B, dtype=np.uint32), 6)


def test_random_trees(ref, oracle):
    """randomly generated kinematic trees (mixed revolute / prismatic / fixed joints, unbounded variables)"""
    for seed in (1, 2, 3):
        rm, groups = robots.random_tree(seed)
        g = groups["all"]
        gl = [G.PoseGoal(t) for t in g.tip_links[:2]] + [G.PositionGoal(t) for t in g.tip_links[2:]]
        pr = Problem().initialize(rm, g, gl)
        rng = np.random.default_rng(seed)
        B = 8
        targets = workloads.sample_configurations(rm, pr.active_variables, B, rng)
        seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
        tips = oracle.fk(rm, pr, targets, libm=True)
        gp = np.repeat(pr.default_goal_params()[None], B, 0)
        for gi, rec in enumerate(pr.goal_list):
            gp[:, gi, 0:7] = tips[:, rec["tip"], 0:7]
        cfg = oracle_lib.make_cfg(population=18)
        compare(oracle, ref, rm, pr, cfg, gp, seeds, 5 + np.arange(B, dtype=np.uint32), 5)


def balance_problem(first=False):
    rm, groups = robots.balancing_tree()
    g = groups["all"]
    bal = G.BalanceGoal((0.05, -0.02, 0.3), 0.8, axis=(0.1, 0.2, 0.97))
    gl = ([bal] if first else []) + [G.PoseGoal(g.tip_links[0])] + ([] if first else [bal]) + [G.PositionGoal(g.tip_links[1], weight=0.5)]
    return rm, Problem().initialize(rm, g, gl)


def test_balance_goal_against_the_references_own_class(ref, oracle):
    """BalanceGoal (goal_types.h:540-568, src/goal_types.cpp:231-272, compiled in place through a urdf::ModelInterface shim that
    carries the link inertials): every link with mass becomes a tip link (12 here), the centre of mass is accumulated in link
    order.  Approximate fitness and whole solver trajectories are bit-identical to the reference's class.
    The reference can only take a BalanceGoal that is NOT the first goal of a query: BalanceGoal::describe reads
    GoalContext::getRobotModel() (goal_types.cpp:236) before Problem::initialize has set joint_model_group_ (problem.cpp:136 vs
    :180) - an uninitialised pointer that happens to hold the previous goal's value from the second goal on.  Oracle and device
    take it in any position (checked against each other below)."""
    rm, pr = balance_problem()
    assert len(pr.tip_link_indices) == 12 and pr.tip_link_indices[0] == 9  # the PoseGoal's tip first, then the links with mass in link order
    rng = np.random.default_rng(1)
    B, M, n = 12, 6, len(pr.active_variables)
    base = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    seeds = workloads.sample_configurations(rm, pr.active_variables, B, rng)
    genes = base[:, pr.active_variables][:, None, :] + rng.normal(0, 0.2, (B, M, n))
    gp = np.repeat(pr.default_goal_params()[None], B, 0)
    b = ref.approx_fitness(rm, pr, gp, seeds, base, genes)
    oracle.component_flags(LIBM)
    try:
        prim, _ = oracle.approx_fitness(ref.effective_robot(rm), pr, ref.effective_goal_params(rm, pr, gp, B), seeds, base, genes)
    finally:
        oracle.component_flags(0)
    assert reference_store.same(prim, b["primary"]) and np.abs(prim).min() > 0
    compare(oracle, ref, rm, pr, oracle_lib.make_cfg(population=18), gp, seeds, 1 + np.arange(B, dtype=np.uint32), 5)
    # the goal really contributes: without it the fitness differs
    rm2, groups2 = robots.balancing_tree()
    pr0 = Problem().initialize(rm2, groups2["all"], [G.PoseGoal(groups2["all"].tip_links[0]), G.PositionGoal(groups2["all"].tip_links[1], weight=0.5)])
    p0, _ = oracle.approx_fitness(rm2, pr0, np.repeat(pr0.default_goal_params()[None], B, 0), seeds, base, genes)
    assert not np.array_equal(p0, prim)
