"""TEST INFRASTRUCTURE ONLY -- generate ``tests/golden/*.npz`` from the UNMODIFIED reference.

Run in the build container (where ``/root/reference`` exists):

    PYTHONDONTWRITEBYTECODE=1 OMP_NUM_THREADS=1 python -m oracle.make_golden

Every fixture stores the *outputs of the reference itself* (``mici`` imported from
``/root/reference/src``) for inputs that are regenerated deterministically from
``mici_b200.problems`` (seeded), plus a checksum of those inputs.  The GPU box has no
``/root/reference``; there the fixtures are the pinned statement of the reference's behaviour
that both the oracle port (``tests/test_oracle.py``) and the CUDA path
(``tests/test_parity_gpu.py``) are compared against.
"""

from __future__ import annotations

import os

import numpy as np

from mici_b200 import problems as pb

from . import drivers as dr

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name -> (config, problem kwargs, step counts, integrator overrides)
CASES = {
    "c0_std_gaussian": ("C0", {}, (1, 5, 20), {}),
    "c1_funnel_dense": ("C1", {"n_chains": 32}, (1, 5, 20), {}),
    "c1_funnel_dense_d24": ("C1", {"n_chains": 16, "dim": 24}, (1, 20), {}),
    "c1_funnel_diag": ("C1", {"n_chains": 16, "dim": 40, "metric_kind": "diagonal"}, (1, 20), {}),
    "c1_funnel_identity": ("C1", {"n_chains": 16, "dim": 7, "metric_kind": "identity"}, (1, 20), {}),
    "c2_softabs_banana": ("C2", {"n_chains": 16}, (1, 5, 20), {}),
    "c2_softabs_banana_d8": ("C2", {"n_chains": 32, "dim": 8}, (1, 5, 20), {}),
    # beyond shared memory: the SoftAbs matrices live in the per-CTA global workspace
    "c2_softabs_banana_d128": ("C2", {"n_chains": 6, "dim": 128}, (1, 3), {}),
    "c6_softabs_quartic_d160": ("C6", {"n_chains": 4, "dim": 160}, (1, 2), {}),
    # SoftAbs on a target with a DENSE Hessian and third-derivative tensor
    "c6_softabs_quartic_d12": ("C6", {"n_chains": 16, "dim": 12}, (1, 5, 20), {}),
    "c6_softabs_quartic_d64": ("C6", {"n_chains": 12, "dim": 64}, (1, 5), {}),
    "c3_torus": ("C3", {"n_chains": 64}, (1, 5, 20), {}),
    "c3_torus_inner3": ("C3", {"n_chains": 32}, (1, 5), {"n_inner_step": 3}),
    # GaussianEuclideanMetricSystem (exact h2 flow in the eigenbasis of the metric)
    "n4_gaussian_split_dense_d32": ("G1", {"n_chains": 12}, (1, 5, 20), {}),
    "n4_gaussian_split_diag_d40": ("G1", {"n_chains": 8, "dim": 40, "metric_kind": "diagonal"}, (1, 20), {}),
    "n4_gaussian_split_identity_funnel_d9": ("G1", {"n_chains": 8, "dim": 9, "metric_kind": "identity", "target": "neal_funnel"}, (1, 20), {}),
    "n4_gaussian_split_bcss3_dense_d70": ("G1", {"n_chains": 6, "dim": 70, "integrator": "bcss3"}, (1, 5), {}),
    "n4_bcss2_funnel_d24": ("C1", {"n_chains": 12, "dim": 24, "integrator": "bcss2"}, (1, 5, 20), {}),
    "n4_bcss3_funnel_d40_diag": ("C1", {"n_chains": 8, "dim": 40, "metric_kind": "diagonal", "integrator": "bcss3"}, (1, 20), {}),
    "n4_bcss4_funnel_d130": ("C1", {"n_chains": 6, "dim": 130, "integrator": "bcss4"}, (1, 5), {}),
    "n4_midpoint_softabs_d8": ("C2", {"n_chains": 16, "dim": 8, "integrator": "implicit_midpoint"}, (1, 5, 20), {}),
    "n4_midpoint_dense_d32": ("C4", {"n_chains": 6, "dim": 32, "integrator": "implicit_midpoint"}, (1, 5), {}),
    "n4_steffensen_softabs_d8": ("C2", {"n_chains": 16, "dim": 8}, (1, 5), {"fixed_point_solver": "steffensen"}),
    "n4_steffensen_midpoint_dense_d16": ("C4", {"n_chains": 6, "dim": 16, "integrator": "implicit_midpoint"}, (1, 5), {"fixed_point_solver": "steffensen"}),
    "n4_quasi_newton_torus": ("C3", {"n_chains": 32}, (1, 5, 20), {"projection_solver": "quasi_newton"}),
    "n4_line_search_torus": ("C3", {"n_chains": 32}, (1, 5, 20), {"projection_solver": "newton_with_line_search"}),
    "n4_quasi_newton_sphere_dense_d10": ("S1", {"n_chains": 16, "dim": 10}, (1, 5), {"projection_solver": "quasi_newton", "n_inner_step": 2}),
    "n4_line_search_sphere_diag_d12": ("S1", {"n_chains": 16, "dim": 12, "metric_kind": "diagonal"}, (1, 5), {"projection_solver": "newton_with_line_search"}),
    "s1_sphere_dense_d10": ("S1", {"n_chains": 32, "dim": 10}, (1, 5, 20), {}),
    "s1_sphere_diag_d70_inner2": ("S1", {"n_chains": 8, "dim": 70, "metric_kind": "diagonal"}, (1, 5), {"n_inner_step": 2}),
    "s1_sphere_identity_d5": ("S1", {"n_chains": 16, "dim": 5, "metric_kind": "identity"}, (1, 20), {}),
    # density with respect to the Lebesgue measure (dens_wrt_hausdorff=False): h1 carries
    # log det gram / 2, dh1_dpos the constraint's matrix-Hessian product
    "c3_torus_lebesgue": ("C3", {"n_chains": 32, "dens_wrt_hausdorff": False}, (1, 5, 20), {}),
    "s1_sphere_dense_d10_lebesgue": ("S1", {"n_chains": 16, "dim": 10, "dens_wrt_hausdorff": False}, (1, 5, 20), {}),
    # several constraints: full C x C Gram / residual-Jacobian matrices (C = 2, 4, 8)
    "s2_multi_sphere_c2_identity_d12": ("S2", {"n_chains": 16, "dim": 12, "n_constr": 2, "metric_kind": "identity"}, (1, 5, 20), {}),
    "s2_multi_sphere_c4_dense_d16": ("S2", {"n_chains": 16, "dim": 16, "n_constr": 4}, (1, 5, 20), {}),
    "s2_multi_sphere_c8_dense_d32_lebesgue": ("S2", {"n_chains": 12, "dim": 32, "n_constr": 8, "dens_wrt_hausdorff": False}, (1, 5), {}),
    "s2_multi_sphere_c4_diag_d72_inner2": ("S2", {"n_chains": 8, "dim": 72, "n_constr": 4, "metric_kind": "diagonal"}, (1, 5), {"n_inner_step": 2}),
    "s2_multi_sphere_c8_quasi_newton_d16": ("S2", {"n_chains": 12, "dim": 16, "n_constr": 8}, (1, 5), {"projection_solver": "quasi_newton"}),
    "c4_dense_riemannian_d64": ("C4", {"n_chains": 8, "dim": 64}, (1, 5), {}),
    "c4_dense_riemannian_d512": ("C4", {"n_chains": 8, "dim": 512}, (1, 5), {}),
    # full-rank position-dependent metric M(q) = B + c (q q^T) o S: generic dense path only
    "c5_hadamard_d24": ("C5", {"n_chains": 8, "dim": 24}, (1, 5, 20), {}),
    "c5_hadamard_d100": ("C5", {"n_chains": 6, "dim": 100}, (1, 5), {}),
    "c5_hadamard_d512": ("C5", {"n_chains": 8, "dim": 512}, (1, 5), {}),
}

# failure-path fixtures: step sizes chosen so that some chains raise IntegratorError
FAILURE_CASES = {
    "c2_softabs_banana_bigstep": ("C2", {"n_chains": 32, "dim": 8}, 0.6, (3,), {}),
    "c3_torus_bigstep": ("C3", {"n_chains": 64}, 0.4, (3,), {}),
    "n4_quasi_newton_torus_bigstep": ("C3", {"n_chains": 64}, 0.4, (3,), {"projection_solver": "quasi_newton"}),
    "n4_line_search_torus_bigstep": ("C3", {"n_chains": 64}, 0.45, (3,), {"projection_solver": "newton_with_line_search"}),
    "n4_midpoint_softabs_bigstep": ("C2", {"n_chains": 32, "dim": 8, "integrator": "implicit_midpoint"}, 0.9, (3,), {}),
}


def input_checksum(problem):
    return np.array([problem.pos.sum(), problem.mom.sum(), np.abs(problem.pos).sum()])


def mixed_dirs(n):
    d = np.ones(n, dtype=np.int32)
    d[1::3] = -1
    return d


def generate_case(name, cfg, kwargs, step_counts, overrides, step_size=None):
    problem = pb.make_problem(cfg, **kwargs)
    if step_size is not None:
        problem.step_size = step_size
    dirs = mixed_dirs(problem.n_chains)
    out = {
        "input_checksum": input_checksum(problem),
        "dirs": dirs,
        "step_size": np.array(problem.step_size),
        "step_counts": np.array(step_counts),
    }
    for n_steps in step_counts:
        r = dr.reference_run(problem, n_steps, dirs=dirs, **overrides)
        o = dr.oracle_run(problem, n_steps, dirs=dirs, **overrides)
        assert np.array_equal(r["status"], o["status"]), (name, r["status"], o["status"])
        assert np.array_equal(r["n_done"], o["n_done"]), name
        np.testing.assert_allclose(o["pos"], r["pos"], rtol=1e-12, atol=1e-14, err_msg=name)
        np.testing.assert_allclose(o["mom"], r["mom"], rtol=1e-12, atol=1e-14, err_msg=name)
        for key in ("pos", "mom", "status", "n_done", "h", "h_init"):
            out[f"{key}_{n_steps}"] = r[key]
        n_fail = int((r["status"] != 0).sum())
        print(f"{name:32s} steps={n_steps:3d} chains={problem.n_chains:3d} failed={n_fail}")
    np.savez(os.path.join(GOLDEN_DIR, name + ".npz"), **out)


def solver_known_answers():
    """Reference ``solve_fixed_point_direct`` on its own test problems
    (reference tests/test_solvers.py:25-39)."""
    mici = dr.import_reference()
    y = np.array([3.0, 5.0, 7.0])
    probs = {
        "babylonian": (lambda x: (y / x + x) / 2, np.ones_like(y)),
        "ratio": (lambda x: (x + y) / (x + 1), np.ones_like(y)),
        "cosine": (lambda x: np.cos(x), np.array([1.0])),
    }
    out = {}
    for k, (f, x0) in probs.items():
        for tol in (1e-6, 1e-8, 1e-10):
            out[f"{k}_{tol:g}"] = mici.solvers.solve_fixed_point_direct(f, x0, convergence_tol=tol)
            out[f"steffensen_{k}_{tol:g}"] = mici.solvers.solve_fixed_point_steffensen(
                f, x0, convergence_tol=tol)
    np.savez(os.path.join(GOLDEN_DIR, "solver_known_answers.npz"), **out)


HMC_CASES = {
    # name -> (config, kwargs, n_iter, n_step, seed)
    "hmc_c1_funnel_d16": ("C1", {"n_chains": 12, "dim": 16}, 6, 5, 11),
    "hmc_c0_std_gaussian": ("C0", {"n_chains": 6, "dim": 10}, 8, 7, 12),
    # momentum refresh of the non-Euclidean systems (sqrt(M(q)) z; cotangent-space projection)
    "hmc_c2_softabs_d8": ("C2", {"n_chains": 6, "dim": 8}, 4, 3, 13),
    "hmc_c4_dense_d12": ("C4", {"n_chains": 6, "dim": 12}, 4, 3, 14),
    "hmc_c3_torus": ("C3", {"n_chains": 10}, 6, 4, 15),
    # per-chain random trajectory lengths (MetropolisRandomIntegrationTransition)
    "hmc_c1_random_n_step": ("C1", {"n_chains": 10, "dim": 16}, 6, (2, 9), 17),
    "hmc_g1_gaussian_split_d16": ("G1", {"n_chains": 8, "dim": 16}, 6, 4, 18),
    "hmc_s1_sphere_d20_dense": ("S1", {"n_chains": 6, "dim": 20, "metric_kind": "dense"}, 5, 4, 16),
}


# step sizes chosen so that the fixtures contain rejections (and, for the implicit / constrained
# integrators, a few failed trajectories)
HMC_STEP_SIZES = {
    "hmc_c1_funnel_d16": 0.35,
    "hmc_c1_random_n_step": 0.35,
    "hmc_g1_gaussian_split_d16": 0.5,
    "hmc_c2_softabs_d8": 0.3,
    "hmc_c4_dense_d12": 0.8,
    "hmc_c3_torus": 0.25,
    "hmc_s1_sphere_d20_dense": 0.2,
}


def hmc_cases():
    """Static-HMC transitions (row N1) through the reference's own transition classes."""
    for name, (cfg, kwargs, n_iter, n_step, seed) in HMC_CASES.items():
        problem = pb.make_problem(cfg, **kwargs)
        if name in HMC_STEP_SIZES:
            problem.step_size = HMC_STEP_SIZES[name]
        r = dr.reference_hmc(problem, n_iter, n_step, seed)
        o = dr.oracle_hmc(problem, n_iter, n_step, seed)
        np.testing.assert_allclose(o["pos"], r["pos"], rtol=1e-12, atol=1e-14, err_msg=name)
        np.testing.assert_array_equal(o["dir"], r["dir"])
        np.testing.assert_allclose(o["metrop_accept_prob"], r["metrop_accept_prob"], rtol=1e-10)
        acc = float(o["accepted"].mean())
        print(f"{name:32s} iters={n_iter} n_step={n_step} accept rate={acc:.2f}")
        np.savez(os.path.join(GOLDEN_DIR, name + ".npz"), input_checksum=input_checksum(problem),
                 step_size=np.array(problem.step_size), accepted=o["accepted"],
                 **{k: r[k] for k in ("pos", "dir", "n_step", "metrop_accept_prob", "accept_stat")})


NUTS_CASES = {
    # name -> (config, kwargs, step_size, n_iter, seed, options): dynamic integration transitions
    # (row N4) through the reference's own transition classes (transitions.py:487-858)
    "nuts_c1_multinomial_d10": ("C1", {"n_chains": 8, "dim": 10}, 0.2, 6, 77, {}),
    "nuts_c1_slice_euclidean_d16": ("C1", {"n_chains": 8, "dim": 16}, 0.15, 5, 78,
                                    {"variant": "slice", "criterion": "euclidean"}),
    "nuts_c0_depth4_no_extra_checks": ("C0", {"n_chains": 6, "dim": 10}, 0.3, 6, 79,
                                       {"max_tree_depth": 4, "extra_checks": False}),
    "nuts_c1_diag_divergent": ("C1", {"n_chains": 8, "dim": 8, "metric_kind": "diagonal"}, 0.9, 6,
                               80, {"max_delta_h": 5.0}),
    "nuts_c1_identity_d70": ("C1", {"n_chains": 4, "dim": 70, "metric_kind": "identity"}, 0.05, 3,
                             81, {"max_tree_depth": 6}),
    # constrained and implicit integrators inside dynamic transitions: pins the oracle for the
    # systems the fused kernel does not cover yet (failed steps terminate the tree)
    "nuts_c3_torus_constrained": ("C3", {"n_chains": 6}, 0.2, 5, 82, {"max_tree_depth": 5}),
    "nuts_c2_softabs_d4_implicit": ("C2", {"n_chains": 3, "dim": 4}, 0.2, 4, 83,
                                    {"max_tree_depth": 3}),
}
NUTS_DEVICE_CASES = [k for k in NUTS_CASES if not k.startswith(("nuts_c3", "nuts_c2"))]


def nuts_cases():
    import warnings

    for name, (cfg, kwargs, eps, n_iter, seed, opts) in NUTS_CASES.items():
        problem = pb.make_problem(cfg, **kwargs)
        problem.step_size = eps
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            r = dr.reference_nuts(problem, n_iter, seed, **opts)
            o = dr.oracle_nuts(problem, n_iter, seed, **opts)
        for k in r:
            np.testing.assert_allclose(o[k], r[k], rtol=1e-12, atol=1e-14, err_msg=f"{name} {k}")
        print(f"{name:34s} mean n_step={r['n_step'].mean():5.1f} depths={np.unique(r['tree_depth'])}"
              f" diverging={int(r['diverging'].sum())}")
        np.savez(os.path.join(GOLDEN_DIR, name + ".npz"), input_checksum=input_checksum(problem),
                 step_size=np.array(eps), **r)


ADAPT_CASES = {
    # name -> (config, kwargs, adapter specs, windowed-stager kwargs or None, n_warm_up, n_main,
    #          n_step, seed): staged adaptive sampling (row N3) through the reference's own
    # StaticMetropolisHMC.sample_chains with its adapters and stagers
    "adapt_c1_dualavg_variance": (
        "C1", {"n_chains": 6, "dim": 16}, [("dual_averaging", {}), ("online_variance", {})],
        {"n_init_slow_window_iter": 5, "n_init_fast_stage_iter": 4, "n_final_fast_stage_iter": 3},
        20, 5, 4, 21),
    "adapt_c1_dualavg_covariance": (
        "C1", {"n_chains": 5, "dim": 12},
        [("dual_averaging", {"log_step_size_reducer": "geometric_mean_log_step_size_reducer"}),
         ("online_covariance", {})],
        {"n_init_slow_window_iter": 8, "n_init_fast_stage_iter": 5, "n_final_fast_stage_iter": 4},
        40, 6, 5, 33),
    "adapt_c0_dualavg_min": (
        "C0", {"n_chains": 4, "dim": 10},
        [("dual_averaging", {"adapt_stat_target": 0.65,
                             "log_step_size_reducer": "min_log_step_size_reducer"})],
        None, 15, 5, 6, 33),
    # step-size adaptation of the constrained and the implicit integrators (per-chain step sizes
    # in the device kernels; failed steps drive the coarse initial search)
    "adapt_c3_torus_dualavg": (
        "C3", {"n_chains": 6}, [("dual_averaging", {})], None, 15, 5, 4, 41),
    "adapt_c2_softabs_d6_dualavg": (
        "C2", {"n_chains": 4, "dim": 6}, [("dual_averaging", {})], None, 10, 3, 3, 42),
    "adapt_c0_variance_first": (
        "C0", {"n_chains": 4, "dim": 10},
        [("online_variance", {"reg_iter_offset": 3}), ("dual_averaging", {})], None, 30, 4, 3, 33),
    # the reference's default sampler: DynamicMultinomialHMC with dual averaging (n_step = the
    # keyword arguments of the dynamic transition)
    "adapt_nuts_c0_dualavg": (
        "C0", {"n_chains": 4, "dim": 10}, [("dual_averaging", {})], None, 12, 4,
        {"max_tree_depth": 5}, 51),
    "adapt_nuts_c1_dualavg_variance": (
        "C1", {"n_chains": 4, "dim": 8, "metric_kind": "diagonal"},
        [("dual_averaging", {}), ("online_variance", {})],
        {"n_init_slow_window_iter": 6, "n_init_fast_stage_iter": 4, "n_final_fast_stage_iter": 3},
        16, 3, {"max_tree_depth": 6, "variant": "slice", "criterion": "euclidean"}, 52),
}
STAGE_CODES = {None: 0, "fast": 1, "all": 2}


def reference_stage_list(specs, stager_kwargs, n_warm_up_iter, n_main_iter):
    """Stage list ``[(n_iter, None | "fast" | "all")]`` from the reference's own stagers
    (default choice as in samplers.py:1075-1082)."""
    mici = dr.import_reference()

    class _Flag:
        def __init__(self, fast):
            self.is_fast = fast

    flags = [_Flag(name == "dual_averaging") for name, _ in specs]
    if stager_kwargs is not None:
        stager = mici.stagers.WindowedWarmUpStager(**stager_kwargs)
    elif all(f.is_fast for f in flags):
        stager = mici.stagers.WarmUpStager()
    else:
        stager = mici.stagers.WindowedWarmUpStager()
    stages = stager.stages(n_warm_up_iter, n_main_iter, {"k": flags}, None)
    return [(v.n_iter, None if v.adapters is None else
             ("all" if len(v.adapters["k"]) == len(flags) else "fast")) for v in stages.values()]


def adapt_cases():
    import warnings

    for name, (cfg, kwargs, specs, sk, n_warm, n_main, n_step, seed) in ADAPT_CASES.items():
        problem = pb.make_problem(cfg, **kwargs)
        stages = reference_stage_list(specs, sk, n_warm, n_main)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")  # overflow in the coarse step-size search (eps = 1)
            dyn = n_step if isinstance(n_step, dict) else None
            r = dr.reference_sample_chains(problem, n_warm, n_main, n_step, seed, specs, sk,
                                           dynamic=dyn)
            o = dr.oracle_sample_chains(problem, stages, n_step, seed, specs, dynamic=dyn)
        for k in r:
            np.testing.assert_allclose(o[k], r[k], rtol=1e-12, atol=1e-14, err_msg=f"{name} {k}")
        print(f"{name:32s} stages={stages} step_size={float(r['step_size']):.4f} "
              f"accept={r['accept_stat'].mean():.2f}")
        np.savez(os.path.join(GOLDEN_DIR, name + ".npz"), input_checksum=input_checksum(problem),
                 stage_n_iter=np.array([s[0] for s in stages]),
                 stage_which=np.array([STAGE_CODES[s[1]] for s in stages]),
                 step_size_trace=o["step_size_trace"], **r)


# the three step fixtures that tests/test_oracle.py also checks at 5 steps with tighter tolerances
REFERENCE_5_STEP_CASES = ("c1_funnel_dense_d24", "c2_softabs_banana_d8", "c3_torus_inner3")


def reference_5_steps():
    """Five reference steps of each of ``REFERENCE_5_STEP_CASES`` (same inputs and directions
    as the step fixtures), in one file."""
    out = {}
    for name in REFERENCE_5_STEP_CASES:
        cfg, kwargs, _, overrides = CASES[name]
        problem = pb.make_problem(cfg, **kwargs)
        r = dr.reference_run(problem, 5, dirs=mixed_dirs(problem.n_chains), **overrides)
        out[f"{name}_input_checksum"] = input_checksum(problem)
        for key in ("status", "pos", "mom"):
            out[f"{name}_{key}"] = r[key]
    np.savez(os.path.join(GOLDEN_DIR, "reference_5_steps.npz"), **out)


DROPIN_CASES = {
    # name: (config, kwargs, sampler, n_iter, sampler kwargs); seed DROPIN_SEED
    "c1_static": ("C1", {"n_chains": 4, "dim": 16}, "StaticMetropolisHMC", 6, {"n_step": 5}),
    "c0_static": ("C0", {"n_chains": 4, "dim": 10}, "StaticMetropolisHMC", 6, {"n_step": 7}),
    "c3_static": ("C3", {"n_chains": 4}, "StaticMetropolisHMC", 5, {"n_step": 4}),
    "c2_static": ("C2", {"n_chains": 3, "dim": 8}, "StaticMetropolisHMC", 3, {"n_step": 3}),
    "c4_static": ("C4", {"n_chains": 3, "dim": 12}, "StaticMetropolisHMC", 3, {"n_step": 3}),
    "c1_dynamic": ("C1", {"n_chains": 4, "dim": 10}, "DynamicMultinomialHMC", 4,
                   {"max_tree_depth": 4}),
    "c2_dynamic": ("C2", {"n_chains": 2, "dim": 8}, "DynamicMultinomialHMC", 2,
                   {"max_tree_depth": 3}),
}
DROPIN_SEED = 4242
DROPIN_STATS = ("n_step", "accept_stat", "convergence_error", "non_reversible_step")


def dropin_cases():
    """The reference's own samplers (``sample_chains``, one worker, no adapters) over the
    reference's own system and integrator: final positions, position traces and statistics,
    all ``[chain, ...]``."""
    mici = dr.import_reference()
    for name, (cfg, kwargs, sampler_name, n_iter, skw) in DROPIN_CASES.items():
        problem = pb.make_problem(cfg, **kwargs)
        system, integrator = dr.build_reference(problem)
        sampler = getattr(mici.samplers, sampler_name)(
            system, integrator, np.random.default_rng(DROPIN_SEED), **skw)
        init = [mici.states.ChainState(pos=problem.pos[i].copy(), mom=None, dir=1)
                for i in range(problem.n_chains)]
        final, traces, stats = sampler.sample_chains(
            0, n_iter, init, adapters=[], n_worker=1, display_progress=False,
            trace_funcs=[lambda state: {"pos": state.pos}])
        print(f"dropin_{name:24s} accept={np.mean(stats['accept_stat']):.2f}")
        np.savez(os.path.join(GOLDEN_DIR, f"dropin_{name}.npz"),
                 input_checksum=input_checksum(problem),
                 final_pos=np.stack([np.asarray(s.pos) for s in final]),
                 trace_pos=np.asarray(traces["pos"]),
                 **{k: np.asarray(stats[k]) for k in DROPIN_STATS})


def main(argv=None):
    """No arguments: regenerate every fixture.  With arguments: only the named step fixtures
    (keys of CASES / FAILURE_CASES)."""
    import sys  # noqa: PLC0415

    names = list(sys.argv[1:] if argv is None else argv)
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    if names:
        for name in names:
            if name in CASES:
                cfg, kwargs, steps, ov = CASES[name]
                generate_case(name, cfg, kwargs, steps, ov)
            else:
                cfg, kwargs, eps, steps, ov = FAILURE_CASES[name]
                generate_case(name, cfg, kwargs, steps, ov, step_size=eps)
        return
    hmc_cases()
    nuts_cases()
    adapt_cases()
    for name, (cfg, kwargs, steps, ov) in CASES.items():
        generate_case(name, cfg, kwargs, steps, ov)
    for name, (cfg, kwargs, eps, steps, ov) in FAILURE_CASES.items():
        generate_case(name, cfg, kwargs, steps, ov, step_size=eps)
    solver_known_answers()
    reference_5_steps()
    dropin_cases()


if __name__ == "__main__":
    main()
