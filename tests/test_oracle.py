"""CPU tests: the oracle port against the committed reference fixtures and the reference's own
solver known answers."""

import numpy as np
import pytest

from oracle import drivers as dr
from oracle import mici_oracle as mo
from oracle.make_golden import REFERENCE_5_STEP_CASES

from golden_util import assert_matches_golden, case_names, load_case

HMC_NAMES = ["hmc_c1_funnel_d16", "hmc_c0_std_gaussian", "hmc_c2_softabs_d8", "hmc_c4_dense_d12",
             "hmc_c3_torus", "hmc_s1_sphere_d20_dense", "hmc_c1_random_n_step",
             "hmc_g1_gaussian_split_d16"]


@pytest.mark.parametrize("name", case_names() + case_names(failures=True))
def test_oracle_matches_reference_fixture(name):
    problem, dirs, overrides, g = load_case(name)
    if problem.dim >= 512:
        pytest.skip("large-D fixture checked in test_oracle_large (slow)")
    for n_steps in g["step_counts"]:
        out = dr.oracle_run(problem, int(n_steps), dirs=dirs, **overrides)
        assert_matches_golden(out, g, int(n_steps), rtol=1e-12, atol=1e-14, label=name)


def test_oracle_large_dim_fixture():
    problem, dirs, overrides, g = load_case("c4_dense_riemannian_d512")
    out = dr.oracle_run(problem, 1, dirs=dirs, **overrides)
    assert_matches_golden(out, g, 1, rtol=1e-12, atol=1e-14)


def test_failure_fixtures_cover_both_error_kinds():
    _, _, _, g = load_case("c3_torus_bigstep")
    st = g["status_3"]
    assert (st == mo.STATUS_OK).any() and (st == mo.STATUS_CONVERGENCE).any()
    assert (st == mo.STATUS_NON_REVERSIBLE).any()


# reference tests/test_solvers.py:25-39, 65-121
Y = np.array([3.0, 5.0, 7.0])
FIXED_POINT_PROBLEMS = {
    "babylonian": (lambda x: (Y / x + x) / 2, Y**0.5, np.ones_like(Y)),
    "ratio": (lambda x: (x + Y) / (x + 1), Y**0.5, np.ones_like(Y)),
    "cosine": (lambda x: np.cos(x), np.array([0.7390851332151607]), np.array([1.0])),
}


@pytest.mark.parametrize("prob", list(FIXED_POINT_PROBLEMS))
@pytest.mark.parametrize("tol", [1e-6, 1e-8, 1e-10])
def test_fixed_point_direct_known_answers(prob, tol):
    import os

    from oracle.make_golden import GOLDEN_DIR

    func, fixed_point, x0 = FIXED_POINT_PROBLEMS[prob]
    x, _ = mo.solve_fixed_point_direct(func, x0, convergence_tol=tol)
    assert mo.maximum_norm(x - fixed_point) < tol
    g = np.load(os.path.join(GOLDEN_DIR, "solver_known_answers.npz"))
    np.testing.assert_array_equal(x, g[f"{prob}_{tol:g}"])  # same iterate sequence
    xs, _ = mo.solve_fixed_point_steffensen(func, x0, convergence_tol=tol)
    assert mo.maximum_norm(xs - fixed_point) < tol
    np.testing.assert_array_equal(xs, g[f"steffensen_{prob}_{tol:g}"])


@pytest.mark.parametrize("func", [lambda x: 2 * x, lambda x: 1 + x**2])
def test_fixed_point_direct_divergence(func):
    with pytest.raises(mo.OracleIntegratorError):
        mo.solve_fixed_point_direct(func, np.arange(3.0), max_iters=10000)


def test_fixed_point_direct_max_iters():
    with pytest.raises(mo.OracleIntegratorError):
        mo.solve_fixed_point_direct(np.cos, np.array([1.0]), convergence_tol=1e-10, max_iters=1)


def test_fixed_point_direct_handles_value_error():
    def func(_):
        raise ValueError

    with pytest.raises(mo.OracleIntegratorError):
        mo.solve_fixed_point_direct(func, np.array([1.0]))


@pytest.mark.parametrize("name", REFERENCE_5_STEP_CASES)
def test_oracle_matches_reference_5_steps(name):
    """Five steps against the reference's own (tests/golden/reference_5_steps.npz), with tighter
    tolerances than the step fixtures."""
    import os

    from oracle.make_golden import GOLDEN_DIR, input_checksum

    problem, dirs, overrides, _ = load_case(name)
    r = np.load(os.path.join(GOLDEN_DIR, "reference_5_steps.npz"))
    np.testing.assert_allclose(input_checksum(problem), r[f"{name}_input_checksum"], rtol=1e-13)
    o = dr.oracle_run(problem, 5, dirs=dirs, **overrides)
    np.testing.assert_array_equal(o["status"], r[f"{name}_status"])
    np.testing.assert_allclose(o["pos"], r[f"{name}_pos"], rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(o["mom"], r[f"{name}_mom"], rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("name", HMC_NAMES)
def test_oracle_hmc_transition_matches_reference_fixture(name):
    """Row N1: momentum refresh + Metropolis transition (transitions.py:129-142, 256-352)."""
    from golden_util import load_hmc_case

    problem, n_iter, n_step, seed, g = load_hmc_case(name)
    o = dr.oracle_hmc(problem, n_iter, n_step, seed)
    np.testing.assert_allclose(o["pos"], g["pos"], rtol=1e-12, atol=1e-14)
    np.testing.assert_array_equal(o["dir"], g["dir"])
    np.testing.assert_array_equal(o["n_step"], g["n_step"])
    np.testing.assert_allclose(o["metrop_accept_prob"], g["metrop_accept_prob"], rtol=1e-11)
    assert 0.0 < o["accepted"].mean() <= 1.0


ADAPT_NAMES = ["adapt_c1_dualavg_variance", "adapt_c1_dualavg_covariance", "adapt_c0_dualavg_min",
               "adapt_c0_variance_first", "adapt_c3_torus_dualavg", "adapt_c2_softabs_d6_dualavg",
               "adapt_nuts_c0_dualavg", "adapt_nuts_c1_dualavg_variance"]
NUTS_NAMES = ["nuts_c1_multinomial_d10", "nuts_c1_slice_euclidean_d16",
              "nuts_c0_depth4_no_extra_checks", "nuts_c1_diag_divergent", "nuts_c1_identity_d70",
              "nuts_c3_torus_constrained", "nuts_c2_softabs_d4_implicit"]


@pytest.mark.parametrize("name", ADAPT_NAMES)
def test_oracle_adaptive_sampling_matches_reference_fixture(name):
    """Row N3: dual averaging / online variance / online covariance adapters and the windowed
    stager, against the reference's own ``sample_chains`` (adapters.py, stagers.py)."""
    import warnings

    from golden_util import load_adapt_case

    problem, specs, _, _, _, n_step, seed, stages, g = load_adapt_case(name)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = dr.oracle_sample_chains(problem, stages, n_step, seed, specs,
                                    dynamic=n_step if isinstance(n_step, dict) else None)
    for k in ("pos", "accept_stat", "n_step", "final_pos", "final_mom", "step_size", "metric"):
        np.testing.assert_allclose(o[k], g[k], rtol=1e-12, atol=1e-14, err_msg=k)
    np.testing.assert_array_equal(o["final_dir"], g["final_dir"])


@pytest.mark.parametrize("name", NUTS_NAMES)
def test_oracle_dynamic_transition_matches_reference_fixture(name):
    """Row N4: the iterative restatement of ``DynamicIntegrationTransition`` (multinomial and
    slice variants, both no-U-turn criteria, divergences) against the reference's recursion
    (transitions.py:487-858) -- positions, statistics and the returned ``dir``."""
    import warnings

    from golden_util import load_nuts_case

    problem, n_iter, seed, opts, g = load_nuts_case(name)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = dr.oracle_nuts(problem, n_iter, seed, **opts)
    np.testing.assert_allclose(o["pos"], g["pos"], rtol=1e-12, atol=1e-14)
    for k in ("n_step", "tree_depth", "diverging", "dir"):
        np.testing.assert_array_equal(o[k], g[k], err_msg=k)
    for k in ("av_metrop_accept_prob", "accept_stat", "reject_prob"):
        np.testing.assert_allclose(o[k], g[k], rtol=1e-12, atol=1e-15, err_msg=k)
