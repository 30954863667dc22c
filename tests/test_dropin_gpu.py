"""Drop-in proof (VERDICT r1 X2): a ``mici_b200`` system + integrator, driven one NumPy-held chain
state at a time through the calls the reference's sampler / transition layer makes, reproduces
the chains the stock reference sampler produced over the reference's own system and integrator
(``tests/golden/dropin_*.npz``, ``oracle/make_golden.py``).  The sampler layer here is the
oracle's port of the reference transitions (``mo.static_hmc_transition`` / ``mo.nuts_transition``,
themselves pinned to the reference by tests/test_oracle.py), with the reference's per-chain
generators ``default_rng(rng.bit_generator.jumped(i))`` (samplers.py:559-560).

What the reference layer touches on the replaced objects (reference file:line):
``integrator.step(state)`` transitions.py:291, 657; ``system.h(state)`` transitions.py:281, 301;
``system.sample_momentum(state, rng)`` transitions.py:141; ``system.dh_dmom(state)``
transitions.py:434-435, 472-473 (dynamic criteria); ``state.copy()`` / ``state.dir`` flips.
"""

import os

import numpy as np
import pytest

from mici_b200 import engine, errors, problems
from oracle import mici_oracle as mo
from oracle.make_golden import DROPIN_CASES, DROPIN_SEED, DROPIN_STATS, GOLDEN_DIR, input_checksum

pytestmark = pytest.mark.gpu


class NumpyChainState:
    """A foreign chain state with the reference ``ChainState``'s storage (states.py:160-305):
    NumPy vectors, ``dir`` an int, ``copy()`` and the ``in`` test."""

    def __init__(self, pos, mom, dir):  # noqa: A002
        self.pos, self.mom, self.dir = pos, mom, dir

    def __contains__(self, name):
        return name in self.__dict__

    def copy(self):
        return NumpyChainState(self.pos.copy(), None if self.mom is None else self.mom.copy(),
                               self.dir)


def _run_sampler_port(system, integrator, problem, sampler_name, n_iter, seed, **kw):
    """``sample_chains(0, n_iter, ...)`` of the reference's ``StaticMetropolisHMC`` /
    ``DynamicMultinomialHMC`` (one worker, no adapters) over ``system`` / ``integrator``."""

    def step(q, p, d):
        try:
            new = integrator.step(NumpyChainState(q, p, d))
        except errors.ConvergenceError as e:
            raise mo.OracleIntegratorError(mo.STATUS_CONVERGENCE) from e
        except errors.NonReversibleStepError as e:
            raise mo.OracleIntegratorError(mo.STATUS_NON_REVERSIBLE) from e
        assert isinstance(new, NumpyChainState) and isinstance(new.pos, np.ndarray)
        return new.pos, new.mom

    def h(q, p):
        return float(system.h(NumpyChainState(q, p, 1)))

    def velocity(q, p):
        return np.asarray(system.dh_dmom(NumpyChainState(q, p, 1)))

    def sample_momentum(q, rng):
        return np.asarray(system.sample_momentum(NumpyChainState(q, None, 1), rng))

    base = np.random.default_rng(seed)
    # chains given without momentum get one drawn from the base generator first
    # (samplers.py:1259-1260); the first momentum transition replaces it
    for i in range(problem.n_chains):
        sample_momentum(problem.pos[i], base)
    final, traces, stats = [], [], {k: [] for k in DROPIN_STATS}
    for i in range(problem.n_chains):
        rng = np.random.default_rng(base.bit_generator.jumped(i))
        q, d = problem.pos[i].copy(), 1
        trace, chain_stats = [], {k: [] for k in DROPIN_STATS}
        for _ in range(n_iter):
            if sampler_name == "StaticMetropolisHMC":
                q, _, d, st = mo.static_hmc_transition(q, None, d, rng, step, h, sample_momentum,
                                                       kw["n_step"])
            else:
                p = sample_momentum(q, rng)
                q, _, st = mo.nuts_transition(q, p, rng.uniform, step, h, velocity,
                                              max_tree_depth=kw["max_tree_depth"])
            trace.append(q)
            for k in DROPIN_STATS:
                chain_stats[k].append(st[k])
        final.append(q)
        traces.append(trace)
        for k in DROPIN_STATS:
            stats[k].append(chain_stats[k])
    return np.stack(final), np.asarray(traces), {k: np.asarray(v) for k, v in stats.items()}


@pytest.mark.parametrize("name", sorted(DROPIN_CASES))
def test_mici_b200_integrator_reproduces_stock_sampler_chains(name):
    cfg, kwargs, sampler_name, n_iter, skw = DROPIN_CASES[name]
    problem = problems.make_problem(cfg, **kwargs)
    g = dict(np.load(os.path.join(GOLDEN_DIR, f"dropin_{name}.npz")))
    np.testing.assert_allclose(input_checksum(problem), g["input_checksum"], rtol=1e-13)

    integrator = engine.build_integrator(problem)
    new_final, new_trace, new_stats = _run_sampler_port(
        integrator.system, integrator, problem, sampler_name, n_iter, DROPIN_SEED, **skw)

    np.testing.assert_array_equal(new_stats["n_step"], g["n_step"])
    np.testing.assert_array_equal(new_stats["convergence_error"], g["convergence_error"])
    np.testing.assert_array_equal(new_stats["non_reversible_step"], g["non_reversible_step"])
    np.testing.assert_allclose(new_stats["accept_stat"], g["accept_stat"], rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(new_trace, g["trace_pos"], rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(new_final, g["final_pos"], rtol=1e-8, atol=1e-10)


def test_integrator_step_raises_reference_compatible_errors():
    """``integrator.step`` on a single NumPy chain raises ``ConvergenceError`` /
    ``NonReversibleStepError``, subclasses of the ``IntegratorError`` that the reference's
    ``except IntegratorError`` clauses catch (transitions.py:292, 670)."""
    problem = problems.make_problem("C3", n_chains=16)
    problem.step_size = 0.6
    integrator = engine.build_integrator(problem)
    raised = 0
    for i in range(problem.n_chains):
        state = NumpyChainState(problem.pos[i].copy(), problem.mom[i].copy(), 1)
        try:
            for _ in range(3):
                state = integrator.step(state)
        except Exception as e:  # noqa: BLE001
            raised += 1
            assert type(e).__name__ in ("ConvergenceError", "NonReversibleStepError"), repr(e)
            assert isinstance(e, errors.IntegratorError), repr(e)
    assert raised > 0
