"""CPU: the oracle against the reference's UNMODIFIED host code, live
(FakeEnv / ModelSampler / ModelBuffer / CPOBuffer / statics / average_dkl / discount_cumsum imported
through oracle/ref_stubs.py from the reference source tree, CMBPO_REFERENCE_ROOT).  The tests that import it
are skipped where that tree is absent."""
import numpy as np
import pytest

from oracle import cmbpo_oracle as orc, ref_stubs

needs_reference = pytest.mark.skipif(not ref_stubs.reference_available(), reason="reference source tree not present")
GAE = dict(gamma=0.99, lam=0.95, cgamma=0.97, clam=0.5)
TASKS = [("HalfCheetahSafe-v2", 17, 6), ("AntSafe-v2", 29, 8), ("HumanoidSafe-v2", 47, 17)]


@needs_reference
@pytest.mark.parametrize("task,O,A", TASKS)
@pytest.mark.parametrize("mode", [False, "uncertainty"])
def test_full_cycle_bit_exact(task, O, A, mode):
    from oracle import ref_harness
    dyn, actor, v, vc = orc.make_problem(1, O, A, hidden=(48, 48), vf_hidden=(32, 32), a_hidden=(32, 32), task=task)
    obs, act = orc.make_states(2, 96, O, A, dyn)
    T = 12
    noise = orc.TableNoise(3, T, 96, A, len(dyn.elite_inds))
    lim = None
    if mode:
        env = orc.OracleFakeEnv(O, A, task, orc.OracleModel(dyn), lambda e, n: np.zeros(n, int))
        lim = float(np.median(env.step(obs, act)[3]["ensemble_dkl_path"]) * 4)
    with np.errstate(all="ignore"):
        r = ref_harness.reference_rollout(dyn, actor, v, vc, task, obs, noise, T, mode, lim,
                                          max_samples=700, stop_alive_ratio=0.1, **GAE)
        o = orc.run_rollout(dyn, actor, v, vc, task, obs, noise, T, mode, lim, max_samples=700,
                            stop_alive_ratio=0.1, **GAE)
    assert all(np.array_equal(x, y) and x.dtype == y.dtype for x, y in zip(r[0], o[0]))
    assert all(np.array_equal(r[3][k], o[3][k]) for k in r[3])
    assert r[1] == o[1]
    for k in o[2]:
        assert np.isclose(float(r[2][k]), float(o[2][k]), rtol=1e-12, equal_nan=True), k


def test_choice_equals_randint_positions():
    """np.random.choice(elite_inds, n) (fake_env.py:176) consumes the global stream exactly like
    elite_inds[np.random.randint(0, len, n)] -- what cmbpo_b200.FakeEnv.random_inds relies on."""
    elite = [4, 0, 6, 2, 2]
    np.random.seed(123)
    a = np.random.choice(elite, 1000)
    np.random.seed(123)
    b = np.asarray(elite)[np.random.randint(0, len(elite), 1000)]
    assert np.array_equal(a, b)


@needs_reference
def test_mpi_statistics_scalar():
    ref = ref_stubs.load()
    x = np.random.default_rng(0).standard_normal(5001).astype(np.float32) * 3 + 1
    assert ref.mpi_statistics_scalar(x) == orc.stats_scalar(x)


@needs_reference
def test_boltz_dist_and_policy_kl_formula_live():
    """Oracle boltz_dist / epochs_list against the reference's CPOBuffer methods on a fresh case."""
    from oracle import gen_golden
    ref = ref_stubs.load()
    ep, kls = gen_golden.make_archive_case(77, n_rows=1234, archive_size=1500, n_ep=5)
    buf = ref.CPOBuffer(10, len(ep), ref_stubs.Space(3), ref_stubs.Space(2))
    buf.epoch_archive[:] = ep
    assert np.array_equal(orc.epochs_list(ep), buf.epochs_list)
    for alpha in (0.5, 1, 3):
        a, b = orc.boltz_dist(ep, kls, alpha), buf.boltz_dist(kls, alpha=alpha)
        assert a.dtype == b.dtype and np.array_equal(a, b)
