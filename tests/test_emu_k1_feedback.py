"""K1's mean-length feedback on the SIMT emulator: the launcher gives a launch a queue B (exact requests for the last two
rounds' worth of episodes) unless the PREVIOUS launch's mean episode length says the episodes are ragged.  A stale mean
therefore hands a launch the other regime's geometry; DESIGN 5.1 promises that this only changes the geometry.  The
sequence below drives both stale decisions (a generation-0 launch after a converged one gets a tail, a converged launch
after a generation-0 one gets none) and demands the twin's bits from every launch.  tests/test_gpu_k1_full_size.py runs
the same sequence on the B200 at P = 65536."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

D = 226
E = 5
SMS, CTAS = 2, 2                  # 2 emulated SMs x 2 CTAs x 4 warps: a round is R = 16 x 32 = 512 episodes
MAX_STEP = 100                    # a generation-0 mean (~17 steps) is "ragged" below 0.25 * MAX_STEP, a converged one is not
P = 300                           # 1500 episodes: queue A + B when the launch gets a tail (tail_start = 475), all queue A when not


def _state():
    import bench
    return bench.bench_state()


def _tail_start(n_ep, resident_warps, tail):
    """ses_abi.cu launch_slots: the first episode of queue B."""
    R = resident_warps * 32
    if n_ep <= R:
        return 0
    t = 2 * R if tail else 0
    return (n_ep - t) // E * E if n_ep > t else 0


@pytest.fixture(scope="module")
def emu():
    from simt_emu import emu_engine
    emu_engine.load()
    return emu_engine.EmuEngine


@pytest.fixture(scope="module")
def populations(twin):
    """(label, generation, sigma, mu, twin fitness, twin steps) of the two regimes, each rolled out once by the twin."""
    st = _state()
    zero = np.zeros((1, D), np.float32)
    out = {}
    for label, gen, sigma, mu in [("converged", 30, st["sigma"], st["mu"][None]), ("gen0", 0, 0.2, zero)]:
        tf, ts = twin.population_cartpole(mu, sigma=sigma, seed=0, gen=gen, group=P, n_head=1, n=P, E=E, max_step=MAX_STEP,
                                          nthreads=os.cpu_count())
        out[label] = (gen, sigma, mu, tf, ts)
    assert out["converged"][4].mean() / E >= 0.25 * MAX_STEP           # the regimes are the ones the launcher tells apart
    assert out["gen0"][4].mean() / E < 0.25 * MAX_STEP
    return out


# (population, whether the launch gets a tail): the first launch knows no mean and assumes long episodes; afterwards each
# launch's decision is read off the launch before it
SEQUENCE = [("converged", True), ("converged", True), ("gen0", True), ("gen0", False), ("converged", False), ("converged", True)]


def _run_sequence(eng, populations, fresh_outputs):
    for i, (label, tail) in enumerate(SEQUENCE):
        gen, sigma, mu, tf, ts = populations[label]
        fit, steps = eng.rollout(gen, sigma, mu, **fresh_outputs())
        g = eng.test_k1_geometry()
        assert g["resident_warps"] == SMS * CTAS * 4 and g["lanes"] == 32 and g["sparse_rank"] < 0, (i, g)
        assert g["tail_start"] == _tail_start(P * E, g["resident_warps"], tail), (i, label, g)
        assert np.array_equal(steps, ts), (i, label)
        assert np.array_equal(fit, tf), (i, label)


def test_emu_k1_feedback_regime_changes(emu, populations, monkeypatch):
    """converged, converged, generation 0 (stale "long": tail), generation 0, converged (stale "ragged": no tail),
    converged: every launch equals the twin, and the geometry hook shows the stale decisions were taken."""
    monkeypatch.setenv("SES_SIMT_EMU_SMS", str(SMS))
    monkeypatch.setenv("SES_SIMT_EMU_CTAS_PER_SM", str(CTAS))
    eng = emu(population=P, group=P, n_head=1, eval_ep_num=E, seed=0, max_step=MAX_STEP)
    _run_sequence(eng, populations, lambda: {})
    eng.close()


def test_emu_k1_feedback_reused_output_buffers(emu, populations, monkeypatch):
    """The same sequence writing into ONE fitness / steps pair poisoned before each launch: every offspring is written by
    every launch, whichever queue and warp its episodes ran in (an offspring split across warps is published once, by the
    part that completes it)."""
    monkeypatch.setenv("SES_SIMT_EMU_SMS", str(SMS))
    monkeypatch.setenv("SES_SIMT_EMU_CTAS_PER_SM", str(CTAS))
    eng = emu(population=P, group=P, n_head=1, eval_ep_num=E, seed=0, max_step=MAX_STEP)
    fit = np.empty(P); steps = np.empty(P, dtype=np.int64)

    def poisoned():
        fit.fill(np.nan); steps.fill(-1)
        return {"fitness": fit, "steps": steps}
    _run_sequence(eng, populations, poisoned)
    eng.close()


@pytest.mark.parametrize("tail_env", ["0", "2"])
def test_emu_k1_forced_tail_ignores_feedback(emu, populations, tail_env, monkeypatch):
    """SES_K1_TAIL overrides the feedback (0: queue A only, 2: two rounds of queue B) in either regime: the geometry follows
    the knob and the bits stay the twin's."""
    monkeypatch.setenv("SES_SIMT_EMU_SMS", str(SMS))
    monkeypatch.setenv("SES_SIMT_EMU_CTAS_PER_SM", str(CTAS))
    monkeypatch.setenv("SES_K1_TAIL", tail_env)
    eng = emu(population=P, group=P, n_head=1, eval_ep_num=E, seed=0, max_step=MAX_STEP)
    for label in ("gen0", "converged", "gen0"):
        gen, sigma, mu, tf, ts = populations[label]
        fit, steps = eng.rollout(gen, sigma, mu)
        g = eng.test_k1_geometry()
        assert g["tail_start"] == _tail_start(P * E, g["resident_warps"], tail_env == "2"), (label, g)
        assert np.array_equal(steps, ts) and np.array_equal(fit, tf), label
    eng.close()
