"""sep_cma_es host logic without a GPU (DESIGN.md section 4.11): the constants against Hansen's formulas, the exact fma the
numpy restatement relies on, config validation, the refused antithetic mode and a resume state of another run."""
import math
import os
import sys
from fractions import Fraction

import numpy as np
import pytest
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cma_reference as cref  # noqa: E402

from simple_es_b200.engine import population_layout, sep_cma_constants, sep_cma_threshold  # noqa: E402
from simple_es_b200.strategies import STRATEGIES, SepCMAES  # noqa: E402


@pytest.mark.parametrize("D,lam,mu", [(226, 65536, 32768), (6562, 4097, 2048), (195, 2085, 1), (581, 2085, 2085), (2, 2, 1)])
def test_constants_follow_the_formulas(D, lam, mu):
    k = sep_cma_constants(D, lam, mu)
    w = np.array([math.log(mu + 0.5) - math.log(i) for i in range(1, mu + 1)])
    w = w / w.sum()
    assert np.allclose(k["weights"], w, rtol=1e-14, atol=0) and abs(k["weights"].sum() - 1.0) < 1e-12
    assert np.all(np.diff(k["weights"]) <= 0) and np.all(k["weights"] > 0)
    me = 1.0 / np.sum(w ** 2)
    cs = (me + 2) / (D + me + 5)
    ds = 1 + 2 * max(0.0, math.sqrt((me - 1) / (D + 1)) - 1) + cs
    cc = (4 + me / D) / (D + 4 + 2 * me / D)
    c1 = 2 / ((D + 1.3) ** 2 + me)
    cmu = min(1 - c1, 2 * (me - 2 + 1 / me) / ((D + 2) ** 2 + me))
    c1 *= (D + 2) / 3
    cmu = min(1 - c1, cmu * (D + 2) / 3)
    chi = math.sqrt(D) * (1 - 1 / (4 * D) + 1 / (21 * D * D))
    for name, want in (("mu_eff", me), ("c_sigma", cs), ("d_sigma", ds), ("c_c", cc), ("c1", c1), ("cmu", cmu), ("chi", chi)):
        assert k[name] == pytest.approx(want, rel=1e-12, abs=0), name
    assert k["one_m_cs"] == 1 - k["c_sigma"] and k["one_m_cc"] == 1 - k["c_c"] and k["damp"] == k["c_sigma"] / k["d_sigma"]
    assert k["k_sigma"] == math.sqrt(k["c_sigma"] * (2 - k["c_sigma"]) * k["mu_eff"])
    assert k["k_c"] == math.sqrt(k["c_c"] * (2 - k["c_c"]) * k["mu_eff"]) and k["cc2"] == k["c_c"] * (2 - k["c_c"])
    assert k["c_keep"] == 1 - k["c1"] - k["cmu"] and k["c_keep"] >= 0
    for g in (0, 1, 10, 1000):
        t = (1.4 + 2 / (D + 1)) * chi * math.sqrt(1 - (1 - cs) ** (2 * (g + 1)))
        assert sep_cma_threshold(k, g) == pytest.approx(t, rel=1e-12)


def test_layout_samples_every_offspring():
    assert population_layout("sep_cma_es", 4097, 2048) == (4097, 4097, 0, 1)
    with pytest.raises(ValueError, match="elite_num"):
        sep_cma_constants(10, 8, 9)


def test_fma_emulation_is_exact():
    """cma_reference.fma == the correctly rounded a * b + c (Fractions), on float32 noise and its squares against float64
    weights and sums, with cancellations and products whose tails sit near a rounding tie."""
    rng = np.random.default_rng(0)
    n = 4000
    z = rng.standard_normal(n).astype(np.float32).astype(np.float64)
    w = rng.uniform(0, 1, n) * 2.0 ** rng.integers(-20, 2, n)
    c = rng.standard_normal(n) * 2.0 ** rng.integers(-30, 10, n)
    a = np.concatenate([z, z * z, z, z])
    b = np.concatenate([w, w, w, w])
    c = np.concatenate([c, c, -(z * w), -(z * w) + np.ldexp(np.sign(z), -60)])       # exact cancellation, near-cancellation
    got = cref.fma(a, b, c)
    for i in range(a.size):
        want = float(Fraction(a[i]) * Fraction(b[i]) + Fraction(c[i]))
        assert got[i] == want or (got[i] == 0 and want == 0), (i, a[i], b[i], c[i])


def _strategy_cfg(**over):
    cfg = yaml.load(open(os.path.join(ROOT, "conf", "cartpole_sep_cma.yaml")), Loader=yaml.FullLoader)
    cfg["strategy"].update(over)
    return cfg


@pytest.mark.parametrize("over,match", [
    ({"sigma_decay": 0.99}, "unknown key"), ({"learning_rate": 0.1}, "unknown key"), ({"init_sigma": 0.0}, "init_sigma"),
    ({"init_sigma": -1.0}, "init_sigma"), ({"init_sigma": "big"}, "init_sigma"), ({"init_sigma": float("inf")}, "init_sigma"),
    ({"offspring_num": 1}, "offspring_num"), ({"offspring_num": 10.0}, "offspring_num"), ({"elite_num": 0}, "elite_num"),
    ({"elite_num": 4097}, "elite_num"), ({"elite_num": True}, "elite_num")])
def test_config_errors(over, match):
    cfg = _strategy_cfg(**over)
    with pytest.raises(ValueError, match=match):
        SepCMAES(cfg["strategy"], cfg["env"], cfg["network"], 5, 0, 0, dict(cfg["engine"]))


def test_antithetic_is_refused():
    cfg = _strategy_cfg()
    with pytest.raises(ValueError, match="antithetic"):
        SepCMAES(cfg["strategy"], cfg["env"], cfg["network"], 5, 0, 0, dict(cfg["engine"], antithetic=True))


def test_registered():
    assert STRATEGIES["sep_cma_es"] is SepCMAES


def test_load_state_refuses_another_run():
    """A resume state is refused when the run key differs (here elite_num), before anything is loaded."""
    s = SepCMAES.__new__(SepCMAES)
    s.parents, s.P = torch.zeros(1, 226), 4096
    s._run_key = {"env": "CartPole-v1", "seed": 0, "elite_num": 2048}
    st = {"strategy": "sep_cma_es", "parents": torch.ones(1, 226), "population": 4096, "generation": 7,
          "run_key": {"env": "CartPole-v1", "seed": 0, "elite_num": 100}}
    with pytest.raises(ValueError, match="elite_num was 100, now 2048"):
        s.load_state(st)
    assert torch.all(s.parents == 0)
    with pytest.raises(ValueError, match="strategy"):
        s.load_state(dict(st, strategy="openai_es"))
