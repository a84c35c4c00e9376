"""map_elites (DESIGN.md section 4.12) without a GPU: config refusals, the layout, the cell map of
tests/map_elites_reference.py against exact rationals, resume-key refusal, archive files and eval_es.py --archive."""
import os
import sys
from fractions import Fraction

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import map_elites_reference as mref  # noqa: E402
from simple_es_b200 import checkpoint  # noqa: E402
from simple_es_b200.engine import population_layout  # noqa: E402
from simple_es_b200.strategies import STRATEGIES, MapElites, _Base, _map_params  # noqa: E402

BASE = {"name": "map_elites", "init_sigma": 0.5, "sigma_decay": 0.999, "offspring_num": 1024, "behavior_dims": [0, 1],
        "behavior_low": [-1.2, -0.07], "behavior_high": [0.6, 0.07], "behavior_cells": [32, 32]}
ENV = {"name": "MountainCar-v0", "max_step": 200}
NET = {"name": "gym_model", "num_state": 2, "num_action": 3, "discrete_action": True, "gru": False}


def test_map_elites_is_registered_with_one_parent_row_per_offspring():
    assert STRATEGIES["map_elites"] is MapElites
    for n in (2, 1024, 4097, 65536):
        assert population_layout("map_elites", n) == (n, 1, 0, n)


def test_map_params_accepts_the_shipped_configs():
    import yaml
    for conf, sd, D in (("mountaincar_map_elites.yaml", 2, 195), ("cartpole_map_elites.yaml", 4, 226)):
        cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
        n, dims, low, high, cells = _map_params(cfg["strategy"], sd, D)
        assert n == cfg["strategy"]["offspring_num"] and len(dims) == 2 and cells == [32, 32]


@pytest.mark.parametrize("patch,msg", [
    ({"learning_rate": 0.1}, "unknown key"),
    ({"elite_num": 4}, "unknown key"),
    ({"behavior_dims": None}, "behavior_dims must be a list"),
    ({"behavior_dims": [0, 2]}, r"indices into the final state \[0, 2\)"),
    ({"behavior_dims": [-1, 1]}, "indices into the final state"),
    ({"behavior_dims": [0, 0]}, "distinct"),
    ({"behavior_dims": [0.0, 1]}, "indices into the final state"),
    ({"behavior_dims": [0, 1, 0, 1, 0]}, "1 to 4"),
    ({"behavior_dims": [0]}, "one entry per"),
    ({"behavior_low": [0.6, -0.07]}, "below behavior_high"),
    ({"behavior_low": [0.7, -0.07]}, "below behavior_high"),
    ({"behavior_low": [float("-inf"), -0.07]}, "finite"),
    ({"behavior_high": [0.6, float("nan")]}, "finite"),
    ({"behavior_high": [0.6, True]}, "finite"),
    ({"behavior_cells": [0, 32]}, "integers >= 1"),
    ({"behavior_cells": [32, 2.0]}, "integers >= 1"),
    ({"behavior_cells": [1025, 1024]}, "1049600 cells exceed 2\\^20"),
    ({"offspring_num": 1}, "offspring_num"),
    ({"init_sigma": float("inf")}, "init_sigma"),
])
def test_map_params_refusals(patch, msg):
    with pytest.raises(ValueError, match=msg):
        _map_params(dict(BASE, **patch), 2, 195)


def test_map_params_missing_key():
    cfg = dict(BASE)
    del cfg["behavior_cells"]
    with pytest.raises(ValueError, match="missing key.*behavior_cells"):
        _map_params(cfg, 2, 195)


def test_map_params_cell_caps():
    """2^20 cells are allowed; for the GRU policy (D = 6562) the 4 GiB weight cap allows 163 630 cells, not 163 631."""
    assert _map_params(dict(BASE, behavior_cells=[1024, 1024]), 2, 195)[4] == [1024, 1024]
    assert _map_params(dict(BASE, behavior_cells=[163630, 1]), 2, 6562)[4] == [163630, 1]
    with pytest.raises(ValueError, match=r"163631 cells x 6562 parameters x 4 bytes = 4294986488 bytes .* exceed 4 GiB"):
        _map_params(dict(BASE, behavior_cells=[163631, 1]), 2, 6562)


def test_map_elites_refuses_antithetic():
    with pytest.raises(ValueError, match="antithetic"):
        MapElites(BASE, ENV, NET, 3, 0, 0, {"antithetic": True})


def test_map_elites_refuses_a_bad_descriptor_before_touching_a_device():
    with pytest.raises(ValueError, match="final state"):
        MapElites(dict(BASE, behavior_dims=[0, 3]), ENV, NET, 3, 0, 0, {})
    with pytest.raises(ValueError, match="final state"):
        MapElites(dict(BASE, behavior_dims=[12, 1]), {"name": "simple_spread"}, dict(NET, num_state=18, num_action=5), 3, 0, 0,
                  {"n_agents": 3})


# ---------------------------------------------------------------------------------------------------- the cell map
def exact_cell(x, lo, hi, cells):
    """The cell of coordinate x under the contract, in exact rationals from the float64 operands the device rounds."""
    if np.isnan(x):
        return -1
    w = float(np.float64(hi) - np.float64(lo))
    if np.isinf(x):
        return 0 if x < 0 else cells - 1
    with np.errstate(over="ignore"):
        d = float(np.float64(x) - np.float64(lo))           # each step is one correctly rounded operation
        t = float(np.float64(d) / np.float64(w))
    with np.errstate(over="ignore"):
        s = float(np.float64(t) * np.float64(cells))
    if np.isinf(s):                                          # an overflowed quotient lands in the edge cell of its sign
        return 0 if s < 0 else cells - 1
    fs = Fraction(s)
    if fs < 1:
        return 0
    if fs >= cells - 1:
        return cells - 1
    return int(fs)


def test_exact_cell_helper_rounds_like_the_contract():
    """The rationals agree with the unrounded formula wherever rounding cannot move a value across an edge."""
    for x, want in ((-1.2, 0), (0.6, 31), (-0.3, 16), (0.0, 21)):
        assert exact_cell(x, -1.2, 0.6, 32) == want


@pytest.mark.parametrize("lo,hi,cells", [(-1.2, 0.6, 32), (-0.07, 0.07, 32), (0.0, 1.0, 10), (-2.4, 2.4, 7), (-1.0, 1.0, 1),
                                         (0.0, 3.0, 3), (-5e-324, 5e-324, 2)])
def test_cell_map_against_rationals(lo, hi, cells):
    w = np.float64(hi) - np.float64(lo)
    xs = [lo, hi, np.nextafter(lo, -np.inf), np.nextafter(lo, np.inf), np.nextafter(hi, -np.inf), np.nextafter(hi, np.inf),
          np.inf, -np.inf, np.nan, 5e-324, -5e-324, 0.0, -0.0, 1e308, -1e308]
    for k in range(cells + 1):                                  # exactly on the interior edges, and one ulp either side
        e = np.float64(lo) + np.float64(k) * (w / np.float64(cells))
        xs += [e, np.nextafter(e, -np.inf), np.nextafter(e, np.inf)]
    xs = np.array(xs, dtype=np.float64)
    spec = mref.Spec([0], [lo], [hi], [cells])
    with np.errstate(over="ignore", invalid="ignore"):
        got = mref.cell_index(xs[:, None], spec)
    want = [exact_cell(float(x), lo, hi, cells) for x in xs]
    assert got.tolist() == want
    assert got[0] == 0 and got[1] == cells - 1


def test_cell_map_row_major_over_dims_in_config_order():
    spec = mref.Spec([2, 0], [0, 0], [1, 1], [3, 5])
    b = np.array([[0.5, 9, 0.1, 9], [0.95, 9, 0.9, 9], [0.0, 9, 0.4, 9]])
    assert mref.cell_index(b, spec).tolist() == [0 * 5 + 2, 2 * 5 + 4, 1 * 5 + 0]


def test_stats_qd_order_and_ties():
    F = np.full(3000, np.nan)
    F[::3] = np.tile([1e16, 1.0, -1e16, 3.0, 0.1], 200)
    F[5], F[2000] = 2e16, 2e16
    n, best, bf, qd = mref.stats(F)
    assert n == 1002 and best == 5 and bf == 2e16
    assert mref.stats(np.full(7, np.nan))[:2] == (0, -1)


# ---------------------------------------------------------------------------------------------------- resume keys
def test_resume_key_refuses_another_descriptor():
    """_Base.load_state compares run keys; a map_elites key carries the descriptor spec."""
    s = _Base.__new__(_Base)
    s.name, s.P, s.D = "map_elites", 4, 3
    s.parents = torch.zeros(4, 3)
    s.total_env_steps = torch.zeros(1, dtype=torch.int64)
    s._run_key = {"env": "MountainCar-v0", "behavior_dims": [0, 1], "behavior_low": [-1.2, -0.07], "behavior_high": [0.6, 0.07],
                  "behavior_cells": [32, 32]}
    st = {"strategy": "map_elites", "parents": torch.zeros(4, 3), "population": 4, "generation": 5, "sigma": 0.5, "curr_sigma": 0.5,
          "run_key": dict(s._run_key, behavior_cells=[16, 16])}
    with pytest.raises(ValueError, match="behavior_cells was \\[16, 16\\], now \\[32, 32\\]"):
        s.load_state(st)


# ---------------------------------------------------------------------------------------------------- archive files
def fake_archive(n, obs=4, act=2, gru=False, seed=0):
    D = sum(int(np.prod(s)) for _, s in checkpoint.param_shapes(obs, act, gru))
    rng = np.random.default_rng(seed)
    cells = torch.from_numpy(np.sort(rng.choice(1024, n, replace=False))).to(torch.int64)
    return {"cells": cells, "coords": torch.stack([cells // 32, cells % 32], 1), "fitness": torch.from_numpy(rng.normal(0, 1, n)),
            "behavior": torch.zeros(n, 4, dtype=torch.float64), "weights": torch.from_numpy(rng.normal(0, 1, (n, D)).astype(np.float32)),
            "born_generation": torch.zeros(n, dtype=torch.int64), "born_id": torch.arange(n, dtype=torch.int64),
            "spec": {"behavior_dims": [0, 2], "behavior_low": [-2.4, -0.2095], "behavior_high": [2.4, 0.2095], "behavior_cells": [32, 32]},
            "env": {"name": "CartPole-v1"}, "network": {"num_state": obs, "num_action": act, "gru": gru}}


@pytest.mark.parametrize("gru", [False, True])
def test_archive_weights_round_trip_to_state_dicts(tmp_path, gru):
    import eval_es
    a = fake_archive(5, gru=gru)
    path = str(tmp_path / "archive_ep_10.pt")
    torch.save(a, path)
    W, cells = eval_es.load_archive(path, 4, 2, gru)
    assert torch.equal(cells, a["cells"]) and torch.equal(W, a["weights"])
    for row in W:
        sd = checkpoint.flat_to_state_dict(row, 4, 2, gru)
        assert [k for k, _ in checkpoint.param_shapes(4, 2, gru)] == list(sd)
        assert torch.equal(checkpoint.state_dict_to_flat(sd, 4, 2, gru), row)


def test_load_archive_refusals(tmp_path):
    import eval_es
    p = str(tmp_path / "a.pt")
    torch.save(fake_archive(3), p)
    with pytest.raises(ValueError, match="6562 parameters"):
        eval_es.load_archive(p, 4, 2, True)
    torch.save({"fc1.weight": torch.zeros(32, 4)}, p)
    with pytest.raises(ValueError, match="not a map_elites archive"):
        eval_es.load_archive(p, 4, 2, False)
    torch.save(fake_archive(0), p)
    with pytest.raises(ValueError, match="empty archive"):
        eval_es.load_archive(p, 4, 2, False)


def test_eval_es_archive_arguments():
    import eval_es
    a = eval_es.parse_args(["--cfg-path", "c.yaml", "--archive", "archive_ep_10.pt", "--out", "r.npz"])
    assert a.archive == "archive_ep_10.pt" and a.ckpt_path is None
    a = eval_es.parse_args(["--cfg-path", "c.yaml", "--ckpt-path", "ep_1.pt", "ep_2.pt"])
    assert a.archive is None and a.ckpt_path == ["ep_1.pt", "ep_2.pt"]
    for argv in (["--cfg-path", "c.yaml"],                                                     # neither
                 ["--cfg-path", "c.yaml", "--archive", "a.pt", "--ckpt-path", "ep_1.pt"],        # both
                 ["--cfg-path", "c.yaml", "--archive", "a.pt", "--out", "r.npz", "--record", "2"]):
        with pytest.raises(SystemExit):
            eval_es.parse_args(argv)
