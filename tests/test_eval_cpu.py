"""Policy evaluation without a GPU: eval_es.py's command line, config and checkpoint handling as far as they go without a
device, RolloutEngine.evaluate's argument checks, and B200Loop's engine.eval_every / engine.eval_episodes keys on a stand-in
strategy."""
import os
import sys

import numpy as np
import pytest
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import eval_es  # noqa: E402
from simple_es_b200 import checkpoint  # noqa: E402
from simple_es_b200 import loop as loop_mod  # noqa: E402
from simple_es_b200.engine import RolloutEngine  # noqa: E402


def _conf(name):
    with open(os.path.join(ROOT, "conf", name)) as fh:
        return yaml.load(fh, Loader=yaml.FullLoader)


def test_eval_es_arguments():
    a = eval_es.parse_args(["--cfg-path", "c.yaml", "--ckpt-path", "a.pt", "b.pt"])
    assert a.ckpt_path == ["a.pt", "b.pt"] and a.episodes == 100 and a.seed == 0 and a.round == 0 and a.out is None
    a = eval_es.parse_args(["--cfg-path", "c.yaml", "--ckpt-path", "a.pt", "--episodes", "7", "--seed", "3", "--round", "2",
                            "--out", "r.npz"])
    assert (a.episodes, a.seed, a.round, a.out) == (7, 3, 2, "r.npz")
    for bad in (["--ckpt-path", "a.pt"], ["--cfg-path", "c.yaml"], ["--cfg-path", "c.yaml", "--ckpt-path", "a.pt", "--episodes", "0"],
                ["--cfg-path", "c.yaml", "--ckpt-path", "a.pt", "--round", "-1"]):
        with pytest.raises(SystemExit):
            eval_es.parse_args(bad)


def test_eval_es_engine_config():
    kw = eval_es.engine_config(_conf("cartpole.yaml"))
    assert kw == dict(env_name="CartPole-v1", obs_dim=4, act_dim=2, gru=False, pomdp=False, max_step=500, n_agents=2,
                      discrete_action=True)
    kw = eval_es.engine_config(_conf("simplespread.yaml"))
    assert kw["env_name"] == "simple_spread" and kw["obs_dim"] == 12 and kw["max_step"] == "None" and kw["n_agents"] == 2
    kw = eval_es.engine_config(_conf("pendulum.yaml"))
    assert kw["discrete_action"] is False
    cfg = _conf("cartpole.yaml")
    cfg["network"]["name"] = "other"
    with pytest.raises(ValueError, match="gym_model"):
        eval_es.engine_config(cfg)


def test_eval_es_loads_checkpoints_in_order(tmp_path):
    flats = [torch.randn(6562) for _ in range(2)]
    paths = []
    for i, f in enumerate(flats):
        p = tmp_path / ("ep_%d.pt" % i)
        torch.save(checkpoint.flat_to_state_dict(f, 4, 2, True), p)
        paths.append(str(p))
    W = eval_es.load_policies(paths, 4, 2, True)
    assert W.shape == (2, 6562) and W.dtype == torch.float32
    assert torch.equal(W[0], flats[0]) and torch.equal(W[1], flats[1])
    with pytest.raises(ValueError, match="network needs"):
        eval_es.load_policies(paths, 4, 2, False)                  # a GRU checkpoint under an MLP config
    with pytest.raises(ValueError, match="shape"):
        eval_es.load_policies(paths, 6, 3, True)                   # another env's observation width


def _write(tmp_path, cfg, flat, obs, act, gru):
    c, p = tmp_path / "c.yaml", tmp_path / "ep_1.pt"
    c.write_text(yaml.safe_dump(cfg))
    torch.save(checkpoint.flat_to_state_dict(flat, obs, act, gru), p)
    return ["--cfg-path", str(c), "--ckpt-path", str(p)]


def test_eval_es_unsupported_env_fails_with_the_engine_error(tmp_path):
    cfg = _conf("cartpole.yaml")
    cfg["env"]["name"] = "LunarLander-v2"
    cfg["network"].update(num_state=8, num_action=4)
    with pytest.raises(ValueError, match="not supported by the B200 engine"):
        eval_es.main(_write(tmp_path, cfg, torch.zeros(8 * 32 + 32 + 4 * 32 + 4), 8, 4, False))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a device")
def test_eval_es_without_a_device_fails_loudly(tmp_path):
    with pytest.raises(RuntimeError, match="no CUDA device"):
        eval_es.main(_write(tmp_path, _conf("cartpole.yaml"), torch.zeros(226), 4, 2, False))


def test_engine_evaluate_checks_its_policies():
    eng = object.__new__(RolloutEngine)                            # argument checks run before any device work
    eng.D = 226
    with pytest.raises(ValueError, match=r"expected \[226\] or \[n_pol, 226\]"):
        eng.evaluate(torch.zeros(225), 10)
    with pytest.raises(ValueError, match=r"expected \[226\]"):
        eng.evaluate(torch.zeros(2, 3, 226), 10)
    with pytest.raises(ValueError, match=r"expected \[226\]"):
        eng.evaluate(np.zeros(226, np.float32), 10)
    with pytest.raises(ValueError, match="float32 CUDA tensor"):
        eng.evaluate(torch.zeros(3, 226), 10)


# ------------------------------------------------------------------------------------------------ B200Loop on a stand-in
class _Engine:
    def __init__(self):
        self.calls = []

    def evaluate(self, policies, n_episodes, round=0):
        self.calls.append((tuple(policies.shape), n_episodes, round))
        r = torch.arange(n_episodes, dtype=torch.float64)[None] + round
        return r, torch.full((1, n_episodes), 7, dtype=torch.int32)


class _Strategy:
    exchange = "local"

    def __init__(self, strat_cfg, env_cfg, net_cfg, eval_ep_num, seed, device, engine_cfg):
        self.engine = _Engine()
        self.curr_sigma = 0.5
        self.n = 0

    def step(self):
        self.n += 1

    def best_reward(self):
        return torch.tensor(float(self.n))

    def phase_times(self):
        return (0.25, 0.125)

    def elite_flat(self):
        return torch.zeros(226)


@pytest.fixture
def stand_in(monkeypatch):
    monkeypatch.setattr(loop_mod, "STRATEGIES", {"openai_es": _Strategy})
    monkeypatch.setattr(loop_mod.torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(loop_mod.sdist, "init_from_env", lambda: (0, 1))


def test_loop_without_eval_keys_is_unchanged(stand_in, capsys):
    loop = loop_mod.B200Loop(_conf("cartpole_openai.yaml"), 4, 1, 5, save_model_period=0)
    hist = loop.run()
    out = capsys.readouterr().out.splitlines()
    assert loop.eval_every == 0 and loop.eval_episodes == 100 and loop.strategy.engine.calls == [] and loop.eval_history == []
    assert len(out) == 4 and all(line.startswith("episode: ") for line in out)
    assert [h[:3] for h in hist] == [(i, float(i), 0.5) for i in range(1, 5)]


def test_loop_eval_keys(stand_in, capsys):
    cfg = _conf("cartpole_openai.yaml")
    cfg["engine"].update(eval_every=2, eval_episodes=10)
    loop = loop_mod.B200Loop(cfg, 5, 1, 5, save_model_period=0)
    loop.run()
    out = capsys.readouterr().out.splitlines()
    assert loop.strategy.engine.calls == [((226,), 10, 2), ((226,), 10, 4)]            # keyed by the generation number
    assert [e[:7] for e in loop.eval_history] == [(2, 10, 6.5, float(np.std(np.arange(10))), 2.0, 11.0, 7.0),
                                                   (4, 10, 8.5, float(np.std(np.arange(10))), 4.0, 13.0, 7.0)]
    assert len(out) == 7 and out[2].startswith("  eval: 10 episodes, mean 6.50, std 2.87, min 2.00, max 11.00, mean length 7.0")
    assert out[1].startswith("episode: 2,") and out[3].startswith("episode: 3,")
    cfg["engine"].update(eval_episodes=0)
    with pytest.raises(ValueError, match="eval_episodes"):
        loop_mod.B200Loop(cfg, 1, 1, 5, save_model_period=0)
