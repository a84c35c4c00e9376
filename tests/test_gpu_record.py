"""Episode recording (ses_record, DESIGN.md section 4.9) through the product library on the B200: the twin's episodes and
traces for every env x {MLP, GRU}, the bit rule against RolloutEngine.evaluate at large sizes, and eval_es.py --record on a
checkpoint of a training run."""
import os
import subprocess
import sys

import numpy as np
import pytest
import yaml

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import eval_reference as ref  # noqa: E402
import record_reference  # noqa: E402
from test_emu_record import chunk, same_bits  # noqa: E402
from test_gpu_evaluate import _cfg, _ids, engine, policies  # noqa: E402

CONFIGS = [("CartPole-v1", False, False, 1), ("CartPole-v1", False, True, 1), ("CartPole-v0", False, False, 1),
           ("CartPole-v1", True, True, 1), ("CartPole-v1", True, False, 1),
           ("MountainCar-v0", False, False, 1), ("MountainCar-v0", True, False, 1),
           ("Acrobot-v1", False, False, 1), ("Acrobot-v1", True, False, 1),
           ("Pendulum-v0", False, False, 1), ("Pendulum-v0", True, False, 1),
           ("simple_spread", False, False, 2), ("simple_spread", True, False, 2),
           ("simple_spread", False, False, 3), ("simple_spread", True, False, 3)]


def numpy(tensors):
    return [t.cpu().numpy() for t in tensors]


@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_gpu_record_equals_twin(twin, cfg):
    """Two chunks and a partial third, every array bit for bit (NaN / -1 past each episode's end); the last return of each
    episode is evaluate's."""
    env, gru, pomdp, N = cfg
    eng = engine(env, gru, pomdp, N)
    W = policies(eng, 2, 3)                          # CartPole MLP: a policy that balances for 500 steps next to a random one
    K = 2 * chunk(env, gru, N) + 3
    got = numpy(eng.record(torch.from_numpy(W).cuda(), K, round=4))
    if env == "Pendulum-v0":
        assert got[2].dtype == np.float32
    want = record_reference.record(twin, env, W, K, seed=11, rnd=4, gru=gru, pomdp=pomdp, n_agents=N)
    for name, g, w in zip(("initial", "states", "actions", "returns", "lengths"), got, want):
        assert same_bits(g, w), name
    ret, lng = numpy(eng.evaluate(torch.from_numpy(W).cuda(), K + 40, round=4))
    last = np.take_along_axis(got[3], (got[4] - 1)[..., None].astype(np.int64), axis=2)[..., 0]
    assert np.array_equal(got[4], lng[:, :K]) and same_bits(last, ret[:, :K])


@pytest.mark.parametrize("env,gru,n_pol,K", [("CartPole-v1", False, 4, 4096), ("MountainCar-v0", True, 2, 1024)])
def test_gpu_record_bit_rule_at_scale(twin, env, gru, n_pol, K):
    """K episodes x n_pol policies against evaluate's first K of more episodes; NaN / -1 exactly past each end; a sample of
    episodes against the twin with their initial states given."""
    eng = engine(env, gru)
    W = policies(eng, n_pol, 5)
    Wd = torch.from_numpy(W).cuda()
    initial, states, actions, returns, lengths = eng.record(Wd, K, round=3)
    ret, lng = eng.evaluate(Wd, K + 777, round=3)
    assert torch.equal(lengths, lng[:, :K])
    last = returns.gather(2, (lengths.long() - 1).unsqueeze(-1)).squeeze(-1)
    assert torch.equal(last.view(torch.int64), ret[:, :K].contiguous().view(torch.int64))
    t = torch.arange(eng.max_step, device="cuda")
    live = t[None, None, :] < lengths[..., None]
    assert bool(torch.isnan(returns).eq(~live).all()) and bool(torch.isnan(states).eq(~live[..., None]).all())
    assert bool((actions == -1).eq(~live[..., None]).all())
    assert int(lengths.min()) < eng.max_step or env != "CartPole-v1"                   # short episodes next to long ones
    ms = np.random.default_rng(1).choice(K, 6, replace=False)
    init = initial[ms].cpu().numpy()
    assert same_bits(init, np.stack([ref.eval_init(twin, env, 11, 3, int(m)) for m in ms]))
    want = record_reference.record(twin, env, W, len(ms), gru=gru, init_states=init)
    got = numpy((initial[ms], states[:, ms], actions[:, ms], returns[:, ms], lengths[:, ms]))
    for name, g, w in zip(("initial", "states", "actions", "returns", "lengths"), got, want):
        assert same_bits(g, w), name


def test_gpu_eval_es_record_on_a_training_checkpoint(tmp_path):
    from simple_es_b200 import checkpoint
    from simple_es_b200.engine import RolloutEngine
    from simple_es_b200.loop import B200Loop
    c = _cfg("cartpole_openai.yaml", offspring_num=1024)
    B200Loop(c, 4, 1, 5, save_model_period=2, seed=3, quiet=True, save_dir=str(tmp_path / "run")).run()
    ck = [str(tmp_path / "run" / "saved_models" / f) for f in ("ep_2.pt", "ep_4.pt")]
    cfg_path = tmp_path / "c.yaml"
    cfg_path.write_text(yaml.safe_dump(c))
    out = tmp_path / "r.npz"
    subprocess.run([sys.executable, os.path.join(ROOT, "eval_es.py"), "--cfg-path", str(cfg_path), "--ckpt-path", *ck,
                    "--episodes", "300", "--seed", "5", "--round", "1", "--record", "40", "--out", str(out)],
                   capture_output=True, text=True, cwd=ROOT, check=True)
    z = np.load(out)
    assert z["returns"].shape == (2, 300) and list(z["ckpt_paths"]) == ck
    assert z["initial"].shape == (40, 4) and z["states"].shape == (2, 40, 500, 4)
    assert z["actions"].shape == (2, 40, 500, 1) and z["step_returns"].shape == (2, 40, 500)
    eng = RolloutEngine("CartPole-v1", 4, 2, False, False, 500, 1, 2, 2, 1, 1, seed=5)
    W = torch.stack([checkpoint.state_dict_to_flat(torch.load(p), 4, 2, False) for p in ck]).cuda()
    want = numpy(eng.record(W, 40, round=1))
    for name, w in zip(("initial", "states", "actions", "step_returns", "lengths"), want):
        assert same_bits(z[name] if name != "lengths" else z["lengths"][:, :40], w), name
    ret, _ = eng.evaluate(W, 300, round=1)
    assert np.array_equal(z["returns"], ret.cpu().numpy())
