"""Host-side mirror of the reference interface that needs no GPU: the C ABI surface, the builder
switch, the CLI flags and the checkpoint format."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    """The product library exports exactly what include/ses_b200.h declares -- and none of the test hooks; the test build
    (-DSES_BUILD_TESTS, include/ses_b200_test.h) exports both."""
    from simple_es_b200 import _lib
    _lib.build_all()
    header = open(os.path.join(ROOT, "include", "ses_b200.h")).read()
    declared = set(re.findall(r"\b(ses_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    theader = open(os.path.join(ROOT, "include", "ses_b200_test.h")).read()
    tdeclared = set(re.findall(r"\b(ses_test_[a-z0-9_]+)\s*\(", theader))
    assert tdeclared == set(_lib.TEST_SYMBOLS), tdeclared ^ set(_lib.TEST_SYMBOLS)
    lib = C.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    for name in tdeclared:
        assert not hasattr(lib, name), "test hook %s leaked into the product library" % name
    tlib = C.CDLL(_lib.TEST_LIB_PATH)
    for name in declared | tdeclared:
        assert hasattr(tlib, name), name
    # one rollout kernel per (environment, policy, slots per warp) in the product: no alternative CartPole-MLP variants
    names = subprocess.run(["cuobjdump", "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    variants = set(re.findall(r"CartpoleMlpEnvTILi(\d)E", names))
    assert variants == {"7"}, variants
    lib = _lib.load()
    assert lib.ses_abi_version() == 1
    assert lib.ses_param_count(4, 2, 0) == 226 and lib.ses_param_count(4, 2, 1) == 6562
    assert lib.ses_param_count(12, 5, 0) == 581 and lib.ses_param_count(18, 5, 0) == 773
    assert C.sizeof(_lib.ses_config) == 24 * 4                 # matches the C struct layout


def test_ctypes_struct_matches_the_c_header(tmp_path):
    """simple-es_b200/_lib.py::ses_config must have the layout of include/ses_b200.h's struct (size and every field
    offset), checked with a C program compiled against the header."""
    import ctypes as C
    import subprocess
    from simple_es_b200 import _lib
    names = [n for n, _ in _lib.ses_config._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ses_b200.h"\nint main(void){printf("%zu\\n", sizeof(ses_config));'
                   + "".join('printf("%%zu\\n", offsetof(ses_config, %s));' % n for n in names) + "return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    out = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert out[0] == C.sizeof(_lib.ses_config) == 96
    assert out[1:] == [getattr(_lib.ses_config, n).offset for n in names]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from simple_es_b200 import _lib
    from simple_es_b200.engine import RolloutEngine
    lib = _lib.load()
    cfg = _lib.ses_config(env=0, obs_dim=4, act_dim=2, eval_ep_num=5, population=97, group=97, n_head=2, n_parents=1, id_end=97)
    h = C.c_void_p()
    assert lib.ses_create(C.byref(cfg), C.byref(h)) != 0
    assert b"no CUDA device" in lib.ses_last_error()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        RolloutEngine("CartPole-v1", 4, 2, False, False, 500, 5, 97, 97, 2, 1)


def test_engine_rejects_out_of_scope_envs():
    from simple_es_b200.engine import RolloutEngine
    with pytest.raises(ValueError, match="not supported"):
        RolloutEngine("LunarLander-v2", 8, 4, False, False, 500, 5, 97, 97, 2, 1)


def test_builder_switch_and_configs():
    import builder
    for name in os.listdir(os.path.join(ROOT, "conf")):
        cfg = yaml.load(open(os.path.join(ROOT, "conf", name)), Loader=yaml.FullLoader)
        assert builder.engine_name(cfg) == "b200"
        assert set(cfg) >= {"env", "network", "strategy", "engine"}
    ref_style = yaml.load(open(os.path.join(ROOT, "conf", "cartpole.yaml")), Loader=yaml.FullLoader)
    ref_style.pop("engine")
    with pytest.raises(RuntimeError, match="engine"):           # no silent CPU re-implementation
        builder.build_loop(ref_style, 1, 1, 5, False, 10)
    # max_step: None parses as the string "None", as in the reference (gym_wrapper.py:37)
    spread = yaml.load(open(os.path.join(ROOT, "conf", "simplespread.yaml")), Loader=yaml.FullLoader)
    assert spread["env"]["max_step"] == "None"


def test_configs_without_engine_key_reach_the_reference_builder_by_path(tmp_path, monkeypatch):
    """ADVICE r1: run_es.py / sweep_main.py import THIS repository's top-level `builder` shim, so the reference's module of
    the same name can only be reached by path (SES_REFERENCE_ROOT/builder.py), with the checkout's root importable while
    it executes.  A stand-in checkout records that its own build_loop received the call, through the shim the entry
    points import."""
    import builder
    from simple_es_b200 import builder as impl
    (tmp_path / "envs.py").write_text("NAME = 'stand-in envs package of the checkout'\n")
    (tmp_path / "builder.py").write_text(
        "import envs\n"
        "def build_loop(config, gen_num, process_num, eval_ep_num, log, save_model_period):\n"
        "    return ('reference loop', envs.NAME, config['env']['name'], gen_num, process_num, eval_ep_num, log, save_model_period)\n")
    monkeypatch.setenv("SES_REFERENCE_ROOT", str(tmp_path))
    monkeypatch.setattr(impl, "_REF_BUILDER", None)
    cfg = {"env": {"name": "LunarLander-v2"}, "network": {}, "strategy": {}}
    got = builder.build_loop(cfg, 7, 3, 5, False, 10)
    assert got == ("reference loop", "stand-in envs package of the checkout", "LunarLander-v2", 7, 3, 5, False, 10)
    # a checkout whose dependencies are missing fails loudly and names the module that is missing
    (tmp_path / "builder.py").write_text("import gym_that_is_not_installed\n")
    monkeypatch.setattr(impl, "_REF_BUILDER", None)
    with pytest.raises(RuntimeError, match="gym_that_is_not_installed"):
        builder.build_loop(cfg, 1, 1, 5, False, 10)
    monkeypatch.delenv("SES_REFERENCE_ROOT")
    monkeypatch.setattr(impl, "_REF_BUILDER", None)
    with pytest.raises(RuntimeError, match="SES_REFERENCE_ROOT"):
        builder.build_loop(cfg, 1, 1, 5, False, 10)
    sys.modules.pop("envs", None)


def test_cli_flags_match_reference():
    import run_es
    a = run_es.parse_args([])
    assert (a.seed, a.process_num, a.generation_num, a.eval_ep_num, a.log, a.save_model_period) == (0, 12, 10000, 5, False, 10)
    a = run_es.parse_args(["--cfg-path", "x.yaml", "--seed", "3", "--process-num", "2", "--generation-num", "7",
                           "--eval-ep-num", "9", "--log", "--save-model-period", "4"])
    assert (a.cfg_path, a.seed, a.process_num, a.generation_num, a.eval_ep_num, a.log, a.save_model_period) == ("x.yaml", 3, 2, 7, 9, True, 4)


def test_sweep_cli_overrides_reach_the_engine_config():
    """sweep_main.py keeps the reference's flags (sweep_main.py:33-69: generation-num 1000, --log store_false, the five
    hyper-parameter overrides) and writes every given override into the YAML key of the same name, as change_value does
    (sweep_main.py:16-30); keys a config does not have are not invented."""
    import sweep_main
    a = sweep_main.parse_args([])
    assert (a.seed, a.process_num, a.generation_num, a.eval_ep_num, a.log, a.save_model_period) == (0, 12, 1000, 5, True, 10)
    assert (a.init_sigma, a.sigma_decay, a.learning_rate, a.elite_num, a.offspring_num) == (None,) * 5
    a = sweep_main.parse_args(["--cfg-path=conf/cartpole_openai.yaml", "--init-sigma=0.3", "--learning-rate=0.05",
                               "--offspring-num=4096", "--elite-num=7", "--log"])
    assert a.log is False
    cfg = yaml.load(open(os.path.join(ROOT, a.cfg_path)), Loader=yaml.FullLoader)
    before = dict(cfg["strategy"])
    changed = sweep_main.apply_overrides(cfg, {"init_sigma": a.init_sigma, "sigma_decay": a.sigma_decay, "learning_rate": a.learning_rate,
                                               "elite_num": a.elite_num, "offspring_num": a.offspring_num})
    assert sorted(changed) == ["strategy.init_sigma", "strategy.learning_rate", "strategy.offspring_num"]
    assert cfg["strategy"]["init_sigma"] == 0.3 and cfg["strategy"]["learning_rate"] == 0.05 and cfg["strategy"]["offspring_num"] == 4096
    assert cfg["strategy"]["sigma_decay"] == before["sigma_decay"] and "elite_num" not in cfg["strategy"]
    assert cfg["engine"]["name"] == "b200"
    for name in os.listdir(os.path.join(ROOT, "sweep_config")):
        sw = yaml.load(open(os.path.join(ROOT, "sweep_config", name)), Loader=yaml.FullLoader)
        assert sw["program"] == "sweep_main.py" and sw["metric"]["name"] == "ep5_mean_reward"
        target = yaml.load(open(os.path.join(ROOT, sw["parameters"]["cfg-path"]["value"])), Loader=yaml.FullLoader)
        assert target["engine"]["name"] == "b200"
        flags = {f.lstrip("-") for f, _ in sweep_main.OVERRIDES} | {f[0].lstrip("-") for f in __import__("run_es").FLAGS}
        assert set(sw["parameters"]) <= flags


@pytest.mark.parametrize("obs,act,gru,D", [(4, 2, False, 226), (4, 2, True, 6562), (12, 5, False, 581)])
def test_checkpoint_roundtrip_and_reference_keys(obs, act, gru, D):
    from simple_es_b200 import checkpoint
    flat = torch.arange(D, dtype=torch.float32)
    sd = checkpoint.flat_to_state_dict(flat, obs, act, gru)
    want = ["fc1.weight", "fc1.bias"] + (["gru.weight_ih_l0", "gru.weight_hh_l0", "gru.bias_ih_l0", "gru.bias_hh_l0"] if gru else []) + ["fc2.weight", "fc2.bias"]
    assert list(sd) == want
    assert torch.equal(checkpoint.state_dict_to_flat(sd, obs, act, gru), flat)
    # loads into a torch module shaped like the reference's GymEnvModel (networks/neural_network.py:12-17)
    class M(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1 = torch.nn.Linear(obs, 32)
            if gru:
                self.gru = torch.nn.GRU(32, 32)
            self.fc2 = torch.nn.Linear(32, act)
    m = M()
    m.load_state_dict(sd)
    assert torch.equal(torch.cat([p.detach().reshape(-1) for p in m.parameters()]), flat)


def test_checkpoint_loads_into_reference_model(golden):
    """A checkpoint of the reference's flat GRU parameter vectors (tests/golden/policy_gru.npz: vectors applied to the
    reference's own GymEnvModel(4, 2, True, True) and the fc2 outputs it computed), loaded by name as the reference's
    test.py:39-40 does into a module with GymEnvModel's layout and forward (networks/neural_network.py:12-40), must
    reproduce every logit the reference computed."""
    from simple_es_b200 import checkpoint
    g = golden("policy_gru")
    W, O, Z = g["W"], g["obs"], g["logits"]

    class GymEnvModel(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1 = torch.nn.Linear(4, 32)
            self.gru = torch.nn.GRU(32, 32)
            self.fc2 = torch.nn.Linear(32, 2)

        def forward(self, x, h):
            x, h = self.gru(torch.tanh(self.fc1(x)), h)
            return self.fc2(torch.tanh(x)), h

    model = GymEnvModel()
    worst = 0.0
    with torch.no_grad():
        for i in range(W.shape[0]):
            model.load_state_dict(checkpoint.flat_to_state_dict(torch.from_numpy(W[i]), 4, 2, True))
            h = torch.zeros(1, 1, 32)
            for t in range(O.shape[1]):
                z, h = model(torch.from_numpy(O[i, t]).float().view(1, 1, 4), h)
                worst = max(worst, float(np.abs(z.numpy().ravel() - Z[i, t]).max() / max(1.0, np.abs(Z[i, t]).max())))
    assert worst < 1e-6
