"""Episode recording without a GPU: eval_es.py --record's command line and RolloutEngine.record's argument checks, which run
before any device work."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import eval_es  # noqa: E402
from simple_es_b200.engine import RolloutEngine  # noqa: E402

BASE = ["--cfg-path", "c.yaml", "--ckpt-path", "a.pt"]


def test_eval_es_record_arguments():
    a = eval_es.parse_args(BASE)
    assert a.record is None
    a = eval_es.parse_args(BASE + ["--episodes", "20", "--record", "20", "--out", "r.npz"])
    assert (a.episodes, a.record, a.out) == (20, 20, "r.npz")
    a = eval_es.parse_args(BASE + ["--record", "1", "--out", "r.npz"])
    assert (a.episodes, a.record) == (100, 1)
    for bad in (["--record", "5"],                                           # nowhere to write the recording
                ["--record", "101", "--out", "r.npz"],                       # more than --episodes (100)
                ["--episodes", "4", "--record", "5", "--out", "r.npz"],
                ["--record", "0", "--out", "r.npz"],
                ["--record", "-2", "--out", "r.npz"],
                ["--record", "x", "--out", "r.npz"]):
        with pytest.raises(SystemExit):
            eval_es.parse_args(BASE + bad)


def test_eval_es_record_errors_are_reported(capsys):
    with pytest.raises(SystemExit):
        eval_es.parse_args(BASE + ["--record", "5"])
    assert "--record needs --out" in capsys.readouterr().err
    with pytest.raises(SystemExit):
        eval_es.parse_args(BASE + ["--episodes", "4", "--record", "5", "--out", "r.npz"])
    assert "1 <= K <= --episodes" in capsys.readouterr().err


def test_engine_record_checks_its_arguments():
    eng = object.__new__(RolloutEngine)                            # argument checks run before any device work
    eng.D, eng.max_step, eng.state_dim = 226, 500, 4
    with pytest.raises(ValueError, match=r"expected \[226\] or \[n_pol, 226\]"):
        eng.record(torch.zeros(225), 10)
    with pytest.raises(ValueError, match=r"expected \[226\]"):
        eng.record(torch.zeros(2, 3, 226), 10)
    with pytest.raises(ValueError, match=r"expected \[226\]"):
        eng.record(np.zeros(226, np.float32), 10)
    with pytest.raises(ValueError, match="float32 CUDA tensor"):
        eng.record(torch.zeros(3, 226), 10)
    with pytest.raises(ValueError, match="float32 CUDA tensor"):
        eng.record(torch.zeros(3, 226, dtype=torch.float64), 10)
