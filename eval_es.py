#!/usr/bin/env python
"""Evaluate saved policies on the GPU engine: the per-episode returns of the reference's test.py (test.py:31-68), without
its rendering.

    python eval_es.py --cfg-path conf/cartpole.yaml --ckpt-path logs/CartPole-v1/<ts>/saved_models/ep_100.pt [more.pt ...] \\
        --episodes 100 --seed 0 [--round 0] [--out returns.npz [--record K]]

Each checkpoint is a GymEnvModel state_dict (ep_<n>.pt, as B200Loop and the reference save them).  All checkpoints run in
one call on the same episodes: episode m starts from the env's reset distribution keyed by (seed, round, m), so policies are
compared on identical initial states.  One line per checkpoint; --out writes returns [n_ckpt, episodes] (float64), lengths
[n_ckpt, episodes] (int32) and the checkpoint paths to an .npz file.

--archive PATH evaluates every elite of a map_elites archive file (archive_ep_<n>.pt, as B200Loop saves it) in one call
instead of checkpoints: one summary line, and --out writes returns / lengths [n_elites, episodes] with the archive's cells.
An elite's fitness in the archive comes from the eval_ep_num training episodes of its generation; this re-scores it.

--record K also records the first K of those episodes step by step and adds them to --out: initial [K, state_dim] (the
initial states), states [n_ckpt, K, T, state_dim] (the state after each step; for the gym envs their env.unwrapped.state, so
a gym install can replay them into its renderer), actions [n_ckpt, K, T, n_agents], step_returns [n_ckpt, K, T] (the return
after each step), T = the episode cap; steps past an episode's end hold NaN / -1.  The episodes' lengths are the first K
columns of `lengths`.
"""
import argparse

import numpy as np
import yaml


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--cfg-path", required=True, help="training config (its env and network sections are used).")
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("--ckpt-path", nargs="+", help="GymEnvModel state_dict(s) to evaluate.")
    src.add_argument("--archive", default=None, help="a map_elites archive file (archive_ep_<n>.pt): evaluate every elite.")
    ap.add_argument("--episodes", type=int, default=100, help="episodes per checkpoint (test.py runs 100).")
    ap.add_argument("--seed", type=int, default=0, help="seed of the initial states.")
    ap.add_argument("--round", type=int, default=0, help="another set of initial states under the same seed.")
    ap.add_argument("--out", default=None, help="write returns, lengths and the checkpoint paths to this .npz file.")
    ap.add_argument("--record", type=int, default=None, metavar="K",
                    help="also record the first K episodes step by step (states, actions, returns) into --out.")
    ap.add_argument("--device", type=int, default=0, help="CUDA device.")
    args = ap.parse_args(argv)
    if args.episodes < 1:
        ap.error("--episodes must be >= 1")
    if args.record is not None:
        if args.archive:
            ap.error("--record takes checkpoints (--ckpt-path), not --archive")
        if not args.out:
            ap.error("--record needs --out")
        if not 1 <= args.record <= args.episodes:
            ap.error("--record K needs 1 <= K <= --episodes")
    if not 0 <= args.round < 2 ** 32:
        ap.error("--round must be in [0, 2^32)")
    return args


def engine_config(config):
    """RolloutEngine keyword arguments of a training config's env / network / engine sections."""
    env, net, eng = config["env"], config["network"], config.get("engine") or {}
    if net.get("name", "gym_model") != "gym_model":
        raise ValueError("the B200 engine implements the reference's only network, gym_model")
    return dict(env_name=env["name"], obs_dim=int(net["num_state"]), act_dim=int(net["num_action"]), gru=bool(net["gru"]),
                pomdp=bool(env.get("pomdp", False)), max_step=env.get("max_step"), n_agents=int(eng.get("n_agents", 2)),
                discrete_action=bool(net.get("discrete_action", True)))


def load_policies(paths, obs_dim, act_dim, gru):
    """[n_ckpt, D] float32 (CPU) from GymEnvModel state_dicts."""
    import torch

    from simple_es_b200 import checkpoint
    want = [name for name, _ in checkpoint.param_shapes(obs_dim, act_dim, gru)]
    flats = []
    for p in paths:
        sd = torch.load(p, map_location="cpu")
        if sorted(sd) != sorted(want):
            raise ValueError("%s holds %s; the config's network needs %s" % (p, ", ".join(sd), ", ".join(want)))
        flats.append(checkpoint.state_dict_to_flat(sd, obs_dim, act_dim, gru))
    return torch.stack(flats)


def load_archive(path, obs_dim, act_dim, gru):
    """(weights [n_elites, D] float32 CPU, cells [n_elites] int64) of a map_elites archive file."""
    import torch

    from simple_es_b200 import checkpoint
    a = torch.load(path, map_location="cpu")
    if not isinstance(a, dict) or "weights" not in a or "cells" not in a:
        raise ValueError("%s is not a map_elites archive file (archive_ep_<n>.pt)" % path)
    D = sum(int(np.prod(shape)) for _, shape in checkpoint.param_shapes(obs_dim, act_dim, gru))
    W = torch.as_tensor(a["weights"], dtype=torch.float32)
    if W.dim() != 2 or W.shape[1] != D:
        raise ValueError("%s holds weights of shape %s; the config's network has %d parameters" % (path, tuple(W.shape), D))
    if W.shape[0] == 0:
        raise ValueError("%s holds an empty archive" % path)
    return W, torch.as_tensor(a["cells"], dtype=torch.int64)


def main(argv=None):
    args = parse_args(argv)
    with open(args.cfg_path) as fh:
        config = yaml.load(fh, Loader=yaml.FullLoader)
    kw = engine_config(config)
    if args.archive:
        W, cells = load_archive(args.archive, kw["obs_dim"], kw["act_dim"], kw["gru"])
    else:
        W = load_policies(args.ckpt_path, kw["obs_dim"], kw["act_dim"], kw["gru"])
    from simple_es_b200.engine import RolloutEngine
    # the population layout of the handle plays no part in an evaluation: the smallest valid one
    eng = RolloutEngine(eval_ep_num=1, population=2, group=2, n_head=1, n_parents=1, seed=args.seed, device=args.device, **kw)
    ret, lng = eng.evaluate(W.to(eng.device), args.episodes, round=args.round)
    ret, lng = ret.cpu().numpy(), lng.cpu().numpy()
    if args.archive:
        means = ret.mean(axis=1)
        b = int(np.argmax(means))
        print(f"{args.archive}: {ret.shape[0]} elites x {ret.shape[1]} episodes, mean of elite means {means.mean():.2f}, "
              f"best elite cell {int(cells[b])} mean {means[b]:.2f}, worst elite mean {means.min():.2f}")
        if args.out:
            np.savez(args.out, returns=ret, lengths=lng, cells=cells.numpy(), archive=np.array(args.archive))
        eng.close()
        return ret, lng
    for path, r, n in zip(args.ckpt_path, ret, lng):
        print(f"{path}: {r.size} episodes, mean {r.mean():.2f}, std {r.std():.2f}, min {r.min():.2f}, max {r.max():.2f}, "
              f"mean length {n.mean():.1f}")
    recorded = {}
    if args.record:
        rec = eng.record(W.to(eng.device), args.record, round=args.round)           # its lengths are lng[:, :K]
        recorded = {k: t.cpu().numpy() for k, t in zip(("initial", "states", "actions", "step_returns"), rec[:4])}
    if args.out:
        np.savez(args.out, returns=ret, lengths=lng, ckpt_paths=np.array(args.ckpt_path), **recorded)
    eng.close()
    return ret, lng


if __name__ == "__main__":
    main()
