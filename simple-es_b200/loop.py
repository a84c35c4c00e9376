"""B200Loop: the generation loop of the reference (learning_strategies/evolution/loop.py:14-104)
with the per-offspring multiprocessing fan-out replaced by the GPU engine.

Observable behaviour kept from ESLoop: constructor signature (plus the split config), the per
generation print line (loop.py:89-91), wandb keys (loop.py:94-99), and
``logs/<env.name>/<%Y%m%d%H%M%S>/saved_models/ep_<n>.pt`` holding the elite's
GymEnvModel-compatible state_dict every ``save_model_period`` generations (loop.py:40-47,101-104).

Opt-in (``engine.eval_every: N``): after every generation ep_num with ep_num % N == 0 the policy the loop saves
(``elite_flat()``) is evaluated on ``engine.eval_episodes`` episodes (default 100, test.py's count) keyed by ep_num, so a
resumed run reports what the uninterrupted one does; rank 0 prints one more line, wandb gets ``eval_mean_reward`` /
``eval_std_reward`` and ``eval_history`` one entry.  Every rank runs the same evaluation (identical results, no collective).
"""
import os
import time
from abc import ABCMeta, abstractmethod
from collections import deque
from datetime import datetime

import torch

from . import checkpoint
from . import dist as sdist
from .strategies import STRATEGIES


class BaseESLoop(metaclass=ABCMeta):
    """Same two-method contract as the reference's BaseESLoop (learning_strategies/evolution/abstracts.py:5-12)."""

    @abstractmethod
    def __init__(self):
        pass

    @abstractmethod
    def run(self):
        pass


class B200Loop(BaseESLoop):
    def __init__(self, config, generation_num, process_num, eval_ep_num, log=False, save_model_period=10,
                 seed=0, device=None, save_dir=None, quiet=False):
        super().__init__()
        self.config = config
        env_cfg, net_cfg, strat_cfg = config["env"], config["network"], config["strategy"]
        self.engine_cfg = dict(config.get("engine") or {})
        if net_cfg.get("name") != "gym_model":
            raise ValueError("the B200 engine implements the reference's only network, gym_model (builder.py:17-24)")
        if strat_cfg["name"] not in STRATEGIES:
            raise ValueError("unknown strategy %r" % strat_cfg["name"])
        self.rank, self.world = sdist.init_from_env()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(device)
        self.process_num = process_num                    # accepted for CLI compatibility; the GPU replaces the pool
        self.generation_num = generation_num
        self.eval_ep_num = eval_ep_num
        self.log = log
        self.save_model_period = save_model_period
        self.quiet = quiet
        self.ep5_rewards = deque(maxlen=5)
        self.env_name = env_cfg["name"]
        self.net_cfg = net_cfg
        self.strategy = STRATEGIES[strat_cfg["name"]](strat_cfg, env_cfg, net_cfg, eval_ep_num, seed, device, self.engine_cfg)
        self.history = []
        self.eval_history = []             # (ep_num, episodes, mean, std, min, max, mean length, seconds) per evaluation
        self.eval_every = int(self.engine_cfg.get("eval_every", 0) or 0)
        self.eval_episodes = int(self.engine_cfg.get("eval_episodes", 100))
        if self.eval_every < 0 or self.eval_episodes < 1:
            raise ValueError("engine.eval_every must be >= 0 and engine.eval_episodes >= 1")
        self.start_ep = 0
        # engine.init_from: a reference-format checkpoint (GymEnvModel.state_dict(), e.g. a saved ep_<n>.pt) as the initial
        # mu / elites; engine.resume: a resume_ep_<n>.pt written by this loop (engine.save_state: true) -- continues the
        # run bit for bit (parameters, sigma, Adam state, generation counter)
        if self.engine_cfg.get("init_from") and self.engine_cfg.get("resume"):
            raise ValueError("engine.init_from and engine.resume are exclusive: a resume state already holds the parameters")
        if self.engine_cfg.get("init_from"):
            sd = torch.load(self.engine_cfg["init_from"], map_location="cpu")
            self.strategy.load_elite(checkpoint.state_dict_to_flat(sd, int(net_cfg["num_state"]), int(net_cfg["num_action"]), bool(net_cfg["gru"])))
        if self.engine_cfg.get("resume"):
            st = torch.load(self.engine_cfg["resume"], map_location="cpu")
            self.strategy.load_state(st)
            self.start_ep = int(st["generation"])
            self.ep5_rewards.extend(st.get("ep5_rewards", []))

        self.save_dir = save_dir
        if self.rank == 0 and self.save_model_period and self.save_model_period > 0:
            if self.save_dir is None:
                self.save_dir = f"logs/{self.env_name}/{datetime.now().strftime('%Y%m%d%H%M%S')}"
            os.makedirs(self.save_dir + "/saved_models/", exist_ok=True)
        self._wandb = None
        if self.log and self.rank == 0:
            import wandb
            wandb.init(project=self.env_name, config=config)
            self._wandb = wandb

    def elite_state_dict(self):
        n = self.net_cfg
        return checkpoint.flat_to_state_dict(self.strategy.elite_flat(), int(n["num_state"]), int(n["num_action"]), bool(n["gru"]))

    def evaluate_elite(self, ep_num):
        """Returns of the policy elite_flat() on eval_episodes episodes keyed by ep_num: one eval_history entry."""
        start = time.time()
        ret, lng = self.strategy.engine.evaluate(self.strategy.elite_flat(), self.eval_episodes, round=ep_num)
        ret, lng = ret[0].cpu(), lng[0].to(torch.float64).cpu()
        std = float(ret.std(unbiased=False)) if ret.numel() > 1 else 0.0
        entry = (ep_num, ret.numel(), float(ret.mean()), std, float(ret.min()), float(ret.max()), float(lng.mean()), time.time() - start)
        self.eval_history.append(entry)
        return entry

    def run(self):
        s = self.strategy
        s.timing = True                                      # CUDA-event marks around K1 + exchange and K2 + K3
        ep_num = self.start_ep
        for _ in range(self.generation_num):
            start = time.time()
            ep_num += 1
            s.step()
            best_reward = float(s.best_reward().item())      # the one device->host sync of a generation
            if s.exchange == "peer":
                # the stream is idle now, so this 4-byte read costs nothing: a peer GPU that missed the flag barrier
                # (watchdog, SES_PEER_TIMEOUT_MS) must stop the run instead of letting the ranks drift apart
                s.engine.peer_check()
            consumed = time.time() - start
            # rollout_t / eval_t (loop.py:70-88) are device times here: K1 + fitness exchange, and K2 + K3, taken from CUDA
            # events that the sync above has completed -- the phases are one stream-ordered pass, the host never waits between
            rollout_t, eval_t = s.phase_times() or (consumed, 0.0)
            curr_sigma = s.curr_sigma
            self.history.append((ep_num, best_reward, curr_sigma, consumed, rollout_t, eval_t))
            if self.rank == 0 and not self.quiet:
                print(f"episode: {ep_num}, Best reward: {best_reward:.2f}, sigma: {curr_sigma:.3f}, "
                      f"time: {consumed:.2f}, rollout_t: {rollout_t:.2f}, eval_t: {eval_t:.2f}")
            if self._wandb is not None:
                self.ep5_rewards.append(best_reward)
                self._wandb.log({"ep5_mean_reward": sum(self.ep5_rewards) / len(self.ep5_rewards),
                                 "curr_sigma": curr_sigma})
            if self.eval_every and ep_num % self.eval_every == 0:
                _, n, mean, std, lo, hi, mlen, secs = self.evaluate_elite(ep_num)
                if self.rank == 0 and not self.quiet:
                    print(f"  eval: {n} episodes, mean {mean:.2f}, std {std:.2f}, min {lo:.2f}, max {hi:.2f}, "
                          f"mean length {mlen:.1f}, time: {secs:.2f}")
                if self._wandb is not None:
                    self._wandb.log({"eval_mean_reward": mean, "eval_std_reward": std})
            if self.rank == 0 and self.save_model_period and self.save_model_period > 0 and ep_num % self.save_model_period == 0:
                torch.save(self.elite_state_dict(), self.save_dir + "/saved_models" + f"/ep_{ep_num}.pt")
                if self.engine_cfg.get("save_state"):
                    torch.save(dict(s.state(), ep5_rewards=list(self.ep5_rewards)), self.save_dir + "/saved_models" + f"/resume_ep_{ep_num}.pt")
        return self.history
