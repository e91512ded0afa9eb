"""IMPALA / V-trace learner on synthetic 84x84x4 uint8 observations -- the WORKLOAD that drives the two hot paths.

This is the call sequence of the reference's examples/vtrace/experiment.py:364-531 (accumulator.update ->
has_gradients / wants_gradients -> compute_gradients + reduce_gradients -> actor step -> time_batcher.stack ->
learn_batcher.cat) with hydra/gym/wandb removed (none of them is installed in this image, SURVEY.md section 9) and the
ALE environments replaced by a synthetic observation source with the EnvPool result format
(dict of [B,...] CPU tensors: state u8 [B,4,84,84], reward f32 [B], done bool [B]).

`run_learner(api, ...)` takes the API module as an argument: `moolib_b200` (this repo) or the unmodified reference
(`moolib` from oracle/_ref*) -- the same script drives both, which is the drop-in claim.  The model (the reference's
atari ResNet: 15 conv + 3 linear layers, 1,094,476 parameters) and the V-trace loss are plain PyTorch: they are the
workload, not the product.
"""
import os
import sys
import time
from dataclasses import dataclass

_DEBUG = bool(os.environ.get("BENCH_DEBUG"))

import torch
import torch.nn as nn
import torch.nn.functional as F


# ----------------------------------------------------------------------------------------------------------------------
# model: IMPALA deep ResNet (Espeholt et al. 2018, fig. 3 right); layer shapes follow examples/atari/models.py:9-147
# ----------------------------------------------------------------------------------------------------------------------
class ResidualUnit(nn.Module):
    def __init__(self, ch):
        super().__init__()
        self.c1 = nn.Conv2d(ch, ch, 3, padding=1)
        self.c2 = nn.Conv2d(ch, ch, 3, padding=1)

    def forward(self, x):
        return x + self.c2(F.relu(self.c1(F.relu(x))))


class ImpalaNet(nn.Module):
    def __init__(self, num_actions=18, in_channels=4):
        super().__init__()
        self.num_actions = num_actions
        stages, c = [], in_channels
        for ch in (16, 32, 32):
            stages.append(nn.Sequential(nn.Conv2d(c, ch, 3, padding=1), nn.MaxPool2d(3, stride=2, padding=1),
                                        ResidualUnit(ch), ResidualUnit(ch)))
            c = ch
        self.stages = nn.Sequential(*stages)
        self.fc = nn.Linear(32 * 11 * 11, 256)
        core = 256 + num_actions + 1
        self.policy = nn.Linear(core, num_actions)
        self.baseline = nn.Linear(core, 1)
        self.normalize = None  # optional fused u8 -> float/255 (moolib_b200.u8_to_float); None: x.float() / 255.0

    def initial_state(self, batch_size=1):
        return tuple()

    def forward(self, inputs, core_state=()):
        x = inputs["state"]
        T, B = x.shape[0], x.shape[1]
        x = torch.flatten(x, 0, 1)
        x = self.normalize(x) if (self.normalize is not None and x.is_cuda) else x.float() / 255.0
        x = F.relu(self.stages(x)).reshape(T * B, -1)
        x = F.relu(self.fc(x))
        one_hot = F.one_hot(inputs["prev_action"].reshape(T * B), self.num_actions).float()
        reward = torch.clamp(inputs["reward"], -1, 1).reshape(T * B, 1)
        core = torch.cat([x, reward, one_hot], dim=-1)
        logits = self.policy(core)
        baseline = self.baseline(core)
        action = torch.multinomial(F.softmax(logits, dim=1), num_samples=1)
        return dict(policy_logits=logits.view(T, B, self.num_actions), baseline=baseline.view(T, B),
                    action=action.view(T, B)), core_state


# ----------------------------------------------------------------------------------------------------------------------
# V-trace (Espeholt et al. 2018, eq. 1-2), as examples/common/vtrace.py:156-242 computes it
# ----------------------------------------------------------------------------------------------------------------------
def action_log_probs(logits, actions):
    return -F.nll_loss(F.log_softmax(torch.flatten(logits, 0, 1), dim=-1), torch.flatten(actions, 0, 1),
                       reduction="none").view_as(actions)


@torch.no_grad()
def vtrace_targets(behavior_logits, target_logits, actions, discounts, rewards, values, bootstrap_value,
                   clip_rho=1.0, clip_pg_rho=1.0, fused=None):
    log_rhos = action_log_probs(target_logits, actions) - action_log_probs(behavior_logits, actions)
    if fused is not None and log_rhos.is_cuda:
        # moolib_b200.vtrace_from_importance_weights: the scan below as ONE kernel (bit-identical results)
        return fused(log_rhos, discounts, rewards, values, bootstrap_value, clip_rho, clip_pg_rho)
    rhos = torch.exp(log_rhos)
    clipped_rhos = torch.clamp(rhos, max=clip_rho)
    cs = torch.clamp(rhos, max=1.0)
    values_tp1 = torch.cat([values[1:], bootstrap_value.unsqueeze(0)], dim=0)
    deltas = clipped_rhos * (rewards + discounts * values_tp1 - values)
    acc = torch.zeros_like(bootstrap_value)
    out = []
    for t in range(discounts.shape[0] - 1, -1, -1):
        acc = deltas[t] + discounts[t] * cs[t] * acc
        out.append(acc)
    out.reverse()
    vs = torch.stack(out) + values
    vs_tp1 = torch.cat([vs[1:], bootstrap_value.unsqueeze(0)], dim=0)
    pg_adv = torch.clamp(rhos, max=clip_pg_rho) * (rewards + discounts * vs_tp1 - values)
    return vs, pg_adv


@dataclass
class Flags:
    actor_batch_size: int = 256       # BASELINE.json configs[1]: 256-env EnvPool
    num_actor_batches: int = 2
    unroll_length: int = 20
    batch_size: int = 32
    virtual_batch_size: int = 32
    discounting: float = 0.99
    baseline_cost: float = 0.5
    entropy_cost: float = 0.0006
    grad_norm_clipping: float = 40.0
    reward_clip: float = 1.0
    learning_rate: float = 0.0006
    num_actions: int = 18
    device: str = "cuda:0"
    host_obs: bool = True             # True: observations come from pinned host slabs (EnvPool format), H2D per step
    read_metrics: bool = True         # True: grad-norm .item() per optimizer step, as experiment.py:166 does
    obs_pool: int = 8                 # distinct pre-generated observation slabs per buffer (defeats caching)
    max_queued_batches: int = 24      # back-pressure on the actor side: both buffers' unrolls plus one (24 x 19 MB)
    fused_batcher: bool = True        # moolib_b200 only: UnrollBatcher (stack x T fused with cat, one launch per unroll)
    fused_learner_ops: bool = True    # moolib_b200 only: V-trace scan + u8->float/255 as one kernel each
    paced_actor: bool = True          # at most ceil(actor steps per learner batch) actor steps between two learner steps
                                      # while learner batches are queued: the GPU sees an even mix instead of bursts of
                                      # ~20 actor steps, so the lock-step of N learners does not wait on one peer's burst
    keep_last_batch: bool = False     # LearnerResult.last_batch = the learner batch of the latest gradient computation
    sync_ticks: bool = False          # finish all device work before every loop iteration: which iteration sees a
                                      # reduction's result then no longer depends on device progress, so the actor /
                                      # learner interleaving (and with it every result) repeats from run to run
    seed: int = 1234


def compute_gradients(model, data, flags, fused_vtrace=None):
    """experiment.py:109-156"""
    env_outputs, actor_outputs = data["env_outputs"], data["actor_outputs"]
    model.train()
    learner_outputs, _ = model(env_outputs, data.get("initial_core_state", ()))
    bootstrap_value = learner_outputs["baseline"][-1]
    learner_outputs = {k: v[:-1] for k, v in learner_outputs.items()}
    env_outputs = {k: v[1:] for k, v in env_outputs.items()}
    actor_outputs = {k: v[:-1] for k, v in actor_outputs.items()}
    rewards = env_outputs["reward"]
    if flags.reward_clip:
        rewards = torch.clip(rewards, -flags.reward_clip, flags.reward_clip)
    discounts = (~env_outputs["done"]).float() * flags.discounting
    vs, pg_adv = vtrace_targets(actor_outputs["policy_logits"], learner_outputs["policy_logits"],
                                actor_outputs["action"], discounts, rewards, learner_outputs["baseline"],
                                bootstrap_value, fused=fused_vtrace)
    logits = learner_outputs["policy_logits"]
    policy, log_policy = F.softmax(logits, dim=-1), F.log_softmax(logits, dim=-1)
    entropy_loss = flags.entropy_cost * -torch.mean(torch.sum(-policy * log_policy, dim=-1))
    pg_loss = torch.mean(-action_log_probs(logits, actor_outputs["action"]) * pg_adv.detach())
    baseline_loss = flags.baseline_cost * 0.5 * torch.mean((vs - learner_outputs["baseline"]) ** 2)
    total = entropy_loss + pg_loss + baseline_loss
    total.backward()
    return total.detach()


class SyntheticEnvPool:
    """Stand-in for moolib.EnvPool with the same calling convention (step(batch_index, action) -> future,
    future.result() -> dict of [B,...] CPU tensors aliasing internal slabs) but no Python environments behind it:
    observations are pre-generated.  host=True keeps the slabs in pinned host memory (what EnvStepperFuture.result
    returns, src/env.cc:389-401); host=False keeps them on the device (inputs resident in HBM)."""

    def __init__(self, flags, device):
        g = torch.Generator().manual_seed(flags.seed)
        B, P = flags.actor_batch_size, flags.obs_pool
        self.slabs = []
        for _ in range(flags.num_actor_batches):
            pool = []
            for _ in range(P):
                d = {"state": torch.randint(0, 256, (B, 4, 84, 84), dtype=torch.uint8, generator=g),
                     "reward": torch.randn(B, generator=g),
                     "done": torch.rand(B, generator=g) < 0.01}
                d = {k: (v.pin_memory() if flags.host_obs and torch.cuda.is_available() else v) for k, v in d.items()}
                if not flags.host_obs:
                    d = {k: v.to(device) for k, v in d.items()}
                pool.append(d)
            self.slabs.append(pool)
        self.tick = [0] * flags.num_actor_batches
        self.h2d_bytes = B * (4 * 84 * 84 + 4 + 1)
        self.d2h_bytes = B * 8

    def step(self, index, action):
        # the real EnvStepper copies the action to pinned memory and scatters it to the workers (src/env.cc:309-345)
        self.tick[index] += 1
        return _Ready(self.slabs[index][self.tick[index] % len(self.slabs[index])])


class _Ready:
    def __init__(self, v):
        self.v = v

    def result(self):
        return self.v


class LearnerResult:
    def __init__(self):
        self.optimizer_steps = 0
        self.env_train_steps = 0
        self.actor_steps = 0
        self.last_loss = None
        self.last_batch = None
        self.grad_norm_sum = 0.0
        # where the host thread spends its ticks (wall seconds, counts)
        self.t_learn = self.t_act = self.t_opt = self.t_idle = 0.0
        self.n_learn = self.n_skip = self.n_idle = 0


class LearnerLoop:
    """One learner peer: the body of the training loop of experiment.py:364-531 as a `tick()`, so that several
    peers can share one process (the way the reference's own tests fake a cluster) or one process can own one."""

    def __init__(self, api, flags, accumulator, model, optimizer, envs, group=None, broker=None, hooks=None):
        self.api, self.flags, self.acc, self.model, self.opt, self.envs = api, flags, accumulator, model, optimizer, envs
        self.group, self.broker, self.hooks = group, broker, hooks
        self.device = torch.device(flags.device)
        T, B = flags.unroll_length + 1, flags.actor_batch_size

        class EnvState:
            pass

        # moolib_b200 extensions, used when the API module has them (the reference module does not):
        #   UnrollBatcher = Batcher(T).stack x T fused with Batcher(batch_size, dim=1).cat, one launch per unroll;
        #   to_device     = EnvStepperFuture.result(device=...): all keys of a pinned result in one launch.
        self.fused = bool(flags.fused_batcher and hasattr(api, "UnrollBatcher"))
        self.to_device = getattr(api, "to_device", None)
        #   vtrace_from_importance_weights / u8_to_float = the learner's V-trace scan and input normalisation, one launch each
        self.fused_vtrace = getattr(api, "vtrace_from_importance_weights", None) if flags.fused_learner_ops else None
        if flags.fused_learner_ops and hasattr(api, "u8_to_float"):
            model.normalize = api.u8_to_float
        self.T = T
        self.env_states = []
        for _ in range(flags.num_actor_batches):
            s = EnvState()
            s.future = None
            s.prev_action = torch.zeros(B, dtype=torch.int64, device=self.device)
            s.core_state = ()
            s.initial_core_state = ()
            s.count = 0
            if self.fused:
                s.unroll = api.UnrollBatcher(T, flags.batch_size, flags.device, cat_dim=1)
            else:
                s.time_batcher = api.Batcher(T, flags.device)
            self.env_states.append(s)
        self.learn_batcher = api.Batcher(flags.batch_size, flags.device, dim=1)
        self.learn_sources = [s.unroll for s in self.env_states] if self.fused else [self.learn_batcher]
        self._next_source = 0
        # one unroll (unroll_length new actor steps) yields actor_batch_size / batch_size learner batches
        per_batch = flags.unroll_length * flags.batch_size / max(flags.actor_batch_size, 1)
        self.actor_budget = max(1, int(-(-per_batch // 1)))
        self.actor_since_learn = 0
        self.res = LearnerResult()
        self.next_env_index = 0
        self.grad_norm_dev = torch.zeros((), device=self.device)
        self._last_dbg = time.time()

    def tick(self):
        """One loop iteration.  Returns True when it performed an optimizer step."""
        flags, acc, model = self.flags, self.acc, self.model
        if flags.sync_ticks:
            torch.cuda.synchronize(self.device)
        if _DEBUG and time.time() - self._last_dbg > 5 and hasattr(acc, "debug_state"):
            self._last_dbg = time.time()
            print(f"[dbg pid {os.getpid()}] steps={self.res.optimizer_steps} actor={self.res.actor_steps} "
                  f"queued={self.learn_size()} connected={acc.connected()} wants={acc.wants_gradients()} "
                  f"{acc.debug_state()}", file=sys.stderr, flush=True)
        if self.broker is not None:
            self.broker.update()
        if self.group is not None:
            self.group.update()
        acc.update()
        if acc.wants_state():
            acc.set_state({"optimizer": self.opt.state_dict(), "steps": self.res.optimizer_steps})
        if acc.has_new_state():
            st = acc.state()
            try:
                self.opt.load_state_dict(st["optimizer"])
            except Exception:
                pass
        if not acc.connected():
            time.sleep(0.0005)
            return False
        t_tick = time.perf_counter()
        if acc.has_gradients():
            norm = nn.utils.clip_grad_norm_(model.parameters(), flags.grad_norm_clipping)
            self.opt.step()
            if flags.read_metrics:
                self.res.grad_norm_sum += norm.item()  # the per-step device->host read of experiment.py:166
            else:
                self.grad_norm_dev += norm
            acc.zero_gradients()
            self.res.optimizer_steps += 1
            self.res.t_opt += time.perf_counter() - t_tick
            return True
        if self.learn_size() and acc.wants_gradients():
            batch = self.learn_get()
            if flags.keep_last_batch:
                self.res.last_batch = batch
            self.res.last_loss = compute_gradients(model, batch, flags, self.fused_vtrace)
            self.res.env_train_steps += flags.unroll_length * flags.batch_size
            acc.reduce_gradients(flags.batch_size)
            self.actor_since_learn = 0
            self.res.n_learn += 1
            self.res.t_learn += time.perf_counter() - t_tick
            return False
        if acc.wants_gradients():
            acc.skip_gradients()
            self.res.n_skip += 1
        queued = self.learn_size()
        if queued >= self.flags.max_queued_batches or (
                flags.paced_actor and queued > 0 and self.actor_since_learn >= self.actor_budget):
            # (not in the reference loop) never let unconsumed learner batches pile up in device memory while the
            # accumulator is not asking for gradients, and do not enqueue a burst of actor steps ahead of the next
            # optimizer / learner step either
            time.sleep(0.0001)
            self.res.n_idle += 1
            self.res.t_idle += time.perf_counter() - t_tick
            return False
        cur = self.next_env_index
        self.next_env_index = (self.next_env_index + 1) % flags.num_actor_batches
        es = self.env_states[cur]
        if es.future is None:
            es.future = self.envs.step(cur, es.prev_action)
        cpu_env_outputs = es.future.result()
        if self.to_device is not None:
            env_outputs = self.to_device(cpu_env_outputs, flags.device)  # one launch for all keys (pinned slabs)
        else:
            env_outputs = {k: v.to(self.device, copy=True, non_blocking=True) for k, v in cpu_env_outputs.items()}
        env_outputs["prev_action"] = es.prev_action
        prev_core_state = es.core_state
        model.eval()
        with torch.no_grad():
            actor_outputs, es.core_state = model({k: v.unsqueeze(0) for k, v in env_outputs.items()}, es.core_state)
        actor_outputs = {k: v.squeeze(0) for k, v in actor_outputs.items()}
        action = actor_outputs["action"]
        es.prev_action = action
        del cpu_env_outputs
        es.future = self.envs.step(cur, action)
        self.res.actor_steps += 1
        self.actor_since_learn += 1
        last_data = {"env_outputs": env_outputs, "actor_outputs": actor_outputs}
        if self.fused:
            es.count += 1
            if es.count == self.T:
                # this item completes the unroll: [T, B, ...] is gathered straight into B/32 learner batches
                es.unroll.set_extra("initial_core_state", es.initial_core_state)
                self._op("unroll_gather", es.unroll.stack, last_data, self.T)
                es.initial_core_state = prev_core_state
                es.unroll.stack(last_data)
                es.count = 1
            else:
                es.unroll.stack(last_data)  # retained, no copy
        else:
            self._op("stack", es.time_batcher.stack, last_data, 1)
            if not es.time_batcher.empty():
                data = es.time_batcher.get()
                data["initial_core_state"] = es.initial_core_state
                self._op("cat", self.learn_batcher.cat, data, 1)
                es.initial_core_state = prev_core_state
                self._op("stack", es.time_batcher.stack, last_data, 1)
        self.res.t_act += time.perf_counter() - t_tick
        return False

    def learn_size(self):
        return sum(b.size() for b in self.learn_sources)

    def learn_get(self):
        for _ in range(len(self.learn_sources)):
            b = self.learn_sources[self._next_source]
            self._next_source = (self._next_source + 1) % len(self.learn_sources)
            if not b.empty():
                return b.get()
        raise RuntimeError("learn_get() without a queued learner batch")

    def _op(self, name, fn, item, items_moved):
        """Run one Batcher call; bench.py's hooks time it with CUDA events (items_moved = how many items' payload the
        call moves: an UnrollBatcher gather moves the whole unroll)."""
        if self.hooks is not None:
            self.hooks.batch_op(name, fn, item, items_moved)
        else:
            fn(item)

    def finish(self):
        if not self.flags.read_metrics:
            self.res.grad_norm_sum = float(self.grad_norm_dev.item())
        return self.res


def run_learner(api, flags, accumulator, model, optimizer, envs, on_optimizer_step, max_seconds=1e9, group=None,
                broker=None, hooks=None):
    """Drive one LearnerLoop.  `on_optimizer_step(result) -> bool` runs after every optimizer step; False stops."""
    loop = LearnerLoop(api, flags, accumulator, model, optimizer, envs, group, broker, hooks)
    t_start = time.time()
    while time.time() - t_start < max_seconds:
        if loop.tick() and not on_optimizer_step(loop.res):
            break
    return loop.finish()


def make_learner(flags):
    # algorithm selection only (no precision change): let cuDNN pick its fastest kernels for the fixed conv shapes
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(flags.seed)
    device = torch.device(flags.device)
    model = ImpalaNet(flags.num_actions).to(device)
    optimizer = torch.optim.Adam(model.parameters(), lr=flags.learning_rate)
    return model, optimizer
