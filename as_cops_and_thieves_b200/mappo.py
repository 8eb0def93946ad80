"""MAPPO learner over the batched environment (SURVEY.md §8 f-1; BASELINE.json config 5).

skrl is not installable in this image, so this module restates the part of
``skrl.multi_agents.torch.mappo.MAPPO`` + ``SequentialTrainer`` that the reference drives
(``/root/reference/src/training/orchestration.py:100-249``,
``/root/reference/src/utils/agent_learning_utils.py:172-231``) with the reference's hyper-parameters
(``/root/reference/src/configs/mappo_config.py:5-63``) and model architectures
(``/root/reference/src/models/lstm_policy_net.py:25-53`` — 340,388 parameters,
``lstm_value_net.py:47-86`` — 522,337, ``policy_net.py:17-33``, ``value_net.py:18-28``) in plain PyTorch:

* rollout memory on the device, ``rollouts`` steps x N worlds, one policy + one centralised critic per agent;
* GAE + advantage normalisation through the CUDA kernels (``gae.compute_gae`` -> ``cat_gae`` /
  ``cat_adv_normalize``);
* PPO-clip surrogate, entropy bonus, scaled value loss, KL early stop, grad-norm clip (skrl's ``_update``);
* under ``torchrun`` the gradients of every minibatch are all-reduced over NCCL in one flat bucket
  (every parameter's ``.grad`` is a view into it) — the only collective in the system besides the optional advantage
  statistics.

Differences from the reference that batching forces (documented, not hidden):

* the reference's LSTM models chop the *batch* dimension into pseudo-sequences of 16 because skrl feeds them
  one environment; here every world carries its own (h, c), reset when its episode ends, and PPO trains on
  true 16-step sequences per world (``sequence_length``, ``lstm_policy_net.py:16``) starting from the hidden
  state recorded during the rollout;
* ``rollouts`` counts lockstep steps of N worlds, so one update sees ``rollouts x N`` transitions per agent.

The dense nets are library PyTorch (cuDNN / cuBLAS) on purpose: SURVEY.md §2 #11 puts them out of scope for
hand-written kernels.
"""
from __future__ import annotations

import itertools
import time
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional, Tuple

import torch
import torch.nn as nn


N_RAYS = 90


# ------------------------------------------------------------------ models
def _ray_features(in_channels: int, length: int, out_features: int = 256) -> nn.Sequential:
    """Conv1d(k5,s2) -> Conv1d(k5,s3) -> Linear -> Tanh over ray channels (lstm_policy_net.py:27-35)."""
    l1 = (length - 5) // 2 + 1
    l2 = (l1 - 5) // 3 + 1
    return nn.Sequential(nn.Conv1d(in_channels, 64, kernel_size=5, stride=2), nn.ReLU(),
                         nn.Conv1d(64, 32, kernel_size=5, stride=3), nn.ReLU(),
                         nn.Flatten(), nn.Linear(32 * l2, out_features), nn.Tanh())


class _Recurrent(nn.Module):
    """Shared sequence logic: an LSTM over (B, L, F) whose state is zeroed wherever ``reset[b, t]`` is set
    BEFORE step t is consumed (an episode of world b ended at step t-1).  Without resets this is one cuDNN
    call; with resets the sequence is cut at the steps where any row resets (the reference cuts at terminated
    steps the same way, ``lstm_policy_net.py:183-210``)."""

    lstm: nn.LSTM

    def run_lstm(self, x: torch.Tensor, hc: Tuple[torch.Tensor, torch.Tensor], reset: Optional[torch.Tensor]):
        h, c = hc
        if reset is not None and x.size(1) == 1:
            # one step (the rollout): mask instead of branching, so the call needs no host sync and can be
            # captured in a CUDA graph
            keep = (~reset[:, 0]).to(x.dtype).view(1, -1, 1)
            return self.lstm_step(x[:, 0], h * keep, c * keep)
        if reset is None or not bool(reset.any()):
            out, (h, c) = self.lstm(x, (h.contiguous(), c.contiguous()))
            return out, (h, c)
        L = x.size(1)
        cuts = [0] + [int(t) for t in torch.nonzero(reset.any(dim=0)).flatten().tolist() if t > 0] + [L]
        outs = []
        for t0, t1 in zip(cuts[:-1], cuts[1:]):
            keep = (~reset[:, t0]).to(x.dtype).view(1, -1, 1)
            h, c = h * keep, c * keep
            o, (h, c) = self.lstm(x[:, t0:t1], (h.contiguous(), c.contiguous()))
            outs.append(o)
        return torch.cat(outs, dim=1), (h, c)

    def lstm_step(self, x: torch.Tensor, h: torch.Tensor, c: torch.Tensor):
        """One time step of ``self.lstm`` as two GEMMs + pointwise gates per layer (gate order i, f, g, o).
        cuDNN's RNN entry point costs ~1 ms per call at sequence length 1 whatever the batch, which would make
        the rollout 30x slower than the environment step it feeds; this is the same arithmetic without it."""
        hs, cs, inp = [], [], x
        for layer in range(self.lstm.num_layers):
            w_ih, w_hh = getattr(self.lstm, f"weight_ih_l{layer}"), getattr(self.lstm, f"weight_hh_l{layer}")
            bias = getattr(self.lstm, f"bias_ih_l{layer}") + getattr(self.lstm, f"bias_hh_l{layer}")
            gates = torch.addmm(bias, inp, w_ih.t()) + h[layer] @ w_hh.t()
            i, f, g, o = gates.chunk(4, dim=1)
            c_new = torch.sigmoid(f) * c[layer] + torch.sigmoid(i) * torch.tanh(g)
            inp = torch.sigmoid(o) * torch.tanh(c_new)
            hs.append(inp)
            cs.append(c_new)
        return inp.unsqueeze(1), (torch.stack(hs), torch.stack(cs))

    def initial_state(self, batch: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
        z = torch.zeros(self.lstm.num_layers, batch, self.lstm.hidden_size, device=device)
        return z, z.clone()


class LSTMPolicyNet(_Recurrent):
    """``LSTMPolicy`` (lstm_policy_net.py:6-53): ray CNN (2 channels: distance | object_type) -> LSTM(256 -> 128)
    -> 128 -> 64 -> 4 logits."""

    recurrent = True

    def __init__(self, n_obs: int = 2 * N_RAYS, n_actions: int = 4, hidden_size: int = 128, num_layers: int = 1):
        super().__init__()
        self.len_ch = n_obs // 2
        self.features_extractor = _ray_features(2, self.len_ch)
        self.lstm = nn.LSTM(256, hidden_size, num_layers=num_layers, batch_first=True)
        self.policy_head = nn.Sequential(nn.Linear(hidden_size, 128), nn.ReLU(), nn.Linear(128, 64), nn.ReLU(),
                                         nn.Linear(64, n_actions))

    def forward(self, obs: torch.Tensor, hc, reset: Optional[torch.Tensor] = None):
        """``obs`` (B, L, 180) -> logits (B, L, 4), new state."""
        B, L, _ = obs.shape
        f = self.features_extractor(obs.reshape(B * L, 2, self.len_ch)).view(B, L, -1)
        out, hc = self.run_lstm(f, hc, reset)
        return self.policy_head(out), hc


class LSTMValueNet(_Recurrent):
    """``LSTMValue`` (lstm_value_net.py:6-86,122-137): 4 ray channels cut from the FIRST 360 state columns
    (own_obj_types, own_distances, object_type_shared, distance_shared of the first agent's block — the
    reference reads that block for every agent's critic, SURVEY.md C-8) -> CNN -> LSTM(256 -> 128, 2 layers) ->
    256 -> 128 -> 64 -> 1."""

    recurrent = True

    def __init__(self, n_state: int = 1090, hidden_size: int = 128, num_layers: int = 2, length: int = N_RAYS):
        super().__init__()
        self.length = length
        self.features_extractor = _ray_features(4, length)
        self.lstm = nn.LSTM(256, hidden_size, num_layers=num_layers, batch_first=True)
        self.value_head = nn.Sequential(nn.Linear(hidden_size, 256), nn.ReLU(), nn.Linear(256, 128), nn.ReLU(),
                                        nn.Linear(128, 64), nn.ReLU(), nn.Linear(64, 1))

    def critic_channels(self, state: torch.Tensor) -> torch.Tensor:
        """(…, S) flattened state -> (…, 4, R) channel stack in the reference's order (lstm_value_net.py:124-137)."""
        R = self.length
        return torch.stack([state[..., 3 * R:4 * R], state[..., 2 * R:3 * R], state[..., R:2 * R], state[..., :R]], dim=-2)

    def forward(self, state: torch.Tensor, hc, reset: Optional[torch.Tensor] = None):
        """``state``: the flattened ``env.state()`` (B, L, S), or the 4-channel ray block the step kernel emits
        directly (``env.critic()``, (B, L, 4 R) — the same numbers, no stack copy: SURVEY.md f-3)."""
        B, L, S = state.shape
        ch = state if S == 4 * self.length else self.critic_channels(state)
        f = self.features_extractor(ch.reshape(B * L, 4, self.length)).view(B, L, -1)
        out, hc = self.run_lstm(f, hc, reset)
        return self.value_head(out).squeeze(-1), hc


class PolicyNet(nn.Module):
    """``Policy`` (policy_net.py:17-33): the same ray CNN -> 256 -> 128 -> 64 -> 4 logits, no memory."""

    recurrent = False

    def __init__(self, n_obs: int = 2 * N_RAYS, n_actions: int = 4):
        super().__init__()
        self.len_ch = n_obs // 2
        self.features_extractor = _ray_features(2, self.len_ch)
        self.net = nn.Sequential(nn.Linear(256, 128), nn.ReLU(), nn.Linear(128, 64), nn.ReLU(), nn.Linear(64, n_actions))

    def forward(self, obs: torch.Tensor, hc=None, reset=None):
        B, L, _ = obs.shape
        return self.net(self.features_extractor(obs.reshape(B * L, 2, self.len_ch))).view(B, L, -1), hc

    def initial_state(self, batch: int, device):
        return None


class ValueNet(nn.Module):
    """``Value`` (value_net.py:18-28): MLP S -> 512 -> 256 -> 128 -> 64 -> 1 on the whole flattened state."""

    recurrent = False

    def __init__(self, n_state: int = 1090):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(n_state, 512), nn.ReLU(), nn.Linear(512, 256), nn.ReLU(),
                                 nn.Linear(256, 128), nn.ReLU(), nn.Linear(128, 64), nn.ReLU(), nn.Linear(64, 1))

    def forward(self, state: torch.Tensor, hc=None, reset=None):
        return self.net(state).squeeze(-1), hc

    def initial_state(self, batch: int, device):
        return None


def n_parameters(module: nn.Module) -> int:
    return sum(p.numel() for p in module.parameters())


# ------------------------------------------------------------------ configuration
@dataclass
class MAPPOConfig:
    """``CFG_AGENT`` of the reference (mappo_config.py:5-50) + the skrl defaults it leaves untouched."""
    rollouts: int = 64                 # lockstep steps per update (reference: 4096 steps of ONE environment)
    learning_epochs: int = 4           # :44
    mini_batches: int = 4              # :45
    discount_factor: float = 0.99      # skrl default
    lambda_: float = 0.95              # skrl default
    learning_rate: float = 1e-4        # :47
    ratio_clip: float = 0.15           # :48
    entropy_loss_scale: float = 0.02   # :46
    value_loss_scale: float = 0.5      # :13
    grad_norm_clip: float = 0.5        # :14
    kl_threshold: float = 0.015        # :11
    random_timesteps: int = 10000      # :9 uniform random actions first
    learning_starts: int = 15000       # :10 no update before this many (lockstep) timesteps
    # CFG_TRAINER (:61-62) + the reference's skrl patch (README.md:78-152): train() starts with every policy frozen and
    # every value net trainable (agent_learning_utils.py:192-194); all value nets are (re-)unfrozen at
    # opponent_freeze_duration and all policies at policy_freeze_duration.  0 = nothing is frozen.
    opponent_freeze_duration: int = 15000
    policy_freeze_duration: int = 15000
    model: str = "lstm"                # "lstm" (self_play_driver.py via initialize_lstm_models_for_mappo) | "mlp"
    sequence_length: int = 16          # lstm_policy_net.py:16
    cuda_graph: bool = True            # replay the whole rollout (nets + env kernels) as one CUDA graph
    # skrl's time_limit_bootstrap: a truncated (timed-out) transition stores rew + discount_factor * V(s_final), V from
    # each agent's critic on the episode's final observation (needs BatchedCopsThievesEnv(final_observations=True))
    time_limit_bootstrap: bool = False
    update_autocast: str = "none"      # "bf16": run the PPO update's forward / backward under torch.autocast (the
                                       # reference trains in fp32, so this is off by default; ~2x faster updates)
    distributed: bool = False          # all-reduce gradients (and advantage statistics) across ranks
    world_size: int = 1


@dataclass
class UpdateStats:
    policy_loss: float = 0.0
    value_loss: float = 0.0
    entropy: float = 0.0
    kl: float = 0.0
    minibatches: int = 0
    gae_ms: float = 0.0
    allreduce_ms: float = 0.0
    update_ms: float = 0.0
    allreduce_events: Optional[list] = None


def ppo_losses(logits: torch.Tensor, actions: torch.Tensor, old_log_prob: torch.Tensor, advantages: torch.Tensor,
               values: torch.Tensor, returns: torch.Tensor, cfg: MAPPOConfig):
    """The loss terms of skrl's ``MAPPO._update`` for one minibatch plus the approximate KL it uses for early
    stopping.  Pure function of tensors (unit-tested on CPU)."""
    dist = torch.distributions.Categorical(logits=logits)
    new_log_prob = dist.log_prob(actions)
    log_ratio = new_log_prob - old_log_prob
    kl = ((torch.exp(log_ratio) - 1.0) - log_ratio).mean()
    ratio = torch.exp(log_ratio)
    surrogate = advantages * ratio
    clipped = advantages * torch.clip(ratio, 1.0 - cfg.ratio_clip, 1.0 + cfg.ratio_clip)
    policy_loss = -torch.min(surrogate, clipped).mean()
    entropy = dist.entropy().mean()
    entropy_loss = -cfg.entropy_loss_scale * entropy
    value_loss = cfg.value_loss_scale * torch.nn.functional.mse_loss(values, returns)
    return policy_loss, entropy_loss, value_loss, kl, entropy


def build_models(agents: Iterable[str], n_obs: int, n_state: int, kind: str, device) -> Dict[str, Dict[str, nn.Module]]:
    """``initialize_lstm_models_for_mappo`` / ``initialize_models_for_mappo`` (utils/model_utils.py:44-120)."""
    out = {}
    for a in agents:
        if kind == "lstm":
            out[a] = {"policy": LSTMPolicyNet(n_obs).to(device), "value": LSTMValueNet(n_state).to(device)}
        elif kind == "mlp":
            out[a] = {"policy": PolicyNet(n_obs).to(device), "value": ValueNet(n_state).to(device)}
        else:
            raise ValueError(f"unknown model kind {kind!r}")
    return out


# ------------------------------------------------------------------ the learner
class MAPPOLearner:
    """Collect ``rollouts`` lockstep steps with the current policies, then one MAPPO update per agent.

    Agents that the environment scripts in every world (``BatchedCopsThievesEnv(scripted=...)``) are played by the step
    kernel's controllers: the learner gives them no models, no memory and no update, and ``agents`` lists only the
    learned ones.  An agent scripted in some worlds but not all is refused, and so is a rollout after the set of scripted
    agents has changed."""

    def __init__(self, env, cfg: Optional[MAPPOConfig] = None, seed: int = 0):
        self.env = env
        self.cfg = cfg or MAPPOConfig()
        self.device = env.device
        self._scripts = self._script_signature()
        partial = [a for a, where in zip(env.possible_agents, self._scripts) if where == "some"]
        if partial:
            raise ValueError(f"agents {partial} are scripted in some worlds but not all: a learner needs each agent "
                             "either scripted everywhere or nowhere")
        self.scripted_agents: List[str] = [a for a, where in zip(env.possible_agents, self._scripts) if where == "all"]
        self.agents: List[str] = [a for a in env.possible_agents if a not in self.scripted_agents]
        if not self.agents:
            raise ValueError("every agent is scripted: there is nothing to learn")
        self.n_obs = 2 * env.worlds.R
        self.n_state = env.state_dim
        if self.cfg.rollouts % self.cfg.sequence_length:
            raise ValueError("rollouts must be a multiple of sequence_length")
        torch.manual_seed(seed)     # identical initial weights on every rank
        self.models = build_models(self.agents, self.n_obs, self.n_state, self.cfg.model, self.device)
        # fused Adam: its step can be switched off by a device-side flag (the KL early stop below) without a host sync
        self.optimizers = {a: torch.optim.Adam(self.parameters(a), lr=self.cfg.learning_rate, fused=True) for a in self.agents}
        self.frozen: Dict[str, Dict[str, bool]] = {a: {"policy": False, "value": False} for a in self.agents}
        # One flat fp32 gradient bucket per agent; every parameter's .grad is a view into it, so the minibatch
        # all-reduce is a single NCCL call on memory autograd already wrote — no gather / scatter copies.
        self._flat_grad: Dict[str, torch.Tensor] = {}
        for a in self.agents:
            ps = self.parameters(a)
            flat = torch.zeros(sum(p.numel() for p in ps), device=self.device)
            off = 0
            for p in ps:
                p.grad = flat[off:off + p.numel()].view_as(p)
                off += p.numel()
            self._flat_grad[a] = flat
        T, N, dev = self.cfg.rollouts, env.num_envs, self.device
        nseg = T // self.cfg.sequence_length
        self.mem = {}
        for a in self.agents:
            m = dict(obs=torch.zeros((T, N, self.n_obs), device=dev), act=torch.zeros((T, N), dtype=torch.int64, device=dev),
                     logp=torch.zeros((T, N), device=dev), rew=torch.zeros((T, N), device=dev),
                     val=torch.zeros((T, N), device=dev))
            for role in ("policy", "value"):
                net = self.models[a][role]
                if net.recurrent:   # hidden state at the start of every training sequence
                    shape = (nseg, net.lstm.num_layers, N, net.lstm.hidden_size)
                    m[role + "_h"] = torch.zeros(shape, device=dev)
                    m[role + "_c"] = torch.zeros(shape, device=dev)
            self.mem[a] = m
        # the LSTM critic reads only the 4-channel ray block of the first agent (SURVEY.md C-8): take it straight from the
        # step kernel (env.critic()) instead of storing / slicing / stacking the 1090-float state
        self.critic_block = self.cfg.model == "lstm" and getattr(env, "critic", None) is not None and env.critic() is not None
        self.n_value_in = 4 * env.worlds.R if self.critic_block else self.n_state
        if self.cfg.time_limit_bootstrap:
            final = getattr(env, "final_critic" if self.critic_block else "final_state", None)
            if final is None or final() is None:
                raise ValueError("time_limit_bootstrap needs an environment that keeps final observations "
                                 "(BatchedCopsThievesEnv(..., final_observations=True))")
        self._no_reset = torch.zeros((N, 1), dtype=torch.bool, device=dev)
        self.mem_state = torch.zeros((T, N, self.n_value_in), device=dev)
        self.mem_done = torch.zeros((T, N), dtype=torch.bool, device=dev)
        self.mem_reset = torch.zeros((T, N), dtype=torch.bool, device=dev)   # episode of world n ended just before step t
        self._obs = None
        self._hc = {a: {r: self.models[a][r].initial_state(N, dev) for r in ("policy", "value")} for a in self.agents}
        self._prev_done = torch.zeros(N, dtype=torch.bool, device=dev)
        self._act = {a: torch.zeros(N, dtype=torch.int64, device=dev) for a in self.agents}   # static action buffers
        self._graphs: Dict[bool, object] = {}
        self.timestep = 0
        self.env_seconds = 0.0

    def _script_signature(self) -> Tuple[str, ...]:
        """Per agent, where the environment scripts it ("all", "none" or "some"), from the host mirror of the modes."""
        where = getattr(self.env, "scripted_in", None)
        return tuple(where(a) if where is not None else "none" for a in self.env.possible_agents)

    # -------------------------------------------------------------- parameters / checkpoints
    def parameters(self, agent: str) -> List[nn.Parameter]:
        return list(itertools.chain(self.models[agent]["policy"].parameters(), self.models[agent]["value"].parameters()))

    def n_parameters(self) -> int:
        return sum(p.numel() for a in self.agents for p in self.parameters(a))

    def freeze(self, agent: str, role: str, frozen: bool = True) -> None:
        """``Model.freeze_parameters`` (agent_learning_utils.py:192-194): frozen nets get no optimiser step."""
        self.frozen[agent][role] = frozen
        for p in self.models[agent][role].parameters():
            p.requires_grad_(not frozen)
        self._rebind_grads(agent)

    def _rebind_grads(self, agent: str) -> None:
        """Frozen parameters get no gradient (Adam then skips them: no momentum drift while frozen); trainable
        ones (re)attach to their slice of the agent's flat bucket."""
        flat, off = self._flat_grad[agent], 0
        for role in ("policy", "value"):
            for p in self.models[agent][role].parameters():
                n = p.numel()
                if self.frozen[agent][role]:
                    p.grad = None
                else:
                    flat[off:off + n].zero_()
                    p.grad = flat[off:off + n].view_as(p)
                off += n

    def state_dict(self) -> Dict[str, Dict[str, dict]]:
        """What ``agent.save`` writes (orchestration.py:225-228): per agent policy / value / optimizer."""
        return {a: {"policy": self.models[a]["policy"].state_dict(), "value": self.models[a]["value"].state_dict(),
                    "optimizer": self.optimizers[a].state_dict()} for a in self.agents}

    def load_state_dict(self, sd: Dict[str, Dict[str, dict]], role_prefix: Optional[str] = None) -> None:
        """Load every agent, or only the agents of one role (``copy_role_models``, utils/model_utils.py:10-41)."""
        for a in self.agents:
            if role_prefix is not None and not a.startswith(role_prefix):
                continue
            if a not in sd:
                continue
            self.models[a]["policy"].load_state_dict(sd[a]["policy"])
            self.models[a]["value"].load_state_dict(sd[a]["value"])
            if role_prefix is None and "optimizer" in sd[a]:
                self.optimizers[a].load_state_dict(sd[a]["optimizer"])

    def save(self, path: str) -> None:
        torch.save(self.state_dict(), path)

    def load(self, path: str, role_prefix: Optional[str] = None) -> None:
        self.load_state_dict(torch.load(path, map_location=self.device), role_prefix)

    # -------------------------------------------------------------- acting
    @torch.no_grad()
    def act(self, obs: Dict[str, torch.Tensor], greedy: bool = False) -> Dict[str, torch.Tensor]:
        """Sampled (or arg-max) actions for every agent from the current observations, advancing the recurrent
        state the learner carries per world (used by the evaluator)."""
        out = {}
        reset = self._prev_done.view(-1, 1)
        for a in self.agents:
            pol = self.models[a]["policy"]
            logits, hc = pol(obs[a].unsqueeze(1), self._hc[a]["policy"], reset)
            if pol.recurrent:
                self._hc[a]["policy"][0].copy_(hc[0]); self._hc[a]["policy"][1].copy_(hc[1])
            logits = logits.squeeze(1)
            out[a] = logits.argmax(-1) if greedy else self._sample(logits, False)[0]
        return out

    def note_done(self, done: torch.Tensor) -> None:
        self._prev_done.copy_(done.view(-1).bool())

    def note_reset(self, mask: torch.Tensor) -> None:
        """Worlds reset outside the rollout (``BatchedCopsThievesEnv.set_map`` returns their (N,) mask): their
        recurrent states are zeroed at the next step, as after an episode end.  In place, so a captured rollout graph
        stays valid and is not recaptured."""
        self._prev_done.logical_or_(mask.to(device=self._prev_done.device).view(-1).bool())

    def reset_recurrent_state(self) -> None:
        """Zero every carried (h, c) and the done flags IN PLACE (the rollout graph holds these buffers)."""
        for a in self.agents:
            for r in ("policy", "value"):
                if self._hc[a][r] is not None:
                    self._hc[a][r][0].zero_(); self._hc[a][r][1].zero_()
        self._prev_done.zero_()

    # -------------------------------------------------------------- rollout
    @staticmethod
    def _sample(logits: torch.Tensor, uniform_random: bool):
        """Categorical sample by the Gumbel-max trick + its log-probability: sync-free and graph-capturable
        (``torch.distributions.Categorical`` validates its arguments with a host round trip)."""
        logp_all = torch.log_softmax(logits, dim=-1)
        if uniform_random:
            act = torch.randint(0, logits.shape[-1], logits.shape[:-1], device=logits.device)
        else:
            u = torch.rand_like(logits).clamp_(1e-20, 1.0)
            act = (logp_all - torch.log(-torch.log(u))).argmax(dim=-1)
        return act, logp_all.gather(-1, act.unsqueeze(-1)).squeeze(-1)

    @torch.no_grad()
    def _rollout_body(self, uniform_random: bool) -> None:
        """``rollouts`` lockstep transitions on static buffers only (no host syncs, no allocations that outlive
        the call): SequentialTrainer.train's inner loop — act -> env.step -> env.state -> record_transition.
        Done worlds are re-spawned inside the step kernel (SURVEY.md C-10).  With ``time_limit_bootstrap`` each critic
        also evaluates the final value input of the step from the hidden state it carries, without advancing that state,
        and a truncated world's stored reward becomes ``rew + discount_factor * V_final``."""
        env, cfg = self.env, self.cfg
        L = cfg.sequence_length
        obs_bufs = env._obs_dict()                 # views of the environment's persistent output buffers
        for t in range(cfg.rollouts):
            state = self._value_input()
            self.mem_state[t].copy_(state)
            self.mem_reset[t].copy_(self._prev_done)
            reset = self._prev_done.view(-1, 1)
            for a in self.agents:
                m, o = self.mem[a], obs_bufs[a]
                m["obs"][t].copy_(o)
                pol, val = self.models[a]["policy"], self.models[a]["value"]
                if t % L == 0:
                    keep = (~self._prev_done).float().view(1, -1, 1)   # the stored state is the one actually used
                    for role, net in (("policy", pol), ("value", val)):
                        if net.recurrent:
                            torch.mul(self._hc[a][role][0], keep, out=m[role + "_h"][t // L])
                            torch.mul(self._hc[a][role][1], keep, out=m[role + "_c"][t // L])
                logits, hc = pol(o.unsqueeze(1), self._hc[a]["policy"], reset)
                if pol.recurrent:
                    self._hc[a]["policy"][0].copy_(hc[0]); self._hc[a]["policy"][1].copy_(hc[1])
                act, logp = self._sample(logits.squeeze(1), uniform_random)
                self._act[a].copy_(act)
                m["act"][t].copy_(act)
                m["logp"][t].copy_(logp)
                v, hc = val(state.unsqueeze(1), self._hc[a]["value"], reset)
                if val.recurrent:
                    self._hc[a]["value"][0].copy_(hc[0]); self._hc[a]["value"][1].copy_(hc[1])
                m["val"][t].copy_(v.view(-1))
            _, rew, term, trunc, _ = env.step(self._act)
            if cfg.time_limit_bootstrap:
                final = self._final_value_input().unsqueeze(1)
                truncated = trunc[self.agents[0]].view(-1).float()
            for a in self.agents:
                if cfg.time_limit_bootstrap:
                    v_final, _ = self.models[a]["value"](final, self._hc[a]["value"], self._no_reset)
                    torch.addcmul(rew[a].view(-1), v_final.view(-1), truncated, value=cfg.discount_factor,
                                  out=self.mem[a]["rew"][t])
                else:
                    self.mem[a]["rew"][t].copy_(rew[a].view(-1))
            done = (term[self.agents[0]] | trunc[self.agents[0]]).view(-1)
            self.mem_done[t].copy_(done)
            self._prev_done.copy_(done)

    def _value_input(self) -> torch.Tensor:
        """What the critics read: the kernel's (N, 4, R) block viewed as (N, 4 R), or the flattened state (N, S)."""
        return self.env.critic().view(self.env.num_envs, -1) if self.critic_block else self.env.state()

    def _final_value_input(self) -> torch.Tensor:
        """``_value_input`` of the last step of the episodes that ended in the step just taken (valid where done)."""
        return self.env.final_critic().view(self.env.num_envs, -1) if self.critic_block else self.env.final_state()

    def collect(self) -> None:
        """One rollout.  The first call per mode runs eagerly (warm-up: cuDNN plans, allocator); later calls
        replay ONE CUDA graph holding every network launch and every environment-step launch of the rollout,
        so the host issues a single graph launch instead of ~10^4 kernel launches."""
        env, cfg = self.env, self.cfg
        if self._script_signature() != self._scripts:
            raise RuntimeError("the environment's scripted agents changed since this learner was built (it learns "
                               f"{self.agents}); build a new learner for the new set")
        if self._obs is None:
            self._obs, _ = env.reset()
        uniform = self.timestep < cfg.random_timesteps
        t0 = time.perf_counter()
        if not cfg.cuda_graph:
            self._rollout_body(uniform)
        else:
            entry = self._graphs.get(uniform)
            if entry is None:                       # warm-up pass, eager, real
                self._rollout_body(uniform)
                self._graphs[uniform] = "warm"
            else:
                if entry == "warm":
                    torch.cuda.synchronize(self.device)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._rollout_body(uniform)
                    self._graphs[uniform] = entry = g
                entry.replay()
        torch.cuda.synchronize(self.device)
        self.timestep += cfg.rollouts
        self.env_seconds += time.perf_counter() - t0

    # -------------------------------------------------------------- update
    def _sequences(self, x: torch.Tensor) -> torch.Tensor:
        """(T, N, ...) -> (T/L * N, L, ...): one row per (segment, world) training sequence."""
        L = self.cfg.sequence_length
        T, N = x.shape[:2]
        x = x.view(T // L, L, N, *x.shape[2:]).transpose(1, 2)
        return x.reshape(T // L * N, L, *x.shape[3:])

    def _hidden(self, m: dict, role: str, idx: torch.Tensor):
        if role + "_h" not in m:
            return None
        h, c = m[role + "_h"], m[role + "_c"]            # (nseg, layers, N, H) -> (layers, nseg * N, H)
        h = h.permute(1, 0, 2, 3).reshape(h.shape[1], -1, h.shape[3])
        c = c.permute(1, 0, 2, 3).reshape(c.shape[1], -1, c.shape[3])
        return h[:, idx].contiguous(), c[:, idx].contiguous()

    def update(self) -> Dict[str, UpdateStats]:
        """skrl ``MAPPO._update`` per agent: last values -> GAE (CUDA) -> epochs x minibatches of PPO."""
        from .gae import compute_gae
        cfg = self.cfg
        stats: Dict[str, UpdateStats] = {}
        if self.timestep < cfg.learning_starts:
            return stats
        N = self.env.num_envs
        last_state = self._value_input()
        for a in self.agents:
            if self.frozen[a]["policy"] and self.frozen[a]["value"]:
                continue
            st = UpdateStats()
            cuda = self.device.type == "cuda"
            ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3)) if cuda else (None, None, None)
            if cuda:
                ev0.record()
            mem = self.mem[a]
            pol, val = self.models[a]["policy"], self.models[a]["value"]
            with torch.no_grad():
                lv, _ = val(last_state.unsqueeze(1), self._hc[a]["value"], self._prev_done.view(-1, 1))
                last_values = lv.view(-1)
            returns, advantages = compute_gae(mem["rew"], self.mem_done, mem["val"], last_values, cfg.discount_factor,
                                              cfg.lambda_, normalize=True, distributed=cfg.distributed)
            if cuda:
                ev1.record()
            self._ppo_update(a, returns, advantages, st)
            if cuda:
                ev2.record()
                ev2.synchronize()
                st.gae_ms, st.update_ms = ev0.elapsed_time(ev1), ev1.elapsed_time(ev2)
                st.allreduce_ms = sum(e0.elapsed_time(e1) for e0, e1 in st.allreduce_events)
            st.allreduce_events = None
            stats[a] = st
        return stats

    def _ppo_update(self, a: str, returns: torch.Tensor, advantages: torch.Tensor, st: UpdateStats) -> UpdateStats:
        """The epochs x minibatches of skrl's ``MAPPO._update`` for agent ``a`` on the recorded rollout (pure PyTorch;
        under ``distributed`` every rank issues the same sequence of collectives whatever its data says)."""
        cfg, dev = self.cfg, self.device
        thr = float(cfg.kl_threshold or 0.0)
        mem = self.mem[a]
        pol, val = self.models[a]["policy"], self.models[a]["value"]
        reset_seq = self._sequences(self.mem_reset)
        state_seq = self._sequences(self.mem_state)
        n_seq = reset_seq.shape[0]
        obs_seq = self._sequences(mem["obs"])
        act_seq, logp_seq = self._sequences(mem["act"]), self._sequences(mem["logp"])
        ret_seq, adv_seq = self._sequences(returns), self._sequences(advantages)
        params = [p for p in self.parameters(a) if p.requires_grad]
        ar_events = []
        opt = self.optimizers[a]
        # skrl's KL early stop ("break" out of the epoch's minibatch loop) as a DEVICE-side, COLLECTIVE decision:
        # the KL is all-reduced (MAX) so that every rank stops at the same minibatch, the sticky flag switches the
        # fused Adam step off for the rest of the epoch, and every rank still issues the same sequence of
        # collectives (a rank-local `break` would pair its gradient all-reduce with another rank's next bucket).
        # No host round trip per minibatch; the skipped minibatches still run forward / backward.
        stop = torch.zeros((), device=dev)
        applied = torch.zeros((), device=dev)
        last = None
        for _epoch in range(cfg.learning_epochs):
            stop.zero_()
            perm = torch.randperm(n_seq, device=self.device)
            for idx in perm.chunk(cfg.mini_batches):
                rs = reset_seq[idx]
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=cfg.update_autocast == "bf16" and dev.type == "cuda"):
                    logits, _ = pol(obs_seq[idx], self._hidden(mem, "policy", idx), rs)
                    values, _ = val(state_seq[idx], self._hidden(mem, "value", idx), rs)
                logits, values = logits.float(), values.float()
                pl, el, vl, kl, ent = ppo_losses(logits.reshape(-1, logits.shape[-1]), act_seq[idx].reshape(-1),
                                                 logp_seq[idx].reshape(-1), adv_seq[idx].reshape(-1),
                                                 values.reshape(-1), ret_seq[idx].reshape(-1), cfg)
                if thr > 0.0:
                    klc = kl.detach().clone()
                    if cfg.distributed:
                        import torch.distributed as dist
                        dist.all_reduce(klc, op=dist.ReduceOp.MAX)
                    stop = torch.maximum(stop, (klc > thr).to(stop.dtype))
                loss = vl if self.frozen[a]["policy"] else (pl + el + vl if not self.frozen[a]["value"] else pl + el)
                opt.zero_grad(set_to_none=False)
                loss.backward()
                if cfg.distributed:
                    import torch.distributed as dist
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    if dev.type == "cuda":
                        e0.record()
                    dist.all_reduce(self._flat_grad[a])          # frozen slices are zero on every rank
                    self._flat_grad[a].div_(cfg.world_size)
                    if dev.type == "cuda":
                        e1.record()
                        ar_events.append((e0, e1))
                if cfg.grad_norm_clip > 0:
                    nn.utils.clip_grad_norm_(params, cfg.grad_norm_clip)
                opt.found_inf = stop                 # fused Adam: a non-zero flag makes this step a no-op, on the device
                opt.step()
                applied += 1.0 - stop
                last = (pl.detach(), vl.detach(), ent.detach(), kl.detach())
        opt.found_inf = None
        st.policy_loss, st.value_loss, st.entropy, st.kl = (float(x) for x in last)   # the update's only host reads
        st.minibatches = int(applied)
        st.allreduce_events = ar_events
        return st

    def train(self, timesteps: int, callback=None) -> List[Dict[str, UpdateStats]]:
        """``SequentialTrainer.train()``: alternate rollout and update until ``timesteps`` lockstep steps."""
        history = []
        cfg = self.cfg
        if cfg.policy_freeze_duration > 0 or cfg.opponent_freeze_duration > 0:
            # train_simultaneously_and_evaluate (agent_learning_utils.py:188-194): every policy frozen, every value
            # net trainable at the start of a training run
            for a in self.agents:
                self.freeze(a, "policy", cfg.policy_freeze_duration > 0)
                self.freeze(a, "value", False)
        start = self.timestep
        while self.timestep < timesteps:
            before = self.timestep - start
            self.collect()
            now = self.timestep - start
            # the reference's skrl patch (README.md:100-152): at `timestep == duration` unfreeze ALL value / policy nets
            if cfg.opponent_freeze_duration > 0 and before < cfg.opponent_freeze_duration <= now:
                for a in self.agents:
                    self.freeze(a, "value", False)
            if cfg.policy_freeze_duration > 0 and before < cfg.policy_freeze_duration <= now:
                for a in self.agents:
                    self.freeze(a, "policy", False)
            s = self.update()
            history.append(s)
            if callback is not None:
                callback(self, s)
        return history
