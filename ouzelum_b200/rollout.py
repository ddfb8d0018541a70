"""Rollout collection for the recurrent trainers (BASELINE config 5): env kernels + a torch LSTM policy.

The policy side is deliberately plain PyTorch (a library consumer, like the reference's trainers); what this module
contributes is the collection LOOP of isaacgymenvs/RPO-LSTM/main.py:89-112 without its host round trips:
  * `envs.step` is one kernel launch; the sensor-fault wrapper is one more (ouzelum_b200.pomdp.POMDPWrapper);
  * episode statistics come from the env's metrics vector instead of the O(N) Python scan with `.item()` (main.py:105-110).
`RecurrentActor` has the architecture of isaacgymenvs/RPO-LSTM/model.py:11-68 (MLP 13->512->256 tanh, LSTM 256->128,
mean head 128->4, state-independent log-std, RPO mean perturbation U(-alpha, alpha) at update time) with any num_envs and
device (the reference hard-codes "cuda:0", model.py:65, and reshape(16, 4096), agent.py:61).
"""
import math

import torch
import torch.nn as nn


def _ortho(layer, gain=math.sqrt(2.0)):
    nn.init.orthogonal_(layer.weight, gain)
    nn.init.zeros_(layer.bias)
    return layer


class RecurrentActor(nn.Module):
    def __init__(self, num_obs=13, num_actions=4, rpo_alpha=0.5):
        super().__init__()
        self.rpo_alpha = rpo_alpha
        self.network = nn.Sequential(_ortho(nn.Linear(num_obs, 512)), nn.Tanh(), _ortho(nn.Linear(512, 256)), nn.Tanh())
        self.lstm = nn.LSTM(256, 128)
        for name, p in self.lstm.named_parameters():
            nn.init.zeros_(p) if "bias" in name else nn.init.orthogonal_(p, 1.0)
        self.actor_mean = _ortho(nn.Linear(128, num_actions), gain=0.01)
        self.actor_logstd = nn.Parameter(torch.zeros(1, num_actions))

    def initial_state(self, num_envs, device):
        z = torch.zeros(self.lstm.num_layers, num_envs, self.lstm.hidden_size, device=device)
        return z, z.clone()

    def get_states(self, obs, lstm_state, done):
        """model.py:35-53: MLP, then the LSTM over the leading time axis ([T*B, obs] with B = lstm_state batch), state zeroed
        where `done`.  The cell is written as two GEMMs + pointwise on the nn.LSTM's own parameters: cuDNN's persistent RNN kernel
        needs 8.4 ms for (seq 1, batch 32768, hidden 128) on B200, the GEMM form 0.2 ms (profiles/r01_configs.md)."""
        x = self.network(obs)
        batch = lstm_state[0].shape[1]
        x = x.reshape(-1, batch, self.lstm.input_size)
        done = done.reshape(-1, batch)
        L = self.lstm
        bias = L.bias_ih_l0 + L.bias_hh_l0
        h, c = lstm_state[0][0], lstm_state[1][0]
        out = []
        for xt, dt in zip(x, done):
            keep = (1.0 - dt).view(-1, 1)
            h, c = keep * h, keep * c
            gates = torch.addmm(bias, xt, L.weight_ih_l0.t()).addmm_(h, L.weight_hh_l0.t())
            i, f, g, o = gates.chunk(4, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
            h = torch.sigmoid(o) * torch.tanh(c)
            out.append(h)
        hidden = out[0] if len(out) == 1 else torch.cat(out, 0)
        return hidden, (h.unsqueeze(0), c.unsqueeze(0))

    def distribution(self, obs, lstm_state, done):
        """(action mean, action std, new LSTM state) of the Normal policy (model.py:56-59)."""
        hidden, lstm_state = self.get_states(obs, lstm_state, done)
        mean = self.actor_mean(hidden)
        return mean, torch.exp(self.actor_logstd.expand_as(mean)), lstm_state

    @staticmethod
    def log_prob_entropy(mean, std, action):
        """Normal(mean, std).log_prob(action).sum(1) and .entropy().sum(1) (model.py:67)."""
        logp = (-((action - mean) ** 2) / (2 * std * std) - torch.log(std) - 0.5 * math.log(2 * math.pi)).sum(1)
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(std)).sum(1)
        return logp, ent

    def forward(self, obs, lstm_state, done, action=None):
        """model.py:55-68, same signature and return: (action, log-prob, entropy, lstm_state).  With `action` given (the update
        path) the mean is perturbed by U(-alpha, alpha) -- RPO -- on the module's own device (the reference hard-codes "cuda:0")."""
        mean, std, lstm_state = self.distribution(obs, lstm_state, done)
        if action is None:
            action = mean + std * torch.randn_like(mean)
        else:
            mean = mean + (torch.rand_like(mean) * 2 - 1) * self.rpo_alpha
        logp, ent = self.log_prob_entropy(mean, std, action)
        return action, logp, ent, lstm_state


class RolloutStorage:
    """The buffers of main.py:70-78 for any (rollout_steps, num_envs).  `num_states` > 0 adds `states` [T, N, num_states]: the
    env's obs_dict["states"] (privileged critic input, env.asymmetric_observations) stored next to `obs`."""

    def __init__(self, steps, num_envs, num_obs, num_actions, device, num_states=0):
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=device)
        self.obs, self.pomdps = z(steps, num_envs, num_obs), z(steps, num_envs, num_obs)
        self.actions, self.logprobs = z(steps, num_envs, num_actions), z(steps, num_envs)
        self.rewards, self.dones = z(steps, num_envs), z(steps, num_envs)
        self.states = z(steps, num_envs, num_states) if num_states > 0 else None


@torch.no_grad()
def collect_rollout(env, actor, storage, state, pomdp=None):
    """One `rollout_steps` collection pass (main.py:91-103).  `state` = dict(next_obs, pomdp_obs, next_done, lstm_state)
    carried between calls.  Returns the updated state; env-side episode statistics accumulate in `env.metrics()`."""
    steps = storage.obs.shape[0]
    next_obs, pomdp_obs, next_done, lstm_state = state["next_obs"], state["pomdp_obs"], state["next_done"], state["lstm_state"]
    next_states = state.get("next_states")
    for t in range(steps):
        storage.obs[t], storage.pomdps[t], storage.dones[t] = next_obs, pomdp_obs, next_done
        if storage.states is not None:
            storage.states[t] = next_states
        action, logp, _, lstm_state = actor(pomdp_obs, lstm_state, next_done)
        storage.actions[t], storage.logprobs[t] = action, logp
        obs_dict, rew, done, _ = env.step(action)
        next_obs = obs_dict["obs"]
        if storage.states is not None:
            next_states = obs_dict["states"]
        storage.rewards[t] = rew
        next_done = done.to(torch.float32)
        pomdp_obs = pomdp.observation(next_obs) if pomdp is not None else next_obs
    out = dict(next_obs=next_obs, pomdp_obs=pomdp_obs, next_done=next_done, lstm_state=lstm_state)
    if next_states is not None:
        out["next_states"] = next_states
    return out


def initial_rollout_state(env, actor):
    first = env.reset()
    obs = first["obs"]
    out = dict(next_obs=obs, pomdp_obs=obs.clone(), next_done=torch.zeros(env.num_envs, device=obs.device),
               lstm_state=actor.initial_state(env.num_envs, obs.device))
    if "states" in first:            # a copy: the env's states buffer is overwritten by every step
        out["next_states"] = first["states"].clone()
    return out


class GraphedRollout:
    """One whole `rollout_steps` collection pass -- T x (policy forward, env step, sensor-fault wrapper) -- captured in ONE CUDA
    graph and replayed.  Possible because nothing on the env side takes a host-changing argument: the step kernels, the vehicle
    kernel and the sensor-fault wrapper all follow the env's DEVICE step counter.  SURVEY section 8f rank 1."""

    def __init__(self, env, actor, storage, pomdp=None):
        self.env, self.actor, self.storage, self.pomdp = env, actor, storage, pomdp
        if pomdp is not None:
            pomdp.follow_step_counter(env)
        self.state = initial_rollout_state(env, actor)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                      # warm-up outside capture (allocator, cuBLAS workspaces, autotune)
            for _ in range(2):
                self._assign(collect_rollout(env, actor, storage, self.state, pomdp))
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._assign(collect_rollout(env, actor, storage, self.state, pomdp))

    def _assign(self, new):
        s = self.state
        s["next_obs"].copy_(new["next_obs"])
        s["pomdp_obs"].copy_(new["pomdp_obs"])
        s["next_done"].copy_(new["next_done"])
        s["lstm_state"][0].copy_(new["lstm_state"][0])
        s["lstm_state"][1].copy_(new["lstm_state"][1])
        if "next_states" in s:
            s["next_states"].copy_(new["next_states"])

    def run(self):
        self.graph.replay()
        return self.storage


def save_actor(actor, tag):
    """Checkpoint file of the reference's trainers: `<tag>_actor` = torch.save(state_dict) (RPO-LSTM/agent.py:136-140)."""
    torch.save(actor.state_dict(), f"{tag}_actor")


def load_actor(actor, tag, map_location=None):
    actor.load_state_dict(torch.load(f"{tag}_actor", map_location=map_location))     # RPO-LSTM/agent.py:142-147
    return actor
