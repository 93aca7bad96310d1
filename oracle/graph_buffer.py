"""numpy float32 restatement of the reference's training input (TEST INFRASTRUCTURE ONLY):

* ``GraphReplayBuffer.compute_returns`` (onpolicy/utils/graph_buffer.py:285-366), every branch;
* ``ValueNorm`` (onpolicy/utils/valuenorm.py: beta 0.99999, epsilon 1e-5, variance clamped at 1e-2);
* the advantage lines of ``GR_MAPPO.train`` (onpolicy/algorithms/graph_mappo.py:280-300);
* the buffer's three mini-batch generators, given the epoch's permutation (the reference draws it with
  ``torch.randperm``).

Arrays are in the reference's layout: ``[T(+1), B, N, ...]``, with ``share_obs``, ``share_agent_id`` and ``adj`` stored
per agent.  Every arithmetic line keeps the reference's operation order; numpy >= 2 keeps float32 arrays float32 when a
Python float multiplies them (NEP 50), as torch does.
"""
from __future__ import annotations

import warnings

import numpy as np

# the order in which GR_MAPPO.ppo_update unpacks a mini-batch
SAMPLE_FIELDS = ("share_obs", "obs", "node_obs", "adj", "agent_id", "share_agent_id", "rnn_states", "rnn_states_critic",
                 "actions", "value_preds", "returns", "masks", "active_masks", "old_action_log_probs", "adv_targ",
                 "available_actions")


class ValueNorm:
    """valuenorm.py ValueNorm(input_shape=1) in float32 (norm_axes 1, per_element_update False)."""

    def __init__(self, beta: float = 0.99999, epsilon: float = 1e-5):
        self.beta, self.epsilon = beta, epsilon
        self.running_mean = np.zeros(1, np.float32)
        self.running_mean_sq = np.zeros(1, np.float32)
        self.debiasing_term = np.zeros((), np.float32)

    def running_mean_var(self):
        d = np.maximum(self.debiasing_term, np.float32(self.epsilon))
        mean, mean_sq = self.running_mean / d, self.running_mean_sq / d
        return mean, np.maximum(mean_sq - mean ** 2, np.float32(1e-2))

    def update(self, x: np.ndarray) -> None:
        x = np.asarray(x, np.float32)
        w = self.beta
        self.running_mean = self.running_mean * w + x.mean(axis=0) * np.float32(1.0 - w)
        self.running_mean_sq = self.running_mean_sq * w + (x ** 2).mean(axis=0) * np.float32(1.0 - w)
        self.debiasing_term = self.debiasing_term * w + np.float32(1.0 * (1.0 - w))

    def denormalize(self, x: np.ndarray) -> np.ndarray:
        mean, var = self.running_mean_var()
        return np.asarray(x, np.float32) * np.sqrt(var) + mean


def compute_returns(buf: dict, next_value: np.ndarray, value_normalizer=None, *, use_gae: bool = True,
                    use_proper_time_limits: bool = False, gamma: float = 0.99, gae_lambda: float = 0.95) -> np.ndarray:
    """Writes buf['value_preds'][-1] (GAE) or buf['returns'][-1], then buf['returns'][:T]; returns buf['returns']."""
    v, r, m, bad, ret = buf["value_preds"], buf["rewards"], buf["masks"], buf["bad_masks"], buf["returns"]
    dn = (lambda x: x) if value_normalizer is None else value_normalizer.denormalize
    T = r.shape[0]
    if use_proper_time_limits:
        if use_gae:
            v[-1] = next_value
            gae = 0
            for step in reversed(range(T)):
                delta = r[step] + gamma * dn(v[step + 1]) * m[step + 1] - dn(v[step])
                gae = delta + gamma * gae_lambda * m[step + 1] * gae
                gae = gae * bad[step + 1]
                ret[step] = gae + dn(v[step])
        else:
            ret[-1] = next_value
            for step in reversed(range(T)):
                ret[step] = (ret[step + 1] * gamma * m[step + 1] + r[step]) * bad[step + 1] + (1 - bad[step + 1]) * dn(v[step])
    else:
        if use_gae:
            v[-1] = next_value
            gae = 0
            for step in reversed(range(T)):
                delta = r[step] + gamma * dn(v[step + 1]) * m[step + 1] - dn(v[step])
                gae = delta + gamma * gae_lambda * m[step + 1] * gae
                ret[step] = gae + dn(v[step])
        else:
            ret[-1] = next_value
            for step in reversed(range(T)):
                ret[step] = ret[step + 1] * gamma * m[step + 1] + r[step]        # no denormalisation in this branch
    return ret


def raw_advantages(buf: dict, value_normalizer=None) -> np.ndarray:
    if value_normalizer is not None:
        return buf["returns"][:-1] - value_normalizer.denormalize(buf["value_preds"][:-1])
    return buf["returns"][:-1] - buf["value_preds"][:-1]


def normalise_advantages(adv: np.ndarray, mean, std) -> np.ndarray:
    """(advantages - mean_advantages) / (std_advantages + 1e-5) with float32 scalars."""
    return (adv - np.float32(mean)) / (np.float32(std) + 1e-5)


def advantages(buf: dict, value_normalizer=None):
    """-> (normalised advantages [T, B, N, 1], nanmean, nanstd) as GR_MAPPO.train computes them."""
    adv = raw_advantages(buf, value_normalizer)
    cp = adv.copy()
    cp[buf["active_masks"][:-1] == 0.0] = np.nan
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)          # all inactive: NaN, as in the reference
        mean, std = np.nanmean(cp), np.nanstd(cp)
    return normalise_advantages(adv, mean, std), mean, std


def _sources(buf: dict, advantages_: np.ndarray):
    """The per-sample arrays of a generator, [T, B, N, ...] each (slabs 0..T-1)."""
    return {"share_obs": buf["share_obs"][:-1], "obs": buf["obs"][:-1], "node_obs": buf["node_obs"][:-1],
            "adj": buf["adj"][:-1], "agent_id": buf["agent_id"][:-1], "share_agent_id": buf["share_agent_id"][:-1],
            "actions": buf["actions"], "value_preds": buf["value_preds"][:-1], "returns": buf["returns"][:-1],
            "masks": buf["masks"][:-1], "active_masks": buf["active_masks"][:-1],
            "old_action_log_probs": buf["action_log_probs"], "adv_targ": advantages_,
            "available_actions": buf["available_actions"][:-1]}


def feed_forward_batches(buf: dict, advantages_: np.ndarray, perm: np.ndarray, num_mini_batch: int,
                         mini_batch_size=None):
    """feed_forward_generator: samples flat over (t, b, n); mini-batch i is perm[i mbs:(i + 1) mbs]."""
    T, B, N = buf["rewards"].shape[0:3]
    if mini_batch_size is None:
        mini_batch_size = B * T * N // num_mini_batch
    sampler = [perm[i * mini_batch_size:(i + 1) * mini_batch_size] for i in range(num_mini_batch)]
    src = {k: a.reshape(-1, *a.shape[3:]) for k, a in _sources(buf, advantages_).items()}
    src["rnn_states"] = buf["rnn_states"][:-1].reshape(-1, *buf["rnn_states"].shape[3:])
    src["rnn_states_critic"] = buf["rnn_states_critic"][:-1].reshape(-1, *buf["rnn_states_critic"].shape[3:])
    for idx in sampler:
        yield tuple(src[k][idx] for k in SAMPLE_FIELDS)


def _cast(x: np.ndarray) -> np.ndarray:
    """[T, B, N, ...] -> [B N T, ...] (graph_buffer.py _cast)."""
    return x.transpose(1, 2, 0, *range(3, x.ndim)).reshape(-1, *x.shape[3:])


def recurrent_batches(buf: dict, advantages_: np.ndarray, perm: np.ndarray, num_mini_batch: int, data_chunk_length: int):
    """recurrent_generator: chunks of L consecutive rows of the (b, n, t) order; each mini-batch is stacked [L, mbs] and
    flattened; the rnn states of a chunk are those of its first row."""
    T, B, N = buf["rewards"].shape[0:3]
    L = data_chunk_length
    data_chunks = B * T * N // L
    mbs = data_chunks // num_mini_batch
    sampler = [perm[i * mbs:(i + 1) * mbs] for i in range(num_mini_batch)]
    src = {k: _cast(a) for k, a in _sources(buf, advantages_).items()}
    rnn = {k: _cast(buf[k][:-1]) for k in ("rnn_states", "rnn_states_critic")}
    for indices in sampler:
        rows = indices[None, :] * L + np.arange(L)[:, None]          # stack([x[ind * L:(ind + 1) * L] ...], axis=1)
        out = {k: a[rows].reshape(L * mbs, *a.shape[1:]) for k, a in src.items()}
        out.update({k: a[indices * L] for k, a in rnn.items()})
        yield tuple(out[k] for k in SAMPLE_FIELDS)


def naive_recurrent_batches(buf: dict, advantages_: np.ndarray, perm: np.ndarray, num_mini_batch: int):
    """naive_recurrent_generator: whole (env, agent) columns; each mini-batch stacked [T, per] and flattened; rnn states
    of t = 0."""
    T, B, N = buf["rewards"].shape[0:3]
    batch_size = B * N
    per = batch_size // num_mini_batch
    src = {k: a.reshape(T, batch_size, *a.shape[3:]) for k, a in _sources(buf, advantages_).items()}
    rnn = {k: buf[k].reshape(-1, batch_size, *buf[k].shape[3:]) for k in ("rnn_states", "rnn_states_critic")}
    for start in range(0, batch_size, per):
        ind = perm[start:start + per]
        if len(ind) < per:
            raise IndexError("naive_recurrent_generator: B N is not divisible by num_mini_batch")
        out = {k: a[:, ind].reshape(T * per, *a.shape[2:]) for k, a in src.items()}
        out.update({k: a[0, ind] for k, a in rnn.items()})
        yield tuple(out[k] for k in SAMPLE_FIELDS)
