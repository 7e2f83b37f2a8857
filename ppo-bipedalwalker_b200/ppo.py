"""Host-side mirror of the reference's PPO surface over libwalker_b200.

Reference classes mirrored (method names and argument meaning kept; numpy arrays replace Matrix[n,1]):
  PPOAgent       Walker/PPO/PPOAgent.cs:23 ctor, :381 SampleActions, :147 Train(Trajectory), :218 Train(Batch), :192 Save
  NeuralNetwork  Walker/PPO/Network/NeuralNetwork.cs:52 FeedForward, :85 Optimise, :94 Load, :159 Save (via PPOAgent.actor/critic)
  Trajectory     Walker/PPO/Trajectory.cs
The compute (forward, clipped-surrogate gradient, backward, Adam, returns) runs in the CUDA library -- for the reference's
default networks on the tensor-core kernel, for any other network the DSL describes (PPOAgent.cs:96-143: dense widths 1..128,
ReLU / LeakyReLU / TanH, any state / action size) on the any-topology kernel; this file only
parses the network DSL, initialises weights (Xavier, host side like Matrix.FromXavier), shuffles mini-batches and
reads/writes the reference's .weights text format.
"""
from __future__ import annotations

import ctypes as C
import re
from dataclasses import dataclass, field

import numpy as np

from ._lib import ACT, OBS, Hyperparams, WalkerB200Error, check, lib, ptr
from .env import default_hyperparams

DENSE, RELU, LEAKYRELU, TANH = 0, 1, 2, 3
DEFAULT_CRITIC = "Input |64| (LeakyReLU) |1| Output"                         # Hyperparameters.cs:91
DEFAULT_ACTOR = "Input |64| (LeakyReLU) |64| (LeakyReLU) |4| (TanH) Output"  # Hyperparameters.cs:92
_DSL = re.compile(r"^Input( \|\d+\|| \((ReLU|TanH|LeakyReLU)\))+ Output$")   # PPOAgent.cs:98


def ParseLayers(structure: str):
    """PPOAgent.ParseLayers (PPOAgent.cs:96-143) -> [(kind, size)]; raises ValueError like the reference throws."""
    if not _DSL.match(structure):
        raise ValueError(f"The neural network structure '{structure}' is invalid.")
    cleaned = re.sub(r"[\[|()]|( Output)|(Input )", "", structure)
    layers = []
    for token in cleaned.split(" "):
        if token.isdigit():
            layers.append((DENSE, int(token)))
        else:
            layers.append(({"ReLU": RELU, "LeakyReLU": LEAKYRELU, "TanH": TANH}[token], 0))
    return layers


def dense_shapes(input_size: int, layers):
    shapes, width = [], input_size
    for kind, size in layers:
        if kind == DENSE:
            shapes.append((size, width))
            width = size
    return shapes


def xavier_flat(input_size: int, layers, rng: np.random.Generator) -> np.ndarray:
    """Matrix.FromXavier per dense layer (Matrix.cs:59-80): N(0, sqrt(2/(out+in))) by the reference's Box-Muller, zero biases."""
    parts = []
    for out, inp in dense_shapes(input_size, layers):
        std = np.float32(np.sqrt(np.float32(2.0) / np.float32(out + inp)))
        u1 = rng.random((out, inp)).astype(np.float32)
        u2 = rng.random((out, inp)).astype(np.float32)
        u1[u1 == 0] = 1.0
        z = np.sqrt(np.float32(-2.0) * np.log(u1)) * np.sin(np.float32(2.0) * np.float32(np.pi) * u2)
        parts.append((std * z).astype(np.float32).ravel())
        parts.append(np.zeros(out, np.float32))
    return np.concatenate(parts)


def resolve_networks(actor: str, critic: str, actionSize: int):
    """PPOAgent.CreateNetworks' fallbacks (PPOAgent.cs:41-93): a DSL string that does not parse, or whose last dense layer has the
    wrong size (one value / actionSize means), is replaced by the default network.  -> (actor, actor layers, critic, critic layers)"""
    try:
        c_layers = ParseLayers(critic)
    except ValueError:
        critic, c_layers = DEFAULT_CRITIC, ParseLayers(DEFAULT_CRITIC)
    try:
        a_layers = ParseLayers(actor)
    except ValueError:
        actor, a_layers = DEFAULT_ACTOR, ParseLayers(DEFAULT_ACTOR)
    if [s for k, s in c_layers if k == DENSE][-1:] != [1]:
        critic, c_layers = DEFAULT_CRITIC, ParseLayers(DEFAULT_CRITIC)
    if [s for k, s in a_layers if k == DENSE][-1:] != [actionSize]:
        actor, a_layers = DEFAULT_ACTOR, ParseLayers(DEFAULT_ACTOR)
    return actor, a_layers, critic, c_layers


@dataclass
class Trajectory:
    """Walker/PPO/Trajectory.cs (lists of per-step values for ONE episode)."""
    States: list = field(default_factory=list)
    Actions: list = field(default_factory=list)
    LogProbabilities: list = field(default_factory=list)
    Rewards: list = field(default_factory=list)
    Values: list = field(default_factory=list)
    Returns: list = field(default_factory=list)
    Advantages: list = field(default_factory=list)


class _Net:
    """View of one network inside the policy handle (NeuralNetwork surface)."""

    def __init__(self, agent: "PPOAgent", which: int, structure: str, layers):
        self._a, self._which, self.structure, self.layers = agent, which, structure, layers
        n = C.c_int32(0)
        check(lib().wb_policy_num_params(agent._h, which, C.byref(n)))
        self.num_params = n.value
        self.shapes = dense_shapes(agent.stateSize, layers)

    def set_flat(self, flat):
        flat = np.ascontiguousarray(flat, np.float32)
        assert flat.size == self.num_params
        check(lib().wb_policy_set_weights(self._a._h, self._which, ptr(flat)))

    def get_flat(self):
        out = np.empty(self.num_params, np.float32)
        check(lib().wb_policy_get_weights(self._a._h, self._which, ptr(out)))
        return out

    def get_grads(self):
        out = np.empty(self.num_params, np.float32)
        check(lib().wb_policy_get_grads(self._a._h, self._which, ptr(out)))
        return out

    def get_adam(self):
        m = np.empty(self.num_params, np.float32)
        v = np.empty(self.num_params, np.float32)
        it = np.zeros(len(self.shapes), np.int32)
        check(lib().wb_policy_get_adam(self._a._h, self._which, ptr(m), ptr(v), ptr(it)))
        return m, v, it

    def set_adam(self, m, v, it):
        check(lib().wb_policy_set_adam(self._a._h, self._which, ptr(np.ascontiguousarray(m, np.float32)),
                                       ptr(np.ascontiguousarray(v, np.float32)), ptr(np.ascontiguousarray(it, np.int32))))

    def Save(self) -> list[str]:
        return weights_lines(self.structure, self.shapes, self.get_flat())

    # NeuralNetwork.Load / ValidateWeights / DenseLayer.Load / Matrix.Load (NeuralNetwork.cs:94-150, DenseLayer.cs:55-69, Matrix.cs:109-130)
    def Load(self, contents: list[str]) -> bool:
        """Like the reference: the structure line must match, EVERY line is validated (each token parses as a float) before any
        layer is touched, then the dense lines that are present are loaded in order -- a file with fewer lines than layers
        updates the leading layers only; values beyond a layer's size are ignored (Matrix.Load reads height x length of them).
        Where the reference would throw (more lines than layers, too few values in a line) this returns False and loads nothing."""
        if len(contents) < 2 or contents[0] != self.structure:
            return False
        lines = contents[1:]
        if len(lines) > len(self.shapes):
            return False
        parsed = []
        try:
            for line in lines:  # ValidateWeights
                wi, bi = line.index("W") + 2, line.index("B") + 2
                w = [float(tok) for tok in line[wi:bi - 3].split()]
                b = [float(tok) for tok in line[bi:].split()]
                parsed.append((np.array(w, np.float32), np.array(b, np.float32)))
        except ValueError:
            return False
        flat = self.get_flat()
        p = 0
        for (w, b), (out, inp) in zip(parsed, self.shapes):
            if w.size < out * inp or b.size < out:
                return False
            flat[p:p + out * inp] = w[:out * inp]
            p += out * inp
            flat[p:p + out] = b[:out]
            p += out
        self.set_flat(flat)
        return True


# NeuralNetwork.Save / DenseLayer.Save (NeuralNetwork.cs:159-176, DenseLayer.cs:73-79, Matrix.cs:133-153)
def weights_lines(structure: str, shapes, flat) -> list[str]:
    """The lines of a .weights file: the structure line, then "W <weights> B <biases>" per dense layer."""
    lines, p = [structure], 0
    for out, inp in shapes:
        w = flat[p:p + out * inp]
        p += out * inp
        b = flat[p:p + out]
        p += out
        lines.append("W " + " ".join(net_float_str(x) for x in w) + " B " + " ".join(net_float_str(x) for x in b))
    return lines


def net_float_str(x) -> str:
    """float.ToString() of .NET Core 3.0+ (what Matrix.Save joins, Matrix.cs:133-136): the shortest string that round-trips the
    binary32 value; plain decimal notation for 1e-4 <= |x| < 1e7, otherwise d.dddE+XX / d.dddE-XX with at least two exponent digits."""
    v = np.float32(x)
    if np.isnan(v):
        return "NaN"
    if np.isinf(v):
        return "Infinity" if v > 0 else "-Infinity"
    if v == 0:
        return "-0" if np.signbit(v) else "0"
    sci = np.format_float_scientific(v, unique=True, trim="-", exp_digits=2)  # e.g. 1.2345e-06
    mant, exp = sci.split("e")
    e = int(exp)
    if -5 < e < 7:  # the "G" rule: fixed-point iff -5 < exponent < precision (7 for Single)
        return np.format_float_positional(v, unique=True, trim="-")
    return f"{mant}E{'+' if e >= 0 else '-'}{abs(e):02d}"


class PPOAgent:
    """PPOAgent(stateSize, actionSize) (PPOAgent.cs:23-37)."""

    def __init__(self, stateSize: int = OBS, actionSize: int = ACT, hp: Hyperparams | None = None, actor: str = DEFAULT_ACTOR,
                 critic: str = DEFAULT_CRITIC, seed: int | None = None, stream: int | None = None):
        self.stateSize, self.actionSize = stateSize, actionSize
        self.hp = hp if hp is not None else default_hyperparams()
        actor, a_layers, critic, c_layers = resolve_networks(actor, critic, actionSize)
        ak = np.array([k for k, _ in a_layers], np.int32)
        asz = np.array([s for _, s in a_layers], np.int32)
        ck = np.array([k for k, _ in c_layers], np.int32)
        csz = np.array([s for _, s in c_layers], np.int32)
        h = C.c_void_p()
        check(lib().wb_policy_create(stateSize, actionSize, ptr(ak), ptr(asz), len(a_layers), ptr(ck), ptr(csz), len(c_layers),
                                     C.byref(self.hp), C.byref(h)))
        self._h = h
        self.actor = _Net(self, 0, actor, a_layers)
        self.critic = _Net(self, 1, critic, c_layers)
        self.rng = np.random.default_rng(seed)
        self.critic.set_flat(xavier_flat(stateSize, c_layers, self.rng))
        self.actor.set_flat(xavier_flat(stateSize, a_layers, self.rng))
        if stream is not None:
            self.set_stream(stream)

    def close(self):
        if getattr(self, "_h", None) and lib is not None:  # `lib` is None during interpreter shutdown
            lib().wb_policy_destroy(self._h)
            self._h = None

    __del__ = close

    def set_stream(self, cuda_stream: int):
        check(lib().wb_policy_set_stream(self._h, C.c_void_p(cuda_stream)))

    def sync(self):
        check(lib().wb_policy_sync(self._h))

    def set_variant(self, variant: int):
        """0: tcgen05 tensor-core kernel (default); 1: fp32 CUDA-core kernel."""
        check(lib().wb_policy_set_variant(self._h, variant))

    def set_hyperparams(self, hp: Hyperparams):
        self.hp = hp
        check(lib().wb_policy_set_hyperparams(self._h, C.byref(hp)))

    def launch_count(self) -> int:
        out = C.c_int64(0)
        check(lib().wb_policy_launch_count(self._h, C.byref(out)))
        return out.value

    def grad_buffer(self):
        """(device pointer, n_floats) of [actor grads | critic grads | loss sums | skipped] for the all-reduce."""
        p, n = C.c_void_p(), C.c_int32(0)
        check(lib().wb_policy_grad_buffer(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    # -- inference
    def FeedForward(self, states):
        """actor mean [n,act] and critic value [n] (NeuralNetwork.FeedForward for both networks)."""
        s = np.ascontiguousarray(states, np.float32).reshape(-1, self.stateSize)
        mean = np.empty((s.shape[0], self.actionSize), np.float32)
        value = np.empty(s.shape[0], np.float32)
        check(lib().wb_policy_forward(self._h, s.shape[0], ptr(s), ptr(mean), ptr(value)))
        return mean, value

    def SampleActions(self, state, uniforms=None):
        """PPOAgent.SampleActions (PPOAgent.cs:381-398) -> (actions, logProbabilities, mean, std).
        uniforms [n,act,2]: the two System.Random draws of each Box-Muller transform (injected; default: self.rng)."""
        s = np.ascontiguousarray(state, np.float32).reshape(-1, self.stateSize)
        n = s.shape[0]
        if uniforms is None:
            uniforms = self.rng.random((n, self.actionSize, 2))
        u = np.ascontiguousarray(uniforms, np.float32).reshape(n, self.actionSize, 2)
        actions = np.empty((n, self.actionSize), np.float32)
        logp = np.empty((n, self.actionSize), np.float32)
        mean = np.empty((n, self.actionSize), np.float32)
        check(lib().wb_policy_sample(self._h, n, ptr(s), ptr(u), ptr(actions), ptr(logp), ptr(mean)))
        std = np.full((n, self.actionSize), np.exp(np.float32(self.hp.log_std)), np.float32)
        return actions, logp, mean, std

    # -- training
    def _minibatch(self, states, actions, logProbabilities, advantages, returns):
        s = np.ascontiguousarray(states, np.float32).reshape(-1, self.stateSize)
        n = s.shape[0]
        a = np.ascontiguousarray(actions, np.float32).reshape(n, self.actionSize)
        lp = np.ascontiguousarray(logProbabilities, np.float32).reshape(n, self.actionSize)
        adv = np.ascontiguousarray(advantages, np.float32).reshape(n)
        ret = np.ascontiguousarray(returns, np.float32).reshape(n)
        return n, s, a, lp, adv, ret

    def Gradients(self, states, actions, logProbabilities, advantages, returns):
        """Gradient half of PPOAgent.Train(Batch) (PPOAgent.cs:218-342). Returns (criticLoss, actorLoss, skipped)."""
        n, s, a, lp, adv, ret = self._minibatch(states, actions, logProbabilities, advantages, returns)
        losses = np.zeros(2, np.float32)
        skipped = C.c_int32(0)
        check(lib().wb_ppo_grad(self._h, n, ptr(s), ptr(a), ptr(lp), ptr(adv), ptr(ret), ptr(losses), C.byref(skipped)))
        return float(losses[0]), float(losses[1]), skipped.value

    def Optimise(self):  # NeuralNetwork.Optimise on critic and actor (PPOAgent.cs:344-345)
        check(lib().wb_adam_step(self._h))

    def TrainBatch(self, states, actions, logProbabilities, advantages, returns):
        """PPOAgent.Train(Batch) (PPOAgent.cs:218-345): zero, accumulate, Adam -- one call (wb_ppo_train: one launch on the default
        path; page-locked input arrays are read in place). Returns (criticLoss, actorLoss, skipped)."""
        n, s, a, lp, adv, ret = self._minibatch(states, actions, logProbabilities, advantages, returns)
        losses = np.zeros(2, np.float32)
        skipped = C.c_int32(0)
        check(lib().wb_ppo_train(self._h, n, ptr(s), ptr(a), ptr(lp), ptr(adv), ptr(ret), ptr(losses), C.byref(skipped)))
        return float(losses[0]), float(losses[1]), skipped.value

    def CalculateValues(self, trajectory: Trajectory):  # PPOAgent.cs:175-189
        states = np.asarray(trajectory.States, np.float32).reshape(-1, self.stateSize)
        _, values = self.FeedForward(states)
        rewards = np.ascontiguousarray(trajectory.Rewards, np.float32)
        G = np.empty_like(rewards)
        A = np.empty_like(rewards)
        check(lib().wb_returns_advantages(self._h, rewards.size, ptr(rewards), ptr(values), ptr(G), ptr(A)))
        trajectory.Values, trajectory.Returns, trajectory.Advantages = list(values), list(G), list(A)
        return values, G, A

    def Train(self, trajectory: Trajectory, epochs: int = 5):
        """PPOAgent.Train(Trajectory) (PPOAgent.cs:147-172): Epochs x floor(T/B) shuffled mini-batches (remainder dropped)."""
        if len(trajectory.States) == 0:
            return 0.0, 0.0
        self.CalculateValues(trajectory)
        B = self.hp.batch_size
        T = len(trajectory.States)
        S = np.asarray(trajectory.States, np.float32).reshape(T, self.stateSize)
        Acts = np.asarray(trajectory.Actions, np.float32).reshape(T, self.actionSize)
        LP = np.asarray(trajectory.LogProbabilities, np.float32).reshape(T, self.actionSize)
        G = np.asarray(trajectory.Returns, np.float32)
        Adv = np.asarray(trajectory.Advantages, np.float32)
        vloss = aloss = 0.0
        for _ in range(epochs):
            perm = self.rng.permutation(T)  # CreateBatches: sampling without replacement (PPOAgent.cs:501-540)
            for j in range(T // B):
                idx = perm[j * B:(j + 1) * B]
                vloss, aloss, _ = self.TrainBatch(S[idx], Acts[idx], LP[idx], Adv[idx], G[idx])
        return vloss, aloss

    def TrainTrajectories(self, trajectories, epochs: int = 5):
        """PPOAgent.Train(Trajectory) for every trajectory of the list, in list order, as ONE call (wb_ppo_train_trajectories: one
        launch on the default networks). The mini-batch permutations are drawn from self.rng in the same order and number as
        `for t in trajectories: self.Train(t, epochs)` draws them, so an agent in the same RNG state trains on the same mini-batches.
        Fills every trajectory's Values / Returns / Advantages. Returns [(criticLoss, actorLoss)] per trajectory."""
        trajectories = list(trajectories)
        if not trajectories:
            return []
        B = self.hp.batch_size
        lengths = [len(t.States) for t in trajectories]
        offsets = np.zeros(len(trajectories) + 1, np.int32)
        offsets[1:] = np.cumsum(lengths)
        blocks = []
        for T in lengths:
            if T == 0:  # Train returns before drawing
                continue
            for _ in range(epochs):
                perm = self.rng.permutation(T)
                blocks.extend(perm[j * B:(j + 1) * B] for j in range(T // B))
        index = np.ascontiguousarray(np.concatenate(blocks) if blocks else np.zeros(0), np.int32)
        rows = int(offsets[-1])

        def rows_of(attr, width):
            parts = [np.asarray(getattr(t, attr), np.float32).reshape(-1, width) for t in trajectories if len(t.States)]
            return np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros((0, width), np.float32))
        S = rows_of("States", self.stateSize)
        Acts = rows_of("Actions", self.actionSize)
        LP = rows_of("LogProbabilities", self.actionSize)
        R = rows_of("Rewards", 1).reshape(rows)
        V, G, A = (np.empty(rows, np.float32) for _ in range(3))
        losses = np.zeros((len(trajectories), 2), np.float32)
        skipped = np.zeros(len(trajectories), np.int32)
        check(lib().wb_ppo_train_trajectories(self._h, len(trajectories), ptr(offsets), epochs, ptr(S), ptr(Acts), ptr(LP), ptr(R),
                                              ptr(index), ptr(V), ptr(G), ptr(A), ptr(losses), ptr(skipped)))
        for t, o, T in zip(trajectories, offsets, lengths):
            if T:
                t.Values, t.Returns, t.Advantages = list(V[o:o + T]), list(G[o:o + T]), list(A[o:o + T])
        return [(float(c), float(a)) for c, a in losses]

    def Save(self):  # PPOAgent.Save (PPOAgent.cs:192-213) -> the two .weights files' lines
        return self.critic.Save(), self.actor.Save()


__all__ = ["PPOAgent", "Trajectory", "ParseLayers", "xavier_flat", "net_float_str", "DEFAULT_ACTOR", "DEFAULT_CRITIC", "DENSE",
           "RELU", "LEAKYRELU", "TANH"]
