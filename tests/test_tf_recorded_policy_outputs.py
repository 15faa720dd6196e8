"""The policy forward pass against what TensorFlow itself computed.

PPOAlgorithm's EpisodeMemory template is (observ, action, mean, logstd, reward) (rex_gym/agents/ppo/algorithm.py:59-62), and the
variables survive in every checkpoint the reference ships: memory/Variable_3 / _4 hold the action mean and log-stddev TF-1.15
produced for each stored observation.  They were produced by the weights from BEFORE the last one to three optimiser updates (the
stored log-stddevs differ from the checkpoint's by ~3e-3), so they are not bit-level goldens of the saved weights -- but they are sharp
enough to tell the architecture apart: the numpy restatement of StreamingNormalize.transform + ForwardGaussianPolicy
(oracle/agent_oracle.py, which tests/test_gpu_agent.py holds the CUDA kernel to) reproduces them to an rms of 0.02-0.08 (the
policy's own stddev is 0.39), while dropping the mean layer's tanh, using tanh hidden units, not centring the observation or
leaving the 1e-4 out of the variance are 2-25x worse.  The stored actions confirm the sampling law: (action - mean) / exp(logstd)
is a unit normal.

The checkpoints and the recorded memory are golden fixtures (tools/gen_policy_golden.py): tests/golden/policies holds the shipped
checkpoints cut to the networks and normalisers, tests/golden/tf_memory_golden.npz a seeded sample of 1200 of the 25 x 400
recorded (observation, mean) rows for the forward pass, and the log-stddevs and the sampling noise (action - mean, half precision) of
all 25 x 400 rows for the sampling law."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.join(GOLDEN, "policies")
MEMORY = np.load(os.path.join(GOLDEN, "tf_memory_golden.npz"))
CKPTS = [("gallop", "ik"), ("gallop", "ol"), ("standup", "ol"), ("turn", "ik"), ("turn", "ol"), ("walk", "ik"), ("walk", "ol")]


def _load(task, sig):
    """Sampled rows: observation and recorded mean; whole 25 x 400 window: recorded log-stddev and action - mean."""
    from oracle import agent_oracle as AO
    from rex_gym_b200.agents.networks import read_tf_policy
    w, filt = read_tf_policy(os.path.join(ROOT, task, sig))
    obs, mean, logstd, noise = (MEMORY["%s_%s_%s" % (task, sig, k)] for k in ("observ", "mean", "logstd", "noise"))
    f = AO.StreamingNormalize((obs.shape[-1],), True, True, 5)
    f.count, f.mean, f.var_sum = filt[0], np.array(filt[1], np.float64), np.array(filt[2], np.float64)
    return AO, w, f, obs.astype(np.float64), mean, logstd, noise.astype(np.float64)


def _variant(w, f, x, variant):
    W = {k: np.asarray(v, np.float64) for k, v in w.items()}
    if variant == "no_centre":
        xn = np.clip(x / (f.std() + 1e-8), -5, 5)
    elif variant == "no_variance_epsilon":
        xn = np.clip((x - f.mean) / np.sqrt(f.var_sum / (f.count - 1)), -5, 5)
    else:
        xn = f.transform(x)
    act = np.tanh if variant == "tanh_hidden" else (lambda z: np.maximum(z, 0))
    h = act(act(xn @ W["pW1"] + W["pb1"]) @ W["pW2"] + W["pb2"])
    m = h @ W["pW3"] + W["pb3"]
    return m if variant == "no_mean_tanh" else np.tanh(m)


@pytest.mark.parametrize("task,sig", CKPTS)
def test_forward_pass_reproduces_the_means_tensorflow_recorded(task, sig):
    AO, w, f, x, mean, logstd, noise = _load(task, sig)
    _, m, _, _ = AO.perform(w, f, x, False)
    m = np.asarray(m).reshape(mean.shape)
    rms = float(np.sqrt(((m - mean) ** 2).mean()))
    corr = float(np.corrcoef(m.reshape(-1), mean.reshape(-1))[0, 1])
    sigma = float(np.exp(w["logstd"]).mean())                    # the policy's own exploration noise, ~0.39
    assert rms < 0.25 * sigma and corr > 0.975, (rms, corr)      # measured: rms 0.02-0.075, corr 0.979-0.999
    # state-independent log-stddev (networks.py:96-99): a handful of distinct vectors in the whole memory -- one per optimiser
    # update that happened while these episodes were being collected (the 25 agents run in parallel, an update lands in the
    # middle of the others' episodes) -- all within 2e-2 of the saved one
    assert len(np.unique(logstd[..., 0])) <= 6 and np.abs(logstd - w["logstd"]).max() < 2e-2
    z = noise / np.exp(logstd)                                   # action = mean + exp(logstd) * N(0, 1)  (algorithm.py:117-121)
    assert abs(z.mean()) < 0.02 and 0.97 < z.std() < 1.03 and abs((np.abs(z) < 1).mean() - 0.6827) < 0.01


@pytest.mark.parametrize("task,sig,variant,factor", [
    ("gallop", "ol", "no_mean_tanh", 8.0), ("standup", "ol", "no_mean_tanh", 8.0),
    ("gallop", "ol", "tanh_hidden", 4.0), ("walk", "ol", "tanh_hidden", 2.5), ("turn", "ol", "tanh_hidden", 2.5),
    ("gallop", "ol", "no_centre", 8.0), ("standup", "ol", "no_centre", 4.0), ("walk", "ik", "no_centre", 2.0),
    ("gallop", "ol", "no_variance_epsilon", 4.0), ("walk", "ik", "no_variance_epsilon", 8.0), ("turn", "ol", "no_variance_epsilon", 4.0)])
def test_recorded_means_tell_the_architecture_apart(task, sig, variant, factor):
    AO, w, f, x, mean, logstd, noise = _load(task, sig)
    rms = lambda m: float(np.sqrt(((m.reshape(mean.shape) - mean) ** 2).mean()))
    ours, other = rms(_variant(w, f, x, "ours")), rms(_variant(w, f, x, variant))
    _, ref, _, _ = AO.perform(w, f, x, False)
    assert abs(ours - rms(np.asarray(ref))) < 1e-9               # `_variant("ours")` IS the oracle's forward pass
    assert other > factor * ours, (variant, other, ours)
