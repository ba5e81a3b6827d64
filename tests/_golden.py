"""Compact form of tests/golden/sr3_golden.pt (kept under 1 MB).

Random inputs are rounded to float16 before the reference sees them and are stored as float16: nothing is lost, and load() widens them
back to float32.  A large output is stored as a Sample: the values at a fixed set of flat indices (numpy's legacy RandomState, seed 0,
sorted) plus the shape and L2 norm of the whole tensor.  rel() compares a full tensor with a full reference or with a Sample."""
import numpy as np
import torch

SAMPLE_N = 2048


def sample_index(numel, n=SAMPLE_N, seed=0):
    if numel <= n:
        return torch.arange(numel)
    return torch.from_numpy(np.sort(np.random.RandomState(seed).choice(numel, n, replace=False)))


def sample(t, n=SAMPLE_N):
    t = t.detach().float().cpu()
    return {"sample_of": tuple(t.shape), "norm": t.double().norm().item(), "values": t.reshape(-1)[sample_index(t.numel(), n)].clone()}


def is_sample(x):
    return isinstance(x, dict) and "sample_of" in x


def rel(a, b):
    """Relative L2 error of a against b.  b may be a Sample: the error on the sampled elements, or the error of the whole tensor's norm,
    whichever is larger (the norm error never exceeds the full-tensor error, so this is not looser than the sample alone)."""
    a = a.detach().float().cpu()
    if not is_sample(b):
        b = b.detach().float().cpu()
        return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()
    assert tuple(a.shape) == tuple(b["sample_of"]), (tuple(a.shape), b["sample_of"])
    ref = b["values"]
    got = a.reshape(-1)[sample_index(a.numel(), ref.numel())]
    e_sample = ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()
    e_norm = abs(a.double().norm().item() - b["norm"]) / max(b["norm"], 1e-30)
    return max(e_sample, e_norm)


def _widen(x):
    if isinstance(x, torch.Tensor):
        return x.float() if x.dtype == torch.float16 else x
    if isinstance(x, dict):
        return {k: _widen(v) for k, v in x.items()}
    if isinstance(x, tuple):
        return tuple(_widen(v) for v in x)
    if isinstance(x, list):
        return [_widen(v) for v in x]
    return x


def load(path):
    return _widen(torch.load(path, map_location="cpu", weights_only=False))
