"""Pins oracle/sr3_oracle.py against (a) the golden vectors produced by the unmodified
reference (tests/golden/make_golden.py), (b) the KATs listed in SURVEY.md 8c, and
(c) the reference's weights and p_mean_variance recorded by tests/golden/make_reference_golden.py."""
import hashlib
import math
import os

import numpy as np
import pytest
import torch

import _golden
from oracle import sr3_oracle as orc

TINY = orc.UNetConfig(6, 3, 64, 32, (1, 2), (16,), 1, 0.0, 32)
FULL = orc.UNetConfig(6, 3, 64, 32, (1, 2, 4, 8, 8), (16,), 2, 0.2, 128)
UNCOND = orc.UNetConfig(3, 3, 64, 32, (1, 2, 4, 8, 8), (16,), 2, 0.2, 128)
BIG = orc.UNetConfig(6, 3, 64, 16, (1, 2, 4, 8, 16), (), 1, 0.0, 512)


def rel(a, b):
    return _golden.rel(a, b)


def test_schedule_golden(golden_schedules):
    for name, g in golden_schedules.items():
        s = orc.make_schedule(g["opt"])
        assert s.num_timesteps == g["opt"]["n_timestep"]
        for k, v in g["buffers"].items():
            assert torch.equal(s.buffers[k], v) or torch.allclose(s.buffers[k], v, rtol=0, atol=0, equal_nan=True), (name, k)
        assert np.array_equal(s.sqrt_alphas_cumprod_prev, g["sqrt_alphas_cumprod_prev"].numpy())


def test_schedule_kats():
    # SURVEY.md 8c: sr3 linear 1e-6 -> 1e-2, T=2000, indices 0,1,2,1000,1998,1999
    s = orc.make_schedule({"schedule": "linear", "n_timestep": 2000, "linear_start": 1e-6, "linear_end": 1e-2})
    idx = [0, 1, 2, 1000, 1998, 1999]
    kat = {
        "betas": [1.0e-6, 6.0020011e-6, 1.10040019e-5, 5.00300108e-3, 9.99499764e-3, 1.0e-2],
        "alphas_cumprod": [0.999998987, 0.999993026, 0.999981999, 0.0813746303, 4.43028111e-5, 4.38597817e-5],
        "sqrt_recip_alphas_cumprod": [1.00000048, 1.00000346, 1.00000906, 3.50554466, 150.239578, 150.99646],
        "sqrt_recipm1_alphas_cumprod": [1.00000051e-3, 2.64613749e-3, 4.24337666e-3, 3.35988736, 150.236252, 150.993149],
        "posterior_mean_coef1": [1.0, 0.857183993, 0.611130297, 1.55749184e-3, 6.686501e-5, 6.65632761e-5],
        "posterior_mean_coef2": [0.0, 0.142816007, 0.388869703, 0.99705106, 0.994989514, 0.994987011],
        "posterior_log_variance_clipped": [-46.0517006, -13.9696131, -12.3617573, -5.29816294, -4.60567093, -4.60517073],
    }
    for k, vals in kat.items():
        got = s.buffers[k][idx].double().numpy()
        assert np.allclose(got, np.array(vals), rtol=2e-6, atol=1e-12), (k, got)
    sp = s.sqrt_alphas_cumprod_prev[[0, 1, 2, 1001, 1999, 2000]]
    assert np.allclose(sp, [1.0, 0.9999995, 0.999996498996, 0.285262383882, 0.00665603564188, 0.00662267184461], rtol=1e-9)
    T = 2000
    inter = 1 | (T // 10)
    assert [i for i in range(T) if i % inter == 0] == [0, 201, 402, 603, 804, 1005, 1206, 1407, 1608, 1809]


def test_positional_encoding_kat(golden):
    pe = orc.positional_encoding(torch.tensor([[0.5]]), 64)
    assert pe.shape == (1, 1, 64)
    assert np.allclose(pe[0, 0, :3].numpy(), [0.47942555, 0.36622331, 0.27748054], rtol=1e-6)
    assert np.allclose(pe[0, 0, 32:35].numpy(), [0.87758255, 0.93052697, 0.96073127], rtol=1e-6)
    g = golden["pe"]
    assert torch.equal(orc.positional_encoding(g["noise_level"], 64), g["pe"])
    sd = orc.init_state_dict(TINY, 0)
    assert torch.allclose(orc.noise_level_mlp(sd, g["noise_level"], 64), g["mlp"], rtol=1e-5, atol=1e-6)


def test_param_counts():
    for cfg, n in ((FULL, 97807491), (UNCOND, 97805763), (BIG, 155334339)):
        assert sum(int(np.prod(s)) for _, s, _ in orc.param_specs(cfg)) == n
    downs, mid, ups = orc.unet_topology(FULL)
    assert len(downs) == 15 and len(ups) == 19
    assert [(s.cin, s.cout) for s in ups if s.kind == "res"][:4] == [(1024, 512)] * 3 + [(1024, 512)]
    assert sum(s.attn for s in downs + mid + ups) == 6


def test_tiny_unet_golden(golden):
    g = golden["tiny_unet"]
    sd = orc.init_state_dict(TINY, g["seed"])
    taps = {}
    with torch.no_grad():
        eps = orc.unet_forward(sd, TINY, g["x"], g["noise_level"], taps)
    assert rel(eps, g["eps"]) < 2e-6
    for k, v in g["taps"].items():
        assert rel(taps[k], v) < 2e-6, k


def test_tiny_diffusion_golden(golden):
    g = golden["tiny_diffusion"]
    sd = orc.init_state_dict(TINY, 0)
    sch = orc.make_schedule(g["sched"])
    with torch.no_grad():
        for t, (m, lv) in g["pmv"].items():
            om, olv = orc.p_mean_variance(sd, TINY, sch, g["x_t"], t, True, g["cond"])
            assert rel(om, m) < 5e-6 and float(olv) == float(lv)
        loop = orc.p_sample_loop(sd, TINY, sch, g["cond"], g["x_T"], list(g["noises"]), True, continous=True)
    assert tuple(loop.shape) == g["loop_continous"]["sample_of"] == (2 * 11, 3, 32, 32)
    assert rel(loop, g["loop_continous"]) < 2e-5
    last = orc.p_sample_loop(sd, TINY, sch, g["cond"], g["x_T"], list(g["noises"]), True, continous=False)
    assert last.shape == (3, 32, 32)        # reference quirk: ret_img[-1] is the last image only
    assert rel(last, g["loop_last"]) < 2e-5


def test_tiny_losses_golden(golden):
    g = golden["tiny_losses"]
    sd = orc.init_state_dict(TINY, 0)
    sch = orc.make_schedule(golden["tiny_diffusion"]["sched"])
    t, gamma = orc.draw_gamma(sch, 2, np.random.RandomState(g["np_seed"]))
    assert t == g["t"] and torch.equal(gamma, g["gamma"])
    with torch.no_grad():
        loss = orc.p_losses(sd, TINY, sch, g["hr"], g["sr"], gamma, g["noise"])
    assert abs(loss.item() - g["loss"].item()) / g["loss"].item() < 1e-5


@pytest.mark.timeout(600)
def test_full_unet_golden(golden):
    g = golden["full_16_128"]
    sd = orc.init_state_dict(FULL, 0)
    sch = orc.make_schedule({"schedule": "linear", "n_timestep": 2000, "linear_start": 1e-6, "linear_end": 1e-2})
    torch.set_num_threads(os.cpu_count())
    with torch.no_grad():
        for t in (1999, 1):
            nl = orc.noise_level_for_t(sch, t, 1)
            eps = orc.unet_forward(sd, FULL, torch.cat([g["cond"], g["x_t"]], 1), nl)
            assert rel(eps, g["eps"][t]) < 5e-6, t
        m, lv = orc.p_mean_variance(sd, FULL, sch, g["x_t"], 1000, True, g["cond"])
        assert rel(m, g["pmv"][1000][0]) < 5e-6 and float(lv) == float(g["pmv"][1000][1])
    go = golden["full_16_128_orth"]
    sdo = orc.init_state_dict(FULL, go["seed"], orthogonal=True)
    with torch.no_grad():
        eps = orc.unet_forward(sdo, FULL, torch.cat([go["cond"], go["x_t"]], 1), go["noise_level"])
    assert rel(eps, go["eps"]) < 5e-6


def test_uncond_golden(golden):
    g = golden["uncond_128"]
    sd = orc.init_state_dict(UNCOND, 0)
    with torch.no_grad():
        eps = orc.unet_forward(sd, UNCOND, g["x_t"], g["noise_level"])
    assert rel(eps, g["eps"]) < 5e-6


def test_live_reference_matches_oracle():
    """The unmodified reference side by side with the oracle, through what it computed (tests/golden/make_reference_golden.py):
    the weights its define_G draws under seed 11 (bit for bit, as per-tensor sha256 in its key order) and its p_mean_variance."""
    g = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_tiny_pmv.pt"),
                   map_location="cpu", weights_only=False)
    sd = orc.init_state_dict(TINY, g["seed"])
    assert [k for k, _, _ in g["weights"]] == list(sd.keys())
    for k, shape, digest in g["weights"]:
        v = sd[k]
        assert tuple(v.shape) == shape and hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() == digest, k
    sch = orc.make_schedule(g["sched"])
    x, c = g["x"], g["cond"]
    with torch.no_grad():
        for t, (m, lv) in g["pmv"].items():
            om, olv = orc.p_mean_variance(sd, TINY, sch, x, t, True, c)
            assert rel(om, m) < 5e-6 and float(lv) == float(olv), t
