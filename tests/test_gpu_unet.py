"""GPU parity of the whole hot path against the oracle / golden vectors (bf16 operands, fp32 accumulate:
tolerance 1e-2 relative as BASELINE.json's north_star states for bf16)."""
import numpy as np
import pytest
import torch

import _golden
from oracle import sr3_oracle as orc

pytestmark = pytest.mark.gpu
BF16_TOL = 1e-2          # north_star: "within ... 1e-2 bf16" (relative L2)

SCHED = {"schedule": "linear", "n_timestep": 2000, "linear_start": 1e-6, "linear_end": 1e-2}
TINY_UNET = dict(in_channel=6, out_channel=3, inner_channel=64, channel_multiplier=[1, 2], attn_res=[16], res_blocks=1, dropout=0.0)
FULL_UNET = dict(in_channel=6, out_channel=3, inner_channel=64, channel_multiplier=[1, 2, 4, 8, 8], attn_res=[16], res_blocks=2, dropout=0.2)
UNCOND_UNET = dict(FULL_UNET, in_channel=3)
TINY = orc.UNetConfig(6, 3, 64, 32, (1, 2), (16,), 1, 0.0, 32)
FULL = orc.UNetConfig(6, 3, 64, 32, (1, 2, 4, 8, 8), (16,), 2, 0.2, 128)


def make_opt(unet, image_size, conditional=True, phase="val", sched=SCHED):
    return {"phase": phase, "gpu_ids": [0], "distributed": False,
            "model": {"which_model_G": "sr3", "finetune_norm": False, "unet": dict(unet),
                      "beta_schedule": {"train": dict(sched), "val": dict(sched)},
                      "diffusion": {"image_size": image_size, "channels": 3, "conditional": conditional}}}


FP32_TOL = 1e-3          # north_star: "within 1e-3 rel fp32" -- the precise mode (precision="fp32": hi/lo bf16 operand pairs)


def build(unet, image_size, seed, conditional=True, phase="val", sched=SCHED, precision="bf16"):
    import sr3_b200
    torch.manual_seed(seed)
    g = sr3_b200.define_G(make_opt(dict(unet, precision=precision), image_size, conditional, phase, sched)).cuda()
    g.set_loss("cuda")
    g.set_new_noise_schedule(sched, "cuda")
    g.eval()
    return g


def rel(a, b):
    return _golden.rel(a, b)


def test_tiny_unet_layers_and_eps(golden):
    g = golden["tiny_unet"]
    net = build(TINY_UNET, 32, g["seed"])
    eps = net.denoise_fn(g["x"].cuda(), g["noise_level"].cuda())
    eng = net.denoise_fn.engine(2)
    errs = {}
    for name, ref in g["taps"].items():
        errs[name] = rel(eng.read_activation(name), ref)
    print("per-layer rel err:", {k: f"{v:.2e}" for k, v in errs.items()})
    for name, e in errs.items():
        assert e < BF16_TOL, (name, e)
    assert rel(eps, g["eps"]) < BF16_TOL, rel(eps, g["eps"])


def test_tiny_batch_of_one_and_three(golden):
    # odd batches exercise the padded image at the 8x8... (16x16 here) levels and the masked rows
    g = golden["tiny_unet"]
    net = build(TINY_UNET, 32, g["seed"])
    e1 = net.denoise_fn(g["x"][:1].cuda(), g["noise_level"][:1].cuda())
    assert rel(e1, g["eps"][:1]) < BF16_TOL
    x3 = torch.cat([g["x"], g["x"][:1]], 0)
    nl3 = torch.cat([g["noise_level"], g["noise_level"][:1]], 0)
    e3 = net.denoise_fn(x3.cuda(), nl3.cuda())
    assert rel(e3[:2], g["eps"]) < BF16_TOL and rel(e3[2:], g["eps"][:1]) < BF16_TOL


def test_tiny_p_mean_variance_and_loop(golden):
    g = golden["tiny_diffusion"]
    net = build(TINY_UNET, 32, 0, sched=g["sched"])
    for t, (m, lv) in g["pmv"].items():
        mean, logvar = net.p_mean_variance(g["x_t"].cuda(), t, True, condition_x=g["cond"].cuda())
        assert rel(mean, m) < BF16_TOL, (t, rel(mean, m))
        assert float(logvar) == float(lv)
    # p_sample with injected noise == mean + sigma * z
    t = 5
    z = g["noises"][t]
    xs = net.p_sample(g["x_t"].cuda(), t, condition_x=g["cond"].cuda(), noise=z.cuda())
    ref = g["pmv"][t][0] + z * (0.5 * g["pmv"][t][1]).exp()
    assert rel(xs, ref) < BF16_TOL
    # whole seeded loop, continous=True layout [cond ; snapshots...]
    out = net.super_resolution(g["cond"].cuda(), continous=True, x_T=g["x_T"].cuda(), noises=g["noises"].cuda())
    assert tuple(out.shape) == g["loop_continous"]["sample_of"]
    assert torch.equal(out[:2].cpu(), g["cond"])
    assert rel(out, g["loop_continous"]) < BF16_TOL, rel(out, g["loop_continous"])
    last = net.super_resolution(g["cond"].cuda(), continous=False, x_T=g["x_T"].cuda(), noises=g["noises"].cuda())
    assert last.shape == (3, 32, 32)
    assert rel(last, g["loop_last"]) < BF16_TOL


def test_tiny_p_losses(golden):
    g = golden["tiny_losses"]
    net = build(TINY_UNET, 32, 0, sched=golden["tiny_diffusion"]["sched"])
    np.random.seed(g["np_seed"])
    with torch.no_grad():                                  # loss value only: the native path builds no autograd graph
        loss = net.p_losses({"HR": g["hr"].cuda(), "SR": g["sr"].cuda()}, noise=g["noise"].cuda())
    assert abs(loss.item() - g["loss"].item()) / g["loss"].item() < BF16_TOL


def test_philox_loop_is_deterministic_and_shard_invariant(golden):
    g = golden["tiny_diffusion"]
    net = build(TINY_UNET, 32, 0, sched=g["sched"])
    c, xT = g["cond"].cuda(), g["x_T"].cuda()
    a = net.super_resolution(c, continous=True, x_T=xT, seed=77)
    b = net.super_resolution(c, continous=True, x_T=xT, seed=77)
    assert torch.equal(a, b)                              # order-independent GroupNorm sums + fixed-order split-K: repeat runs are bit identical
    # image 1 alone, addressed by its global index, reproduces the batched run (multi-GPU sharding invariant)
    s = net.super_resolution(c[1:], continous=True, x_T=xT[1:], seed=77, first_index=1)
    assert rel(s[-1], a[-1]) < 1e-2
    d = net.super_resolution(c, continous=True, x_T=xT, seed=78)
    assert rel(d[-2:], a[-2:]) > 2e-2
    assert torch.isfinite(a).all()


@pytest.mark.timeout(900)
def test_full_config_eps_and_pmv(golden):
    g = golden["full_16_128"]
    net = build(FULL_UNET, 128, 0)
    sch = orc.make_schedule(SCHED)
    for t in (1999, 1000, 1):
        nl = orc.noise_level_for_t(sch, t, 1)
        eps = net.denoise_fn(torch.cat([g["cond"], g["x_t"]], 1).cuda(), nl.cuda())
        e = rel(eps, g["eps"][t])
        print(f"full 16->128 eps rel err t={t}: {e:.3e}")
        assert e < BF16_TOL, (t, e)
        mean, lv = net.p_mean_variance(g["x_t"].cuda(), t, True, condition_x=g["cond"].cuda())
        assert rel(mean, g["pmv"][t][0]) < BF16_TOL and float(lv) == float(g["pmv"][t][1])


@pytest.mark.timeout(900)
def test_full_config_orthogonal_init(golden):
    g = golden["full_16_128_orth"]
    net = build(FULL_UNET, 128, g["seed"], phase="train")
    eps = net.denoise_fn(torch.cat([g["cond"], g["x_t"]], 1).cuda(), g["noise_level"].cuda())
    e = rel(eps, g["eps"])
    print(f"full 16->128 orthogonal-init eps rel err: {e:.3e}")
    assert e < BF16_TOL, e


@pytest.mark.timeout(900)
def test_unconditional_config(golden):
    g = golden["uncond_128"]
    net = build(UNCOND_UNET, 128, 0, conditional=False)
    eps = net.denoise_fn(g["x_t"].cuda(), g["noise_level"].cuda())
    assert rel(eps, g["eps"]) < BF16_TOL
    net.set_new_noise_schedule({"schedule": "linear", "n_timestep": 4, "linear_start": 1e-6, "linear_end": 1e-2}, "cuda")
    out = net.sample(batch_size=2, continous=True)
    assert out.shape == (2 * (1 + 4), 3, 128, 128) and torch.isfinite(out).all()


@pytest.mark.timeout(1200)
def test_big_64_512_config(golden):
    g = golden["big_64_512"]
    unet = dict(in_channel=6, out_channel=3, inner_channel=64, norm_groups=16, channel_multiplier=[1, 2, 4, 8, 16], attn_res=[], res_blocks=1, dropout=0)
    net = build(unet, 512, 0)
    torch.manual_seed(g["x_seed"])
    xb = torch.randn(1, 6, 512, 512)
    eps = net.denoise_fn(xb.cuda(), g["noise_level"].cuda())
    crop = eps[:, :, 192:320, 192:320]
    assert rel(crop, g["eps_crop"]) < BF16_TOL, rel(crop, g["eps_crop"])
    assert abs(eps.std().item() - g["eps_std"].item()) / g["eps_std"].item() < 1e-2


def test_state_dict_roundtrip_and_reload():
    net = build(TINY_UNET, 32, 1)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    assert len([k for k in sd if not k.startswith("denoise_fn.")]) == 12
    x = torch.randn(2, 6, 32, 32).cuda()
    nl = torch.tensor([[0.3], [0.6]]).cuda()
    e1 = net.denoise_fn(x, nl)
    net2 = build(TINY_UNET, 32, 2)
    e2 = net2.denoise_fn(x, nl)
    assert rel(e2, e1) > 0.1
    net2.load_state_dict(sd, strict=True)
    e3 = net2.denoise_fn(x, nl)
    assert torch.equal(e3, e1)         # same weights, same inputs -> same bits (order-independent statistics)


def test_tiny_unconditional_loop_matches_oracle():
    """sample() path (diffusion.py:180-187, 202-206): unconditional UNet (in_channel=3), seeded loop with injected noise."""
    sched = {"schedule": "linear", "n_timestep": 6, "linear_start": 1e-4, "linear_end": 2e-2}
    unet = dict(TINY_UNET, in_channel=3)
    net = build(unet, 32, 5, conditional=False, sched=sched)
    cfg = orc.UNetConfig(3, 3, 64, 32, (1, 2), (16,), 1, 0.0, 32)
    sd = {k[len("denoise_fn."):]: v.detach().cpu() for k, v in net.state_dict().items() if k.startswith("denoise_fn.")}
    sch = orc.make_schedule(sched)
    g = torch.Generator().manual_seed(9)
    x_T = torch.randn(2, 3, 32, 32, generator=g)
    noises = torch.randn(6, 2, 3, 32, 32, generator=g)
    with torch.no_grad():
        ref = orc.p_sample_loop(sd, cfg, sch, None, x_T, list(noises), conditional=False, continous=True)
    out = net.p_sample_loop((2, 3, 32, 32), continous=True, x_T=x_T.cuda(), noises=noises.cuda())
    assert out.shape == ref.shape == (2 * (1 + 6), 3, 32, 32)
    assert torch.equal(out[:2].cpu(), x_T)
    assert rel(out, ref) < BF16_TOL, rel(out, ref)


def test_sharded_super_resolution_single_rank(golden):
    """parallel.sharded_super_resolution with world size 1 == plain super_resolution with the same Philox seed."""
    from sr3_b200 import parallel
    g = golden["tiny_diffusion"]
    net = build(TINY_UNET, 32, 0, sched=g["sched"])
    a = parallel.sharded_super_resolution(net, g["cond"], x_T=g["x_T"], seed=11)
    b = net.super_resolution(g["cond"].cuda(), continous=True, x_T=g["x_T"].cuda(), seed=11, first_index=0)[-2:]
    assert a.shape == (2, 3, 32, 32) and rel(a, b) < BF16_TOL


@pytest.mark.parametrize("batch", [2, 3])
def test_step_kernel_matches_per_layer_path_bit_for_bit(golden, batch, monkeypatch):
    """One reverse step as ONE persistent cooperative launch (csrc/step_megakernel.cuh) against the same plan run as a CUDA graph of
    per-layer launches (the default; SR3_MEGA=1 selects the step kernel): identical arithmetic, identical bits -- for eps and for a seeded 10-step loop."""
    g = golden["tiny_diffusion"]
    c = g["cond"][:batch] if batch <= g["cond"].shape[0] else torch.cat([g["cond"], g["cond"][:1]], 0)
    xT = g["x_T"][:batch] if batch <= g["x_T"].shape[0] else torch.cat([g["x_T"], g["x_T"][:1]], 0)
    outs = {}
    for mode in ("mega", "layers"):
        if mode == "mega":
            monkeypatch.setenv("SR3_MEGA", "1")
        else:
            monkeypatch.delenv("SR3_MEGA", raising=False)
        net = build(TINY_UNET, 32, 0, sched=g["sched"])
        eng = net.denoise_fn.engine(batch)
        assert eng.uses_step_kernel() == (mode == "mega")
        assert eng.launches_per_step() == (1 if mode == "mega" else eng.ops_per_step())
        x = torch.cat([c, xT], 1).cuda()
        nl = torch.linspace(0.2, 0.9, batch).view(-1, 1).cuda()
        eps = net.denoise_fn(x, nl)
        loop = net.super_resolution(c.cuda(), continous=True, x_T=xT.cuda(), seed=5)
        outs[mode] = (eps.cpu(), loop.cpu())
        del eng, net
    monkeypatch.delenv("SR3_MEGA", raising=False)
    assert torch.equal(outs["mega"][0], outs["layers"][0])
    assert torch.equal(outs["mega"][1], outs["layers"][1])


@pytest.mark.timeout(900)
def test_full_config_is_bit_reproducible(golden):
    """Full 16->128 config, batch 16: two evaluations on the same inputs give the same bits, and a 3-step seeded loop twice as well."""
    g = golden["full_16_128"]
    net = build(FULL_UNET, 128, 0)
    B = 16
    gen = torch.Generator().manual_seed(4)
    cond = (torch.rand(B, 3, 128, 128, generator=gen) * 2 - 1).cuda()
    xT = torch.randn(B, 3, 128, 128, generator=gen).cuda()
    nl = torch.full((B, 1), 0.6).cuda()
    e1 = net.denoise_fn(torch.cat([cond, xT], 1), nl)
    e2 = net.denoise_fn(torch.cat([cond, xT], 1), nl)
    assert torch.equal(e1, e2) and torch.isfinite(e1).all()
    net.set_new_noise_schedule({"schedule": "linear", "n_timestep": 3, "linear_start": 1e-6, "linear_end": 1e-2}, "cuda")
    a = net.super_resolution(cond, continous=True, x_T=xT, seed=3)
    b = net.super_resolution(cond, continous=True, x_T=xT, seed=3)
    assert torch.equal(a, b)


def test_precise_mode_tiny_layers_eps_and_loop(golden):
    """precision="fp32": every tensor-core operand is a (hi, lo) bf16 pair, three passes per product -> the reference's fp32 arithmetic
    (nn.Conv2d / nn.Linear, unet.py:87) within 1e-3 relative, per layer, for eps, p_mean_variance and a seeded 10-step loop."""
    g = golden["tiny_unet"]
    net = build(TINY_UNET, 32, g["seed"], precision="fp32")
    eps = net.denoise_fn(g["x"].cuda(), g["noise_level"].cuda())
    eng = net.denoise_fn.engine(2)
    assert eng.precision == "fp32"
    errs = {name: rel(eng.read_activation(name), ref) for name, ref in g["taps"].items()}
    print("precise mode per-layer rel err:", {k: f"{v:.2e}" for k, v in errs.items()}, "eps", f"{rel(eps, g['eps']):.2e}")
    for name, e in errs.items():
        assert e < FP32_TOL, (name, e)
    assert rel(eps, g["eps"]) < FP32_TOL, rel(eps, g["eps"])
    d = golden["tiny_diffusion"]
    net = build(TINY_UNET, 32, 0, sched=d["sched"], precision="fp32")
    out = net.super_resolution(d["cond"].cuda(), continous=True, x_T=d["x_T"].cuda(), noises=d["noises"].cuda())
    assert rel(out, d["loop_continous"]) < FP32_TOL, rel(out, d["loop_continous"])
    a = net.super_resolution(d["cond"].cuda(), continous=True, x_T=d["x_T"].cuda(), seed=3)
    b = net.super_resolution(d["cond"].cuda(), continous=True, x_T=d["x_T"].cuda(), seed=3)
    assert torch.equal(a, b)


@pytest.mark.timeout(900)
def test_precise_mode_full_config(golden):
    g = golden["full_16_128"]
    net = build(FULL_UNET, 128, 0, precision="fp32")
    sch = orc.make_schedule(SCHED)
    for t in (1999, 1):
        nl = orc.noise_level_for_t(sch, t, 1)
        eps = net.denoise_fn(torch.cat([g["cond"], g["x_t"]], 1).cuda(), nl.cuda())
        e = rel(eps, g["eps"][t])
        print(f"precise mode, full 16->128 eps rel err t={t}: {e:.3e}")
        assert e < FP32_TOL, (t, e)
        mean, lv = net.p_mean_variance(g["x_t"].cuda(), t, True, condition_x=g["cond"].cuda())
        assert rel(mean, g["pmv"][t][0]) < FP32_TOL


@pytest.mark.timeout(1200)
def test_precise_mode_big_64_512_crop(golden):
    """64->512 config in precise mode: covers the three-launch attention (1024 keys) with hi/lo operands."""
    g = golden["big_64_512"]
    unet = dict(in_channel=6, out_channel=3, inner_channel=64, norm_groups=16, channel_multiplier=[1, 2, 4, 8, 16], attn_res=[], res_blocks=1, dropout=0)
    net = build(unet, 512, 0, precision="fp32")
    torch.manual_seed(g["x_seed"])
    xb = torch.randn(1, 6, 512, 512)
    eps = net.denoise_fn(xb.cuda(), g["noise_level"].cuda())
    crop = eps[:, :, 192:320, 192:320]
    assert rel(crop, g["eps_crop"]) < FP32_TOL, rel(crop, g["eps_crop"])
