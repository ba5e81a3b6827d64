"""Generate tests/golden/*.pt by running the UNMODIFIED reference (imported from
/root/reference, CPU fp32).  Run once in the build container:

    python tests/golden/make_golden.py

The GPU box has no /root/reference; tests there only read the committed fixtures.
Weights are never stored: both implementations draw them from torch.manual_seed(seed)
in the reference's construction order (checked here bit-for-bit against
oracle.sr3_oracle.init_state_dict before anything is written).
"""
import os
import sys

sys.dont_write_bytecode = True
REF = os.environ.get("SR3_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import model.networks as ref_networks  # noqa: E402  (the reference)
import _golden  # noqa: E402  (tests/_golden.py: the compact storage form)
from oracle import sr3_oracle as orc  # noqa: E402

torch.set_num_threads(os.cpu_count())

SCHED_SR3 = {"schedule": "linear", "n_timestep": 2000, "linear_start": 1e-6, "linear_end": 1e-2}


def make_opt(unet, image_size, conditional=True, phase="val", sched=SCHED_SR3):
    return {"phase": phase, "gpu_ids": None, "distributed": False,
            "model": {"which_model_G": "sr3", "finetune_norm": False, "unet": dict(unet),
                      "beta_schedule": {"train": dict(sched), "val": dict(sched)},
                      "diffusion": {"image_size": image_size, "channels": 3, "conditional": conditional}}}


TINY = dict(in_channel=6, out_channel=3, inner_channel=64, channel_multiplier=[1, 2], attn_res=[16], res_blocks=1, dropout=0.0)
FULL = dict(in_channel=6, out_channel=3, inner_channel=64, channel_multiplier=[1, 2, 4, 8, 8], attn_res=[16], res_blocks=2, dropout=0.2)
UNCOND = dict(in_channel=3, out_channel=3, inner_channel=64, channel_multiplier=[1, 2, 4, 8, 8], attn_res=[16], res_blocks=2, dropout=0.2)
BIG = dict(in_channel=6, out_channel=3, inner_channel=64, norm_groups=16, channel_multiplier=[1, 2, 4, 8, 16], attn_res=[], res_blocks=1, dropout=0)


def f16(t):
    """Random inputs are drawn in fp32 and rounded to fp16 values before use, so the file can store them as fp16 without loss."""
    return t.half().float()


def build_ref(unet, image_size, seed, conditional=True, phase="val", sched=SCHED_SR3):
    torch.manual_seed(seed)
    g = ref_networks.define_G(make_opt(unet, image_size, conditional, phase, sched))
    g.set_new_noise_schedule(sched, "cpu")
    g.set_loss("cpu")
    g.eval()
    return g


def check_init(g, unet, image_size, seed, orthogonal=False):
    cfg = orc.UNetConfig(in_channel=unet["in_channel"], out_channel=unet["out_channel"], inner_channel=unet["inner_channel"],
                         norm_groups=unet.get("norm_groups", 32), channel_mults=tuple(unet["channel_multiplier"]),
                         attn_res=tuple(unet["attn_res"]), res_blocks=unet["res_blocks"], dropout=unet["dropout"], image_size=image_size)
    sd = orc.init_state_dict(cfg, seed, orthogonal)
    ref_sd = g.denoise_fn.state_dict()
    assert list(ref_sd.keys()) == list(sd.keys()), "key order / names differ"
    for k in ref_sd:
        assert torch.equal(ref_sd[k], sd[k]), k
    return cfg, sd


def main():
    out = {}
    # ---- 1. schedules -------------------------------------------------------------------
    g = build_ref(TINY, 32, 0)
    sch = {k: v.clone() for k, v in g.state_dict().items() if not k.startswith("denoise_fn.")}
    out_s = {"sr3_linear_2000": {"opt": SCHED_SR3, "buffers": sch,
                                  "sqrt_alphas_cumprod_prev": torch.tensor(g.sqrt_alphas_cumprod_prev)}}
    for name in ["quad", "linear", "warmup10", "warmup50", "const", "jsd", "cosine"]:
        o = {"schedule": name, "n_timestep": 50, "linear_start": 1e-4, "linear_end": 2e-2}
        g.set_new_noise_schedule(o, "cpu")
        out_s[name + "_50"] = {"opt": o, "buffers": {k: v.clone() for k, v in g.state_dict().items() if not k.startswith("denoise_fn.")},
                               "sqrt_alphas_cumprod_prev": torch.tensor(g.sqrt_alphas_cumprod_prev)}
    torch.save(out_s, os.path.join(HERE, "schedules.pt"))

    # ---- 2. positional encoding + noise mlp ------------------------------------------------
    g = build_ref(TINY, 32, 0)
    cfg, sd = check_init(g, TINY, 32, 0)
    nl = torch.tensor([[0.5], [0.9999995], [0.00662267184461], [0.285262383882]])
    pe = g.denoise_fn.noise_level_mlp[0](nl)
    mlp = g.denoise_fn.noise_level_mlp(nl)
    assert torch.equal(pe, orc.positional_encoding(nl, 64))
    out["pe"] = {"noise_level": nl, "pe": pe, "mlp": mlp}

    # ---- 3. tiny UNet: eps + per-layer taps ----------------------------------------------
    torch.manual_seed(100)
    x = f16(torch.randn(2, 6, 32, 32))
    nlv = torch.tensor([[0.7], [0.05]])
    taps = {}
    hooks = []
    for coll in ("downs", "mid", "ups"):
        for i, m in enumerate(getattr(g.denoise_fn, coll)):
            hooks.append(m.register_forward_hook(lambda mod, inp, o, n=f"{coll}.{i}": taps.__setitem__(n, o.detach().clone())))
    with torch.no_grad():
        eps = g.denoise_fn(x, nlv)
    for h in hooks:
        h.remove()
    otaps = {}
    with torch.no_grad():
        oeps = orc.unet_forward(sd, cfg, x, nlv, otaps)
    print("tiny eps oracle-vs-ref max abs", (oeps - eps).abs().max().item())
    out["tiny_unet"] = {"seed": 0, "x": x.half(), "noise_level": nlv, "eps": eps, "taps": {k: _golden.sample(v) for k, v in taps.items()}}

    # tiny: p_mean_variance, seeded loop, p_losses
    sched10 = {"schedule": "linear", "n_timestep": 10, "linear_start": 1e-6, "linear_end": 1e-2}
    g.set_new_noise_schedule(sched10, "cpu")
    torch.manual_seed(101)
    cond = f16(torch.rand(2, 3, 32, 32) * 2 - 1)
    xt = f16(torch.randn(2, 3, 32, 32))
    pmv = {}
    with torch.no_grad():
        for t in (9, 5, 1, 0):
            m, lv = g.p_mean_variance(xt, t, True, condition_x=cond)
            pmv[t] = (m.clone(), lv.clone())
    torch.manual_seed(4321)
    x_T = f16(torch.randn(2, 3, 32, 32))
    noises = [f16(torch.randn(2, 3, 32, 32)) for _ in range(10)]      # noises[i] used at step i
    # replay the same draws inside the reference: randn(shape) then randn_like per step t>0
    draws = [x_T] + [noises[i] for i in reversed(range(1, 10))]
    it = iter(draws)
    orig_randn, orig_randn_like = torch.randn, torch.randn_like
    torch.randn = lambda *a, **k: next(it)
    torch.randn_like = lambda *a, **k: next(it)
    try:
        with torch.no_grad():
            loop = g.super_resolution(cond, continous=True)
    finally:
        torch.randn, torch.randn_like = orig_randn, orig_randn_like
    cond16 = cond.half()                                          # one fp16 copy per input, shared by every entry that uses it
    out["tiny_diffusion"] = {"sched": sched10, "cond": cond16, "x_t": xt.half(), "pmv": pmv, "x_T": x_T.half(),
                             "noises": torch.stack(noises).half(), "loop_continous": _golden.sample(loop), "loop_last": loop[-1].clone()}
    # p_losses with the numpy draws replayed and noise injected
    np.random.seed(7)
    hr = f16(torch.rand(2, 3, 32, 32) * 2 - 1)
    noise = f16(torch.randn(2, 3, 32, 32))
    with torch.no_grad():
        loss = g.p_losses({"HR": hr, "SR": cond}, noise=noise)
    rng = np.random.RandomState(7)
    sch10 = orc.make_schedule(sched10)
    t_draw, gamma = orc.draw_gamma(sch10, 2, rng)
    with torch.no_grad():
        oloss = orc.p_losses(sd, cfg, sch10, hr, cond, gamma, noise)
    print("p_losses ref", loss.item(), "oracle", oloss.item())
    out["tiny_losses"] = {"np_seed": 7, "hr": hr.half(), "sr": cond16, "noise": noise.half(), "t": t_draw, "gamma": gamma, "loss": loss.clone()}

    # ---- 4. full 16->128 config, B=1 ----------------------------------------------------
    g = build_ref(FULL, 128, 0)
    cfgF, sdF = check_init(g, FULL, 128, 0)
    nparams = sum(v.numel() for v in sdF.values())
    assert nparams == 97807491, nparams
    torch.manual_seed(200)
    cond = f16(torch.rand(1, 3, 128, 128) * 2 - 1)
    xt = f16(torch.randn(1, 3, 128, 128))
    cond16, xt16 = cond.half(), xt.half()
    full = {"cond": cond16, "x_t": xt16, "eps": {}, "pmv": {}}
    with torch.no_grad():
        for t in (1999, 1000, 1):
            nl = torch.FloatTensor([g.sqrt_alphas_cumprod_prev[t + 1]]).repeat(1, 1)
            full["eps"][t] = _golden.sample(g.denoise_fn(torch.cat([cond, xt], 1), nl))
            m, lv = g.p_mean_variance(xt, t, True, condition_x=cond)
            full["pmv"][t] = (_golden.sample(m), lv.clone())
    out["full_16_128"] = full
    # orthogonal (train-phase) init, one eps
    g = build_ref(FULL, 128, 3, phase="train")
    check_init(g, FULL, 128, 3, orthogonal=True)
    with torch.no_grad():
        nl = torch.FloatTensor([[0.285262383882]])
        out["full_16_128_orth"] = {"seed": 3, "cond": cond16, "x_t": xt16, "noise_level": nl,
                                   "eps": _golden.sample(g.denoise_fn(torch.cat([cond, xt], 1), nl))}

    # ---- 5. unconditional + 64->512: param counts and a cropped eps -------------------------
    g = build_ref(UNCOND, 128, 0, conditional=False)
    cfgU, sdU = check_init(g, UNCOND, 128, 0)
    assert sum(v.numel() for v in sdU.values()) == 97805763
    with torch.no_grad():
        nl = torch.FloatTensor([[0.5]])
        out["uncond_128"] = {"x_t": xt16, "noise_level": nl, "eps": _golden.sample(g.denoise_fn(xt, nl))}
    g = build_ref(BIG, 512, 0)
    cfgB, sdB = check_init(g, BIG, 512, 0)
    assert sum(v.numel() for v in sdB.values()) == 155334339
    torch.manual_seed(300)
    xb = torch.randn(1, 6, 512, 512)
    with torch.no_grad():
        nl = torch.FloatTensor([[0.3]])
        e = g.denoise_fn(xb, nl)
    out["big_64_512"] = {"x_seed": 300, "noise_level": nl, "eps_crop": _golden.sample(e[:, :, 192:320, 192:320]),
                         "eps_mean": e.mean().clone(), "eps_std": e.std().clone(), "eps_absmax": e.abs().max().clone()}
    torch.save(out, os.path.join(HERE, "sr3_golden.pt"))
    for f in ("schedules.pt", "sr3_golden.pt"):
        size = os.path.getsize(os.path.join(HERE, f))
        print(f, size // 1024, "KiB")
        assert size <= 1_000_000, f"{f} is over 1 MB"


if __name__ == "__main__":
    main()
