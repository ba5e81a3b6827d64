#!/usr/bin/env python
"""bench.py -- diffusion steps/sec of the SR3 16->128 sampler at batch 16 (BASELINE.json metric, configs[1]).

    python bench.py --gpus N --steps K --warmup W            # our arm   (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the reference's own code on the host cores

A "step" is one reverse-diffusion step (p_sample) of a batch of 16 images: UNet forward + posterior update.  With N GPUs the ONE batch
of 16 is sharded (16/N images per GPU, no per-step exchange, one all-gather of the finished images): --scaling strong, the default,
is the metric as BASELINE.json / SURVEY.md 8d-8e define it.  --scaling weak gives every GPU its own batch of 16 instead; whichever
mode is not selected is also timed and reported under `other_scaling_mode`.
`value`   : K steps with the sampler state resident in HBM (one persistent cooperative launch per step), CUDA events, max over ranks.
`e2e`     : the same metric through the public API call a user makes on HOST tensors (N=1: GaussianDiffusion.super_resolution's native
            host entry point; N>1: sr3_b200.parallel.sharded_super_resolution): H2D of the condition + K steps + (all-gather +) D2H of
            the images inside the timed region.
`roofline`: the step kernel (the one launch of a step): algorithmic conv+attention FLOPs of a step / its average launch duration (CUDA
            events over the timed region) against the measured bf16 peaks; `by_op` = device time per op class inside that launch.
`cpu_baseline` / --impl reference: the UNMODIFIED reference (oracle/_ref, copied from /root/reference by oracle/build_ref.py) timed on this
            host's cores; falls back to the oracle port when oracle/_ref is absent.  Only these legs touch oracle/ ; the GPU path never does.
`secondary`: configs[2] (64->512, batch 4) and configs[4] (unconditional 128x128, batch 32) on one GPU: ms/step and fraction of bound.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCHED = {"schedule": "linear", "n_timestep": 2000, "linear_start": 1e-6, "linear_end": 1e-2}
UNET = dict(in_channel=6, out_channel=3, inner_channel=64, channel_multiplier=[1, 2, 4, 8, 8], attn_res=[16], res_blocks=2, dropout=0.2)
GLOBAL_BATCH = 16
IMAGE = 128
METRIC = "diffusion steps/sec (batch16, 16->128 SR3)"
# name -> (unet options, image size, conditional, batch, bf16 roofline bound in ms per step on ONE GPU (BASELINE.md section 3), config file)
WORKLOADS = {
    "sr_16_128_b16": (UNET, 128, True, 16, 0.732, "sr_sr3_16_128.json"),
    "sr_64_512_b4": (dict(in_channel=6, out_channel=3, inner_channel=64, norm_groups=16, channel_multiplier=[1, 2, 4, 8, 16], attn_res=[], res_blocks=1, dropout=0),
                     512, True, 4, 2.423, "sr_sr3_64_512.json"),
    "uncond_128_b32": (dict(UNET, in_channel=3), 128, False, 32, 1.463, "sample_sr3_128.json"),
}


def make_opt(sched, unet=UNET, image=IMAGE, conditional=True):
    return {"phase": "val", "gpu_ids": [0], "distributed": False,
            "model": {"which_model_G": "sr3", "finetune_norm": False, "unet": dict(unet),
                      "beta_schedule": {"train": dict(sched), "val": dict(sched)},
                      "diffusion": {"image_size": image, "channels": 3, "conditional": conditional}}}


def algorithmic_flops_per_image(unet=UNET, image=IMAGE):
    """2*MACs of every conv and of QK^T / PV in one UNet forward (SURVEY.md 8d: 92.353 GFLOP for 16->128, 1246.112 for 64->512)."""
    from sr3_b200.model.sr3_modules.unet import layer_table
    layers = layer_table(unet["in_channel"], unet["inner_channel"], unet["channel_multiplier"], unet["attn_res"], unet["res_blocks"], image)
    res, fl = image, 0.0
    for name, kind, cin, cout, attn in layers:
        if kind == "conv":
            fl += 2.0 * res * res * cin * cout * 9
        elif kind == "down":
            res //= 2
            fl += 2.0 * res * res * cin * cout * 9
        elif kind == "up":
            res *= 2
            fl += 2.0 * res * res * cin * cout * 9
        else:
            fl += 2.0 * res * res * (cin * cout * 9 + cout * cout * 9 + (cin * cout if cin != cout else 0))
            if attn:
                hw = res * res
                fl += 2.0 * hw * cout * 3 * cout + 2.0 * hw * cout * cout + 2.0 * 2.0 * hw * hw * cout
    fl += 2.0 * image * image * unet["inner_channel"] * unet["out_channel"] * 9
    return fl


DUMP_BYTES = 64 << 20                            # all arrays of one --dump-outputs together


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every array as <out_dir>/<name>.npy (float32, or float64 where computed so).  DUMP_BYTES is split evenly between the
    arrays; one over its share is replaced by a fixed sample of its flattened elements (the same sorted indices every run, numpy seed 0), so
    two builds stay comparable."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // max(len(arrays), 1)
    total = 0
    for name, a in arrays.items():
        a = np.asarray(a)
        a = np.ascontiguousarray(a, dtype=np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > share:
            a = a.reshape(-1)[np.unique(np.random.default_rng(0).integers(0, a.size, share // a.itemsize))]
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
    assert total <= DUMP_BYTES, total


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"burst": d.get("bf16_tflops"), "sustained": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "hbm_gbs": d.get("hbm_gbs"),
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm_gbs": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self._stop, self._th = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) > 3 + i and s[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU legs (the only code here that touches oracle/)
# ----------------------------------------------------------------------------------------------------------------------
class CpuReference:
    """p_sample of the 16->128 config on the host cores: the unmodified reference from oracle/_ref when it travelled with the repo
    (kind "reference"), else the oracle port (kind "port", pinned to the reference by tests/test_oracle.py)."""

    def __init__(self):
        import torch
        self.torch = torch
        ref_root = os.path.join(ROOT, "oracle", "_ref")
        self.kind = "port"
        if os.path.exists(os.path.join(ref_root, "model", "networks.py")):
            try:
                sys.path.insert(0, ref_root)
                import importlib
                networks = importlib.import_module("model.networks")
                torch.manual_seed(0)
                opt = make_opt(SCHED)
                opt["gpu_ids"] = None
                self.net = networks.define_G(opt)
                self.net.set_new_noise_schedule(SCHED, "cpu")
                self.net.eval()
                self.kind = "reference"
            except Exception as e:            # a broken copy must not take the bench down: say so and use the port
                print(f"bench.py: oracle/_ref is present but unusable ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
                self.kind = "port"
            finally:
                if sys.path and sys.path[0] == ref_root:
                    sys.path.pop(0)
        if self.kind == "port":
            from oracle import sr3_oracle as orc
            self.orc = orc
            self.cfg = orc.UNetConfig(6, 3, 64, 32, (1, 2, 4, 8, 8), (16,), 2, 0.2, 128)
            self.sd = orc.init_state_dict(self.cfg, 0)
            self.sch = orc.make_schedule(SCHED)

    def p_sample(self, x, t, cond):
        torch = self.torch
        with torch.no_grad():
            if self.kind == "reference":
                return self.net.p_sample(x, t, condition_x=cond)          # model/sr3_modules/diffusion.py:166-174, unmodified
            return self.orc.p_sample(self.sd, self.cfg, self.sch, x, t, torch.randn_like(x), cond)

    def tune_threads(self, batch):
        """torch-CPU convs stop scaling (and can collapse) far below the core count of a 100+ core host: probe a few thread counts on
        the very workload that is timed (same batch) and keep the fastest, as anyone running the reference on this box would."""
        torch = self.torch
        n = os.cpu_count() or 1
        cands = sorted({c for c in (n, n // 2, 64, 32, 16, 8) if 1 <= c <= n}, reverse=True)
        torch.manual_seed(0)
        cond = torch.rand(batch, 3, IMAGE, IMAGE) * 2 - 1
        x = torch.randn(batch, 3, IMAGE, IMAGE)
        best, best_t, log = cands[0], float("inf"), {}
        for i, c in enumerate(cands):
            torch.set_num_threads(c)
            if i == 0:
                self.p_sample(x, 1999, cond)            # one-time warm-up (mkldnn primitive caches)
            t0 = time.perf_counter()
            self.p_sample(x, 1999, cond)
            dt = time.perf_counter() - t0
            log[c] = round(dt, 3)
            if dt < best_t:
                best, best_t = c, dt
            if dt > 4 * best_t:
                break
        torch.set_num_threads(best)
        self.threads, self.tune_log = best, log
        return best

    def time_steps(self, batch, reps, warm=1):
        torch = self.torch
        torch.manual_seed(0)
        cond = torch.rand(batch, 3, IMAGE, IMAGE) * 2 - 1
        x = torch.randn(batch, 3, IMAGE, IMAGE)
        ts = []
        for i in range(warm + reps):
            t0 = time.perf_counter()
            x = self.p_sample(x, 1999 - i, cond)
            if i >= warm:
                ts.append(time.perf_counter() - t0)
        return ts


def cpu_baseline_block(reps, warm):
    """Full batch of 16 images per step (no scaling of a sub-sample), thread count tuned on the same batch."""
    ref = CpuReference()
    ref.tune_threads(GLOBAL_BATCH)
    ts = ref.time_steps(GLOBAL_BATCH, reps, warm=warm)
    per = sum(ts) / len(ts)
    return {"value": 1.0 / per, "unit": "steps/s", "cores": ref.threads, "kind": ref.kind, "host_cores": os.cpu_count(),
            "sample": f"p_sample of all 16 images (16->128, fp32, torch-CPU), {reps} steps after {warm} warm-up; thread count tuned at batch 16: {ref.tune_log} s/step",
            "ms_per_step": per * 1e3}


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps = min(args.steps, 8)                 # each CPU step is seconds: a bounded sample keeps the run within minutes
    warm = min(max(args.warmup, 1), 2)
    cb = cpu_baseline_block(steps, warm)
    v = cb["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "sr_sr3_16_128.json sampling, global batch 16, p_sample on host cores", "global_batch": GLOBAL_BATCH,
                       "timed_steps": steps, "timed_warmup": warm},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores")},
            "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
def time_resident(engine, cond, xT, first_index, K, W, T, barrier, dist=None, dev=None):
    """K reverse steps with the sampler state resident in HBM; CUDA events on the launching stream, max over ranks (ms)."""
    import torch
    engine.loop_begin(cond, xT, seed=1234, first_index=first_index)
    engine.steps(T - 1, W)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    remaining, t = K, T - 1 - W
    while remaining > 0:                 # restart from T-1 if K is longer than the schedule
        n = min(remaining, t + 1)
        engine.steps(t, n)
        remaining -= n
        t = T - 1
    e1.record()
    barrier()
    t_ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if dist is not None:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    assert torch.isfinite(engine.read_state()).all(), "sampler state is not finite"
    return float(t_ms.item())


def secondary_workloads(dev, peaks, steps=10):
    """configs[2] and configs[4] of BASELINE.json on one GPU (resident state, CUDA events)."""
    import torch
    import sr3_b200
    out = {}
    for name in ("sr_64_512_b4", "uncond_128_b32"):
        unet, size, cond, B, bound_ms, cfgfile = WORKLOADS[name]
        try:
            torch.manual_seed(0)
            net = sr3_b200.define_G(make_opt(SCHED, unet, size, cond)).to(dev)
            net.set_new_noise_schedule(SCHED, dev)
            eng = net.denoise_fn.engine(B, conditional=cond, channels=3)
            g = torch.Generator().manual_seed(3)
            c = (torch.rand(B, 3, size, size, generator=g) * 2 - 1).to(dev) if cond else None
            x = torch.randn(B, 3, size, size, generator=g).to(dev)
            ms = time_resident(eng, c, x, 0, steps, 3, SCHED["n_timestep"], torch.cuda.synchronize, None, dev) / steps
            fl = algorithmic_flops_per_image(unet, size) * B
            out[name] = {"config": cfgfile, "batch": B, "ms_per_step": ms, "steps_per_s": 1e3 / ms, "launches_per_step": eng.launches_per_step(),
                         "algorithmic_tflop_per_step": fl / 1e12, "achieved_tflops": fl / (ms * 1e-3) / 1e12,
                         "frac_of_measured_burst_bf16": fl / (ms * 1e-3) / 1e12 / peaks["burst"], "roofline_bound_ms_nominal": bound_ms,
                         "frac_of_nominal_bound": bound_ms / ms}
            del eng, net
            torch.cuda.empty_cache()
        except Exception as e:          # a secondary number must never take the headline down
            out[name] = {"error": f"{type(e).__name__}: {e}"}
    # the headline workload in the precise mode (precision="fp32": hi/lo bf16 operand pairs, 3 tensor-core passes; tolerance 1e-3)
    try:
        torch.manual_seed(0)
        net = sr3_b200.define_G(make_opt(SCHED, dict(UNET, precision="fp32"))).to(dev)
        net.set_new_noise_schedule(SCHED, dev)
        eng = net.denoise_fn.engine(GLOBAL_BATCH, conditional=True, channels=3)
        g = torch.Generator().manual_seed(3)
        c = (torch.rand(GLOBAL_BATCH, 3, IMAGE, IMAGE, generator=g) * 2 - 1).to(dev)
        x = torch.randn(GLOBAL_BATCH, 3, IMAGE, IMAGE, generator=g).to(dev)
        ms = time_resident(eng, c, x, 0, steps, 3, SCHED["n_timestep"], torch.cuda.synchronize, None, dev) / steps
        out["sr_16_128_b16_precise_fp32"] = {"config": "sr_sr3_16_128.json", "batch": GLOBAL_BATCH, "dtype": "bf16x3 (hi/lo operand pairs, fp32-level accuracy)",
                                             "ms_per_step": ms, "steps_per_s": 1e3 / ms, "launches_per_step": eng.launches_per_step()}
        del eng, net
        torch.cuda.empty_cache()
    except Exception as e:
        out["sr_16_128_b16_precise_fp32"] = {"error": f"{type(e).__name__}: {e}"}
    # configs[3]: the training step, one GPU's share (8 images) of the global batch of 64
    try:
        ms, _, losses, n_blocks, _ = time_training(dev, 8, 8, 5, 3, torch.cuda.synchronize, None)
        fl = 3.0 * algorithmic_flops_per_image() * 8
        out["train_16_128_b8"] = {"config": "sr_sr3_16_128.json training step (fwd + bwd + Adam), 8 images (one GPU's share of batch 64)", "batch": 8,
                                  "ms_per_step": ms, "steps_per_s": 1e3 / ms, "algorithmic_tflop_per_step": fl / 1e12, "achieved_tflops": fl / (ms * 1e-3) / 1e12,
                                  "frac_of_measured_burst_bf16": fl / (ms * 1e-3) / 1e12 / peaks["burst"], "backward_blocks": n_blocks,
                                  "loss_first_last": [losses[0], losses[-1]]}
    except Exception as e:
        out["train_16_128_b8"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def time_training(dev, per_batch, global_batch, K, W, barrier, dist_mod=None, host_inputs=False, dumps=None):
    """K optimizer iterations (model/model.py:48-58: forward in train() mode incl. Dropout -> backward -> Adam, gradient all-reduce overlapped
    with the backward when world > 1) of sr_sr3_16_128.json on this rank's slice of the global batch.  CUDA events, max over ranks.
    host_inputs: HR / SR come from pinned host memory every step and the loss value is read back (the end-to-end form).
    dumps: a dict that receives the loss of the last timed iteration and the parameters it left (all of them, flattened in order)."""
    import numpy as np
    import torch
    import sr3_b200
    from sr3_b200 import parallel
    torch.manual_seed(0)
    np.random.seed(0)                                   # the (t, gamma) draw of every iteration: same inputs on every run
    opt = make_opt(SCHED)
    opt["phase"] = "train"                              # orthogonal init (networks.py:110-112)
    net = sr3_b200.define_G(opt).to(dev)
    net.set_loss(dev)
    net.set_new_noise_schedule(SCHED, dev)
    net.train()
    g = torch.Generator().manual_seed(5)
    hr_h = (torch.rand(per_batch, 3, IMAGE, IMAGE, generator=g) * 2 - 1).pin_memory()
    sr_h = (torch.rand(per_batch, 3, IMAGE, IMAGE, generator=g) * 2 - 1).pin_memory()
    hr_d, sr_d = hr_h.to(dev), sr_h.to(dev)
    tr = parallel.DataParallelTrainer(net, lr=1e-4)
    losses = []

    def one():
        if host_inputs:
            losses.append(tr.step(hr_h.to(dev, non_blocking=True), sr_h.to(dev, non_blocking=True), global_batch=global_batch))
        else:
            losses.append(tr.step(hr_d, sr_d, global_batch=global_batch))

    for _ in range(W):
        one()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        one()
    e1.record()
    barrier()
    t_ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if dist_mod is not None:
        dist_mod.all_reduce(t_ms, op=dist_mod.ReduceOp.MAX)
    comm_ms = tr.comm_window_ms()
    eng = tr._eng
    n_blocks = eng.num_backward_blocks()
    n_buckets = len(tr.buckets.slices)
    import math
    assert all(math.isfinite(l) for l in losses), "training loss is not finite"
    if dumps is not None:
        dumps["train_loss"] = np.array([losses[-1]], dtype=np.float64)
        dumps["train_params"] = torch.cat([p.detach().reshape(-1) for p in net.parameters()]).cpu().numpy()
    del tr, net
    torch.cuda.empty_cache()
    return float(t_ms.item()) / K, comm_ms, losses, n_blocks, n_buckets


def cpu_train_baseline(steps=2, sample_batch=2, global_batch=64):
    """The unmodified reference's optimize_parameters arithmetic (model/model.py:48-58: netG(data) -> sum / (b c h w) -> backward -> Adam) on the
    host cores, on a bounded sample: `sample_batch` images of the global batch per iteration (fp32, torch-CPU); the per-image cost is linear in the
    batch, so steps/s at the global batch = 1 / (seconds per sample iteration * global_batch / sample_batch)."""
    import torch
    ref_root = os.path.join(ROOT, "oracle", "_ref")
    kind = "port"
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(5)
    hr = torch.rand(sample_batch, 3, IMAGE, IMAGE, generator=g) * 2 - 1
    sr = torch.rand(sample_batch, 3, IMAGE, IMAGE, generator=g) * 2 - 1
    n = os.cpu_count() or 1
    threads = min(n, 32)
    torch.set_num_threads(threads)
    net = None
    if os.path.exists(os.path.join(ref_root, "model", "networks.py")):
        try:
            sys.path.insert(0, ref_root)
            import importlib
            networks = importlib.import_module("model.networks")
            opt = make_opt(SCHED)
            opt["phase"] = "train"
            opt["gpu_ids"] = None
            net = networks.define_G(opt)
            net.set_loss("cpu")
            net.set_new_noise_schedule(SCHED, "cpu")
            net.train()
            kind = "reference"
        except Exception as e:
            print(f"bench.py: oracle/_ref unusable for the training baseline ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
            net = None
        finally:
            if sys.path and sys.path[0] == ref_root:
                sys.path.pop(0)
    ts = []
    if net is not None:
        optim = torch.optim.Adam(list(net.parameters()), lr=1e-4)
        for i in range(steps + 1):
            t0 = time.perf_counter()
            optim.zero_grad()
            l = net({"HR": hr, "SR": sr})
            (l.sum() / hr.numel()).backward()
            optim.step()
            if i > 0:
                ts.append(time.perf_counter() - t0)
    else:
        import numpy as np
        from oracle import sr3_oracle as orc
        cfg = orc.UNetConfig(6, 3, 64, 32, (1, 2, 4, 8, 8), (16,), 2, 0.2, 128)
        sd = orc.init_state_dict(cfg, 0, orthogonal=True)
        sch = orc.make_schedule(SCHED)
        optim = orc.make_adam(sd, 1e-4)
        for i in range(steps + 1):
            t0 = time.perf_counter()
            _, gamma = orc.draw_gamma(sch, sample_batch, np.random.RandomState(i))
            orc.train_step(sd, optim, cfg, sch, hr, sr, gamma, torch.randn(hr.shape))
            if i > 0:
                ts.append(time.perf_counter() - t0)
    per = sum(ts) / len(ts)
    scale = global_batch / sample_batch
    return {"value": 1.0 / (per * scale), "unit": "steps/s", "cores": threads, "kind": kind, "host_cores": n,
            "sample": f"optimize_parameters arithmetic on {sample_batch} of the {global_batch} images per iteration ({steps} iterations after 1 warm-up, fp32 torch-CPU, "
                      f"{per:.2f} s each), scaled by {scale:g} to the global batch", "seconds_per_sample_iteration": per}


def run_reference_train(args, rank, world):
    if rank != 0:
        return
    steps = min(max(args.steps, 1), 3)         # each CPU iteration is seconds, as above
    cb = cpu_train_baseline(steps=steps, global_batch=args.train_batch)
    v = cb["value"]
    line = {"impl": "reference", "metric": "training steps/sec (sr_sr3_16_128 fwd+bwd+Adam, global batch %d)" % args.train_batch, "value": v, "unit": "steps/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": "sr_sr3_16_128.json training step on host cores (bounded sample, see cpu_baseline.sample)",
                                                             "global_batch": args.train_batch},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores")},
            "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_train(args, rank, local, world):
    """--workload train: BASELINE.json configs[3] -- sr_sr3_16_128.json training step (fwd + bwd + Adam), global batch 64, data parallel."""
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py (our arm) needs a B200; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    GB = args.train_batch
    assert GB % world == 0
    per = GB // world
    W, K = max(args.warmup, 3), args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dd = dist if world > 1 else None
    dumps = {} if args.dump_outputs and rank == 0 else None
    with ClockSampler(local) as clk:
        ms, comm_ms, losses, n_blocks, n_buckets = time_training(dev, per, GB, K, W, barrier, dd, host_inputs=False, dumps=dumps)
    if dumps is not None:
        dump_outputs(args.dump_outputs, dumps)
    e2e_ms, _, _, _, _ = time_training(dev, per, GB, max(3, K // 2), 3, barrier, dd, host_inputs=True)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cb = cpu_train_baseline(steps=2, global_batch=GB)
            cpu = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores")}
        except Exception as e:
            cpu = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        peaks = measured_peaks()
        fl = 3.0 * algorithmic_flops_per_image() * GB          # fwd + dgrad + wgrad (SURVEY.md 8d: 277 GFLOP per image)
        img_bytes = per * 3 * IMAGE * IMAGE * 4
        line = {"metric": "training steps/sec (sr_sr3_16_128 fwd+bwd+Adam, global batch %d)" % GB, "value": 1e3 / ms, "unit": "steps/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "sr_sr3_16_128.json training step (configs[3]): p_losses in train() mode (Dropout 0.2) + backward + Adam, random-init "
                                       "(orthogonal) weights, synthetic HR/SR in [-1,1]", "global_batch": GB, "per_gpu_batch": per,
                           "parallelism": f"data parallel x{world}: %d gradient buckets all-reduced (NCCL sum) while the backward of the earlier layers runs; Adam on every rank" % n_buckets,
                           "l2": "per-step working set (activations kept for the backward, several GB) exceeds the 126 MB L2; no explicit flush",
                           "images_per_s": GB * 1e3 / ms},
                "e2e": {"value": 1e3 / e2e_ms, "unit": "steps/s", "h2d_bytes_per_step": 2 * img_bytes, "d2h_bytes_per_step": 8,
                        "api": "sr3_b200.parallel.DataParallelTrainer.step on pinned host HR / SR tensors, loss value read back every step"},
                "gpu_launches": None, "allreduce_window_ms": comm_ms, "backward_blocks": n_blocks,
                "clocks": clk.summary(),
                "roofline": {"bound": "tensor", "kernel": "whole training step (forward tile kernel + data-gradient tile kernel + wgrad_kernel)", "achieved": fl / world / (ms * 1e-3) / 1e12,
                             "peak": peaks["burst"], "unit": "TFLOP/s", "frac": fl / world / (ms * 1e-3) / 1e12 / peaks["burst"], "traffic": None,
                             "algorithmic_flops_per_step_per_gpu": fl / world, "peak_source": peaks["src"]},
                "cpu_baseline": cpu, "losses_first_last": [losses[0], losses[-1]]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50,
                    help="timed steps; --impl reference times at most 8 sampling steps (3 training iterations) and reports the number it timed")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="N>1: strong (default, the metric as defined) = ONE batch of 16 images sharded over the GPUs; "
                         "weak = every GPU samples its own batch of 16 images (global batch 16N, value in batch-16 steps/s)")
    ap.add_argument("--profile-out", default=None, help="write the per-op timing table of one step to this JSON file")
    ap.add_argument("--workload", default="sample", choices=["sample", "train"],
                    help="sample (default): the BASELINE metric; train: configs[3], the training step (fwd + bwd + Adam) at global batch --train-batch")
    ap.add_argument("--train-batch", type=int, default=64)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the timed path computed in its last step as DIR/<name>.npy (same arguments, same inputs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference_train(args, rank, world) if args.workload == "train" else run_reference(args, rank, world)
    if args.workload == "train":
        return run_train(args, rank, local, world)

    if world > 1:
        # communicator set-up at INFO on STDERR (stdout carries exactly one JSON line): the rank count of the job is checkable from the log
        os.environ.setdefault("NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    import torch
    import torch.distributed as dist
    import sr3_b200
    from sr3_b200 import parallel
    assert torch.cuda.is_available(), "bench.py (our arm) needs a B200; there is no CPU fallback"
    assert world == args.gpus or world == 1, f"WORLD_SIZE={world} but --gpus {args.gpus}"
    W = max(args.warmup, 3)
    K = args.steps
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        print(f"bench.py: rank {rank}/{world} on cuda:{local}, backend nccl", file=sys.stderr, flush=True)
    strong = args.scaling == "strong"

    def mode_geometry(is_strong):
        if is_strong:
            assert GLOBAL_BATCH % world == 0
            return GLOBAL_BATCH // world, GLOBAL_BATCH
        return GLOBAL_BATCH, GLOBAL_BATCH * world

    per, global_batch = mode_geometry(strong)
    units = global_batch / GLOBAL_BATCH          # batch-16 steps done per reverse step of the whole job

    torch.manual_seed(0)
    net = sr3_b200.define_G(make_opt(SCHED)).to(dev)
    net.set_new_noise_schedule(SCHED, dev)
    net.eval()
    g = torch.Generator().manual_seed(0)
    cond_all = (torch.rand(global_batch, 3, IMAGE, IMAGE, generator=g) * 2 - 1).pin_memory()
    xT_all = torch.randn(global_batch, 3, IMAGE, IMAGE, generator=g).pin_memory()
    lo = rank * per
    cond_h = cond_all[lo:lo + per].contiguous().pin_memory()
    xT_h = xT_all[lo:lo + per].contiguous().pin_memory()
    eng = net.denoise_fn.engine(per, conditional=True, channels=3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    T = SCHED["n_timestep"]
    dd = dist if world > 1 else None
    with ClockSampler(local) as clk:
        ms = time_resident(eng, cond_h.to(dev), xT_h.to(dev), lo, K, W, T, barrier, dd, dev)
    value = units * K / (ms * 1e-3)
    dumps = {}
    if args.dump_outputs:
        # the images after the last timed step, read before the e2e calls below reuse the engine; all ranks' shards in batch order
        state = eng.read_state()
        if world > 1:
            parts = [torch.empty_like(state) for _ in range(world)]
            dist.all_gather(parts, state)
            state = torch.cat(parts)
        dumps["sample_state"] = state.cpu().numpy()
    step_prof = eng.step_kernel_profile() if eng.uses_step_kernel() else None      # per-op device times of the last timed launch

    # the other scaling mode at N > 1, as a supplementary number (same timing rules)
    other = None
    if world > 1:
        o_per, o_global = mode_geometry(not strong)
        go = torch.Generator().manual_seed(1)
        o_cond = (torch.rand(o_per, 3, IMAGE, IMAGE, generator=go) * 2 - 1).to(dev)
        o_x = torch.randn(o_per, 3, IMAGE, IMAGE, generator=go).to(dev)
        o_eng = net.denoise_fn.engine(o_per, conditional=True, channels=3)
        o_ms = time_resident(o_eng, o_cond, o_x, rank * o_per, K, W, T, barrier, dd, dev)
        other = {"scaling": "weak" if strong else "strong", "value": (o_global / GLOBAL_BATCH) * K / (o_ms * 1e-3), "unit": "steps/s",
                 "ms_per_step": o_ms / K, "per_gpu_batch": o_per, "global_batch": o_global}
        del o_eng

    # ---------------- end to end through the public API on host tensors: `e2e`
    schedK = dict(SCHED, n_timestep=K)
    net.set_new_noise_schedule(schedK, dev)
    e2e_s = []
    for it in range(4):                      # first pass warms the allocator for this schedule; median of the other three
        barrier()
        t0 = time.perf_counter()
        if world == 1:
            out_h = eng.super_resolution_host(cond_h, xT_h, seed=1234, first_index=lo)     # H2D + K steps + D2H inside one native call
        else:
            out_d = parallel.sharded_super_resolution(net, cond_all, x_T=xT_all, seed=1234)  # shard H2D + K steps + NCCL all-gather
            out_h = out_d.to("cpu")                                                        # D2H of the gathered images
        barrier()
        e2e_s.append(time.perf_counter() - t0)
        assert out_h.shape[0] == (per if world == 1 else global_batch) and bool(torch.isfinite(out_h).all())
    e2e_t = torch.tensor([sorted(e2e_s[1:])[1]], device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_val = units * K / float(e2e_t.item())
    img_bytes = per * 3 * IMAGE * IMAGE * 4
    net.set_new_noise_schedule(SCHED, dev)
    if args.dump_outputs and rank == 0:
        dumps["super_resolution"] = out_h.numpy()     # the finished images the last e2e call returned
        dump_outputs(args.dump_outputs, dumps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel.  With the persistent step kernel the step IS one launch: its average duration
    # is the event-timed region / K.  (Per-layer path, the default: the summed event durations of the tile-kernel launches.)
    peaks = measured_peaks()
    alg_flops_step = algorithmic_flops_per_image() * per
    by_op = None
    if step_prof is not None:
        kernel_name = "step_kernel (persistent cooperative launch: the whole reverse step)"
        kernel_ms = ms / K
        by_op = {}
        for t, us in step_prof:
            d = by_op.setdefault(eng.STEP_OP_NAMES[t], {"ops": 0, "us": 0.0})
            d["ops"] += 1
            d["us"] = round(d["us"] + us, 2)
    else:
        prof = eng.profile_step(1000, reps=3)          # eager step, CUDA events around every launch on the launching stream
        kinds = {0: "gemm_tile_kernel", 1: "prep_kernel(groupnorm+silu)", 2: "cast_kernel", 3: "softmax_kernel", 4: "other", 5: "attn_kernel"}
        n_tc = sum(1 for k, _, _, _ in prof if k in (0, 5))
        kernel_name = "gemm_tile_kernel + attn_kernel: the %d tensor-core launches of one step (per-layer path, summed per-launch event times)" % n_tc
        kernel_ms = sum(m for k, m, _, _ in prof if k in (0, 5))
        by_op = {}
        for k, m, fl, by in prof:
            d = by_op.setdefault(kinds[k], {"launches": 0, "us": 0.0, "bytes": 0.0})
            d["launches"] += 1
            d["us"] = round(d["us"] + m * 1e3, 2)
            d["bytes"] += by
        for d in by_op.values():
            d["GB_per_s"] = round(d.pop("bytes") / (d["us"] * 1e-6) / 1e9, 1) if d["us"] > 0 else None
    achieved = alg_flops_step / (kernel_ms * 1e-3) / 1e12
    traffic, traffic_src, whole_step_traffic = None, None, None
    for cand in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", cand)
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            key = "step_kernel_dram_bytes_per_launch" if step_prof is not None else "gemm_tile_kernel_dram_bytes_per_step"
            if key in tj:
                traffic, traffic_src = tj[key], "profiles/" + cand + " (ncu per-launch dram__bytes_read.sum + dram__bytes_write.sum of one step of this build)"
                whole_step_traffic = tj.get("whole_step_dram_bytes")
                break
    roof = {"bound": "tensor", "kernel": kernel_name, "achieved": achieved, "peak": peaks["burst"], "unit": "TFLOP/s",
            "frac": achieved / peaks["burst"], "frac_of_sustained_peak": achieved / peaks["sustained"], "peak_sustained": peaks["sustained"],
            "peak_source": peaks["src"] + ": frac is against the BURST bf16 figure", "traffic": traffic, "traffic_source": traffic_src,
            "traffic_whole_step_incl_groupnorm_apply": whole_step_traffic, "algorithmic_flops_per_launch": alg_flops_step, "algorithmic_bytes_per_launch": 2.98e9 * per / 16.0,
            "kernel_ms_per_launch": kernel_ms, "launches_per_step": eng.launches_per_step(), "ops_per_step": eng.ops_per_step(),
            "frac_of_nominal_bound": (0.732 * per / 16.0) / (ms / K) if per == 16 else None,
            "step_frac_of_burst_peak": (alg_flops_step / (ms / K * 1e-3) / 1e12) / peaks["burst"], "by_op": by_op}
    if args.profile_out:
        os.makedirs(os.path.dirname(os.path.abspath(args.profile_out)), exist_ok=True)
        json.dump({"per_op": [{"op": eng.STEP_OP_NAMES[t], "us": us} for t, us in (step_prof or [])], "summary": roof}, open(args.profile_out, "w"), indent=1)

    secondary = None
    if world == 1 and not args.no_secondary:
        del eng
        torch.cuda.empty_cache()
        secondary = secondary_workloads(dev, peaks)

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cb = cpu_baseline_block(3, 1)
        cpu = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores")}

    lps = roof["launches_per_step"]
    line = {"metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": ("sr_sr3_16_128.json sampling (configs[1]): ONE batch of 16 images%s, T=2000 linear schedule, random-init weights"
                                    % ("" if world == 1 else " sharded over the GPUs")) if strong else
                                   "sr_sr3_16_128.json sampling (configs[1]): batch 16 per GPU, T=2000 linear schedule, random-init weights",
                       "global_batch": global_batch, "per_gpu_batch": per, "parallelism": f"batch-sharded x{world}, no per-step collective, one all-gather of the finished images",
                       "value_unit_note": "steps/s of batch-16 work: (images x reverse steps per second) / 16, summed over all ranks",
                       "l2": "per-step working set (~1.5 GB of activations + weights at batch 16) exceeds the 126 MB L2; no explicit flush",
                       "image_steps_per_s": value * GLOBAL_BATCH},
            "e2e": {"value": e2e_val, "unit": "steps/s", "h2d_bytes_per_step": 2 * img_bytes / K, "d2h_bytes_per_step": (img_bytes if world == 1 else img_bytes * world) / K,
                    "api": ("GaussianDiffusion.super_resolution on host tensors (sr3_super_resolution_host)" if world == 1 else
                            "sr3_b200.parallel.sharded_super_resolution on host tensors (shard, sample, NCCL all-gather) + D2H") + ", schedule length = steps; median of 3 calls",
                    "calls_s": [round(x, 6) for x in e2e_s[1:]]},
            "gpu_launches": lps * K, "launches_per_step": lps,
            "clocks": clk.summary(), "roofline": roof, "cpu_baseline": cpu}
    if secondary is not None:
        line["secondary"] = secondary
    if other is not None:
        line["other_scaling_mode"] = other
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
