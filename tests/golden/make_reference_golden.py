"""Generate tests/golden/reference_tiny_pmv.pt by running the UNMODIFIED reference (CPU fp32):

    SR3_REFERENCE=<checkout of Janspiry/Image-Super-Resolution-via-Iterative-Refinement> python tests/golden/make_reference_golden.py

What tests/test_oracle.py::test_live_reference_matches_oracle compares the oracle with: the tiny conditional UNet built by the
reference's define_G under torch.manual_seed(11) (its weights as one sha256 per state-dict entry, in the reference's key order) and
its p_mean_variance at t = 19, 7, 0 of a 20-step linear schedule on a fixed batch of three images.
"""
import hashlib
import os
import sys

sys.dont_write_bytecode = True
REF = os.environ.get("SR3_REFERENCE")
if not REF or not os.path.isdir(os.path.join(REF, "model")):
    sys.exit("set SR3_REFERENCE to a checkout of the original project (the directory that holds model/)")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)

import torch  # noqa: E402

import model.networks as ref_networks  # noqa: E402  (the reference)

SCHED = {"schedule": "linear", "n_timestep": 20, "linear_start": 1e-6, "linear_end": 1e-2}
TINY = dict(in_channel=6, out_channel=3, inner_channel=64, channel_multiplier=[1, 2], attn_res=[16], res_blocks=1, dropout=0.0)
SEED = 11
TS = (19, 7, 0)


def tensor_sha256(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def main():
    opt = {"phase": "val", "gpu_ids": None, "distributed": False,
           "model": {"which_model_G": "sr3", "finetune_norm": False, "unet": dict(TINY),
                     "beta_schedule": {"train": SCHED, "val": SCHED},
                     "diffusion": {"image_size": 32, "channels": 3, "conditional": True}}}
    torch.manual_seed(SEED)
    g = ref_networks.define_G(opt)
    g.set_new_noise_schedule(SCHED, "cpu")
    g.eval()
    weights = [(k, tuple(v.shape), tensor_sha256(v)) for k, v in g.denoise_fn.state_dict().items()]
    torch.manual_seed(5)
    x, c = torch.randn(3, 3, 32, 32), torch.rand(3, 3, 32, 32) * 2 - 1
    pmv = {}
    with torch.no_grad():
        for t in TS:
            m, lv = g.p_mean_variance(x, t, True, condition_x=c)
            pmv[t] = (m.clone(), float(lv))
    out = {"sched": SCHED, "unet": TINY, "seed": SEED, "weights": weights, "x": x, "cond": c, "pmv": pmv}
    path = os.path.join(HERE, "reference_tiny_pmv.pt")
    torch.save(out, path)
    print(f"wrote {path}: {len(weights)} weight digests, p_mean_variance at t={TS}")


if __name__ == "__main__":
    main()
