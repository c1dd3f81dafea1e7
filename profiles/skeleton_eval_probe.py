"""eval_skeleton.py's sample_once_proj + calc_metric_single on one GPU through the mirrored API: B=64, past 10 + future 10
frames, 1000-step cosine schedule, the fused skeleton correction hook (active on the 11 steps t <= 500, t % 50 == 0).
Times, with CUDA events after warm-up and the L2 overwritten before every timed call:
  get_embeddings  MDM._get_embeddings (gt assembly + the conditioning encoder in the library)
  sample          diffusion.p_sample_loop(..., denoised_fn=FusedSkeletonCorrection())  (the whole loop in the library)
  metrics         Engine.skeleton_metrics on the sample
Weights: the exported checkpoint tensors when INTERDIFF_B200_WEIGHTS (or weights_ref/) holds them, else seeded random init.
Prints one JSON line with the card's name and power limit read in the same run."""
import json
import os
import subprocess
import sys
from argparse import Namespace

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from interdiff_b200 import synthetic as S  # noqa: E402
from interdiff_b200.model.correction_skeleton import ObjProjector  # noqa: E402
from interdiff_b200.model.diffusion_skeleton import create_model_and_diffusion  # noqa: E402
from interdiff_b200.sampling import FusedSkeletonCorrection  # noqa: E402
from interdiff_b200.weights import bench_weights, have_ref_weights  # noqa: E402

B, PAST, FUT, STEPS = 64, 10, 10, 1000
T = PAST + FUT
ARGS = dict(embedding_dim=256, smpl_dim=63, num_joints=21, num_points=12, dropout=0.0, num_heads=4, ff_size=256, activation="gelu",
            latent_usage="memory", past_len=PAST, future_len=FUT, cond_mask_prob=0, diffusion_steps=STEPS, noise_schedule="cosine",
            sigma_small=True, weight_v=1)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1]
    except Exception as e:  # the name from the runtime is still worth reporting
        return torch.cuda.get_device_name(0), "unknown (%r)" % (e,)


class _ObjModel:
    def __init__(self, m):
        self.model = m


def main():
    dev = torch.device("cuda:0")
    model, diffusion = create_model_and_diffusion(Namespace(**ARGS))
    sd = {**bench_weights("diffusion_skeleton"), **bench_weights("diffusion_skeleton_encoder")}
    own = model.state_dict()
    model.load_state_dict({k: (sd[k].reshape(own[k].shape) if k in sd else v) for k, v in own.items()})
    model = model.to(dev).eval()
    proj = ObjProjector(Namespace(num_joints=21, dropout=0.0, past_len=PAST, future_len=FUT, embedding_dim=128))
    psd = bench_weights("correction_skeleton")
    own = proj.state_dict()
    proj.load_state_dict({k: (psd[k].reshape(own[k].shape) if k in psd else v) for k, v in own.items()})
    proj = proj.to(dev).eval()

    b = S.make_skeleton_batch(B=B, T=T)
    xs = torch.from_numpy(b["gt"]).squeeze(1).permute(2, 0, 1).to(dev)
    body, obj, pose = xs[..., :63].reshape(T, B, 21, 3), xs[..., 63:99].reshape(T, B, 12, 3), xs[..., 99:].contiguous()
    zp = torch.from_numpy(b["zero_pose_obj"]).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)        # 256 MB > the 126 MB L2
    hook = FusedSkeletonCorrection()
    state = {}

    def get_embeddings():
        state["emb"], gt = model._get_embeddings(body, obj, pose, zp)
        state["gt"] = gt.permute(1, 2, 0).unsqueeze(1).contiguous()

    def sample():
        gt = state["gt"]
        mask = torch.ones_like(gt, dtype=torch.bool)
        mask[..., PAST:] = False
        kw = {"y": {"cond": state["emb"], "inpainted_motion": gt, "inpainting_mask": mask, "obj_model": _ObjModel(proj)}, "zero_pose_obj": zp}
        noise = torch.randn(gt.shape, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
        state["sample"] = diffusion.p_sample_loop(model, gt.shape, clip_denoised=False, noise=noise, model_kwargs=kw, denoised_fn=hook)

    def metrics():
        state["m"] = model.engine_for(dev).skeleton_metrics(state["sample"], state["gt"], PAST)

    def timed(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        ms = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize(dev)
            ms.append(e0.elapsed_time(e1))
        return dict(median_ms=float(np.median(ms)), min_ms=float(np.min(ms)), max_ms=float(np.max(ms)), reps=reps)

    with torch.no_grad():
        res = dict(get_embeddings=timed(get_embeddings, 50), sample=timed(sample, 10), metrics=timed(metrics, 50))
    m = {k: float(v.mean()) for k, v in state["m"].items()}
    name, power = card()
    print(json.dumps(dict(probe="skeleton_eval", gpu=name, power_limit=power, B=B, past_len=PAST, future_len=FUT, steps=STEPS,
                          hook_steps=sum(1 for t in range(STEPS) if t <= 500 and t % 50 == 0),
                          weights="exported checkpoints" if have_ref_weights("diffusion_skeleton_encoder") else "seeded random init",
                          l2="overwritten (256 MB) before every timed call", timings=res, batch_mean_metrics=m,
                          finite=bool(torch.isfinite(state["sample"]).all()))))


if __name__ == "__main__":
    main()
