"""Generate tests/golden/skeleton_*.npz from the reference's OWN code (imported from the reference tree via oracle.shims, see
oracle.ref_loader):  python -m oracle.make_golden_skeleton
TEST INFRASTRUCTURE.  Inputs are seeded; weights are the seeded random init or the shipped checkpoints (exported by
oracle/export_ref_weights.py and oracle/export_skeleton_weights.py), exactly as tests/test_skeleton_pipeline.py rebuilds them.
"""
import ast
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader as RL  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def main():
    """The skeleton model's first and last steps, from the reference's own code:
      skeleton_encoder_{random,ref}.npz  MDM._get_embeddings of model/diffusion_skeleton.py (inputs, embedding, gt)
      skeleton_metrics.npz               calc_metric_single (eval_skeleton.py) and calc_metric (train_diffusion_skeleton.py)
                                         on seeded predictions, some of whose quaternions are sign-flipped (the `+` branch wins)"""
    from tests.test_skeleton_pipeline import skeleton_encoder_weights, skeleton_batch
    for source in ("random", "ref"):
        sd = skeleton_encoder_weights(source)
        model, _, args = RL.build_mdm_skeleton(state_dict=sd, diffusion_steps=1000)
        body, obj, pose, zp = skeleton_batch(B=3, T=20)
        with torch.no_grad():
            emb, gt = model._get_embeddings(body, obj, pose, zp)
        np.savez_compressed(os.path.join(OUT, "skeleton_encoder_%s.npz" % source), body=body.numpy(), obj=obj.numpy(), pose=pose.numpy(),
                            zero_pose_obj=zp.numpy(), cond=emb.numpy(), gt=gt.numpy(), past_len=np.array(args.past_len))
    # ---- metrics, compiled out of the two scripts with ast
    g = torch.Generator().manual_seed(12)
    T, B, J, P = 20, 4, 21, 12
    gt = torch.randn(B, 1, 3 * J + 3 * P + 7, T, generator=g)
    gt[:, :, -4:] = torch.nn.functional.normalize(gt[:, :, -4:], dim=2)
    pred = gt + 0.1 * torch.randn(gt.shape, generator=g)
    pred[:, :, -4:] = torch.nn.functional.normalize(pred[:, :, -4:], dim=2)
    pred[1:3, :, -4:, 12:17] *= -1                       # sign-flipped quaternions: the (pred + gt) branch is the minimum
    split = lambda x: [a.contiguous() for a in torch.split(x.squeeze(1).permute(2, 0, 1), [3 * J, 3 * P, 7], dim=2)]
    (bp, op, pp), (bg, og, pg) = split(pred), split(gt)
    args = (bp.view(T, B, J, 3), bg.view(T, B, J, 3), op.view(T, B, P, 3), og.view(T, B, P, 3), pp, pg)
    out = dict(pred=pred.numpy(), gt=gt.numpy())
    for script, name, key in (("eval_skeleton.py", "calc_metric_single", "single"), ("train_diffusion_skeleton.py", "calc_metric", "train")):
        path = os.path.join(RL.ref_root(), "interdiff", script)
        nodes = [n for n in ast.walk(ast.parse(open(path).read())) if isinstance(n, ast.FunctionDef) and n.name == name]
        env = {"torch": torch}
        exec(compile(ast.Module(body=nodes[:1], type_ignores=[]), path, "exec"), env)
        fn = env[name]
        with torch.no_grad():
            m = fn(None, *args) if key == "train" else fn(*args)
        for k, v in m.items():
            out["%s_%s" % (key, k)] = np.array(v)
    np.savez_compressed(os.path.join(OUT, "skeleton_metrics.npz"), **out)


if __name__ == "__main__":
    main()
