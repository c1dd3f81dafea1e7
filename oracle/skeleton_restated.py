"""CPU restatement of the skeleton model's first and last steps (TEST INFRASTRUCTURE, see oracle/__init__.py): the conditioning
encoder of MDM._get_embeddings (model/diffusion_skeleton.py:194-215) and the evaluation metrics (eval_skeleton.py:46-68
calc_metric_single, train_diffusion_skeleton.py:65-87 calc_metric).  Builds on oracle.restate (same weight-dict convention);
pinned to the reference's own code by tests/golden/skeleton_*.npz (oracle/make_golden_skeleton.py).  Both functions follow the
dtype of their inputs."""
import torch
import torch.nn.functional as F

from .restate import encoder


def mdm_skeleton_condition(sd, past, zero_pose_obj, nhead=4, rotary=None, faithful=True):
    """(bodyEmbedding(body past) + objEmbedding(keypoint past)) + shapeEmbedding(zero_pose_obj) -> positional encoding -> 8-layer
    encoder.  past: (B,1,C,Tp) = the first past_len frames of the sample tensor (channels [joints | keypoints | 7-D pose], the pose
    is not embedded), zero_pose_obj: (B,P,3).  Returns cond (Tp,B,D)."""
    xs = past.squeeze(1).permute(2, 0, 1).contiguous()  # (Tp,B,C)
    B = xs.shape[1]
    nb = sd["bodyEmbedding.weight"].shape[1]
    no = sd["objEmbedding.weight"].shape[1]
    shape = F.linear(zero_pose_obj.reshape(1, B, -1), sd["shapeEmbedding.weight"], sd["shapeEmbedding.bias"])
    emb = F.linear(xs[..., :nb], sd["bodyEmbedding.weight"], sd["bodyEmbedding.bias"]) \
        + F.linear(xs[..., nb:nb + no], sd["objEmbedding.weight"], sd["objEmbedding.bias"]) + shape
    emb = emb + sd["PositionalEmbedding.pe"][: emb.shape[0]]
    return encoder(sd, emb, nhead, rotary, faithful)


def skeleton_metrics(pred, gt, past_len, n_joints=21):
    """calc_metric_single and calc_metric restated PER SAMPLE: pred / gt (B,1,3J+3P+7,T) sample layout [joints | keypoints |
    trans(3), quat xyzw(4)]; means over the frames t >= past_len (the reference hard-codes 10).  Returns dict of (B,) tensors:
    mpjpe_h, mpjpe_o, translation_error, rotation_error (L1 sign-min, eval_skeleton.py:59-62), rotation_error_l2 (L2 sign-min,
    train_diffusion_skeleton.py:78-81).  Their batch means are the reference's scalars."""
    p = pred.squeeze(1).permute(2, 0, 1)[past_len:]      # (T',B,C)
    g = gt.squeeze(1).permute(2, 0, 1)[past_len:]
    Tf, B, C = p.shape
    J, P = n_joints, (C - 7 - 3 * n_joints) // 3
    bp, bg = p[..., :3 * J].reshape(Tf, B, J, 3), g[..., :3 * J].reshape(Tf, B, J, 3)
    op, og = p[..., 3 * J:3 * (J + P)].reshape(Tf, B, P, 3), g[..., 3 * J:3 * (J + P)].reshape(Tf, B, P, 3)
    pp, pg = p[..., 3 * (J + P):], g[..., 3 * (J + P):]
    out = dict(mpjpe_h=(bp - bg).norm(dim=-1, p=2).mean(dim=(0, 2)), mpjpe_o=(op - og).norm(dim=-1, p=2).mean(dim=(0, 2)),
               translation_error=(pp[..., :3] - pg[..., :3]).norm(dim=-1, p=2).mean(dim=0))
    for name, norm in (("rotation_error", 1), ("rotation_error_l2", 2)):
        v1 = (pp[..., -4:] - pg[..., -4:]).norm(dim=-1, p=norm)
        v2 = (pp[..., -4:] + pg[..., -4:]).norm(dim=-1, p=norm)
        out[name] = torch.stack([v1, v2], dim=0).min(dim=0)[0].mean(dim=0)
    return out
