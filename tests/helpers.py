"""Shared helpers for the parity tests."""
import numpy as np
import torch

from interdiff_b200 import synthetic as S
from interdiff_b200 import weights as W
from oracle import restate as R
from oracle.export_ref_weights import OUT_DIR as REF_WEIGHTS


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


def mdm_weights(variant="smpl", source="auto", seed=233):
    """{name: torch tensor} of the hot-path tensors.  source: 'ref' (exported checkpoint weights,
    skips if absent), 'random' (seeded init), 'auto' (ref if present else random)."""
    F = 1024 if variant == "smpl" else 256
    shapes = W.mdm_hot_shapes(variant, F=F)
    sd = None
    if source in ("ref", "auto"):
        sd = W.load_ref_weights("diffusion_" + variant, REF_WEIGHTS)
        if sd is None and source == "ref":
            import pytest
            pytest.skip("exported reference weights not present (oracle/export_ref_weights.py)")
    if sd is None:
        sd = W.random_state_dict({k: v for k, v in shapes.items() if not k.endswith(".pe")}, seed)
    pe = S.sinusoid_table(5000, 256).reshape(5000, 1, 256)
    sd = dict(sd)
    sd["PositionalEmbedding.pe"] = pe
    sd["embedTimeStep.sequence_pos_encoder.pe"] = pe
    return {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()}


def encoder_weights(source="auto", seed=234):
    """mdm_weights('smpl') + the conditioning path's tensors (encoder.layers.*, pcEmbedding.*): exported checkpoint
    weights ('ref', skips if absent) or seeded init ('random'); 'auto' = ref if present."""
    sd = mdm_weights("smpl", source)
    enc = None
    if source in ("ref", "auto"):
        enc = W.load_ref_weights("diffusion_smpl_encoder", REF_WEIGHTS)
        if enc is None and source == "ref":
            import pytest
            pytest.skip("exported encoder weights not present (oracle/export_ref_weights.py)")
    if enc is None:
        enc = W.random_state_dict({**W.mdm_encoder_shapes("smpl"), **W.pointnet_shapes()}, seed)
    sd = dict(sd)
    sd.update({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in enc.items()})
    return sd


def projector_weights(source="auto", seed=233):
    sd = None
    if source in ("ref", "auto"):
        sd = W.load_ref_weights("correction_smpl", REF_WEIGHTS)
        if sd is None and source == "ref":
            import pytest
            pytest.skip("exported reference weights not present")
    if sd is None:
        sd = W.random_state_dict(W.projector_shapes(), seed)
    return {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()}


def projector_skeleton_weights(source="auto", seed=235):
    sd = None
    if source in ("ref", "auto"):
        sd = W.load_ref_weights("correction_skeleton", REF_WEIGHTS)
        if sd is None and source == "ref":
            import pytest
            pytest.skip("exported reference weights not present")
    if sd is None:
        sd = W.random_state_dict(W.projector_skeleton_shapes(), seed)
    return {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()}


def smplh_torch(smplh_np):
    return {k: torch.from_numpy(np.asarray(v)) for k, v in smplh_np.items()}


def metrics_inputs(smplh_np, T=6, B=3, P=256, seed=5):
    """small synthetic evaluation batch: predicted and ground-truth bodies (through the restated LBS) + objects"""
    g = torch.Generator().manual_seed(seed)
    smplh = {k: torch.from_numpy(np.asarray(v)) for k, v in smplh_np.items()}
    pose, pose_gt = 0.3 * torch.randn(T * B, 156, generator=g), 0.3 * torch.randn(T * B, 156, generator=g)
    betas = torch.randn(T * B, 10, generator=g)
    trans, trans_gt = 0.3 * torch.randn(T * B, 3, generator=g), 0.3 * torch.randn(T * B, 3, generator=g)
    with torch.no_grad():
        verts, jtr = R.smplh_lbs(smplh, pose, betas, trans)
        _, jtr_gt = R.smplh_lbs(smplh, pose_gt, betas, trans_gt)
    body = torch.cat([pose, trans], dim=1).view(T, B, -1)
    body_gt = torch.cat([pose_gt, trans_gt], dim=1).view(T, B, -1)
    obj = torch.cat([0.8 * torch.randn(T, B, 3, generator=g), trans.view(T, B, 3) + 0.15 * torch.randn(T, B, 3, generator=g)], dim=2)
    obj[0, 0, :3] = 0.0                                   # small-angle branch of axis_angle_to_quaternion
    obj_gt = torch.cat([0.8 * torch.randn(T, B, 3, generator=g), trans_gt.view(T, B, 3)], dim=2)
    pts = 0.25 * (torch.rand(B, P, 3, generator=g) - 0.5)
    return dict(obj_pred=obj, body_jtr=jtr.view(T, B, -1, 3), body=body, obj_gt=obj_gt, body_jtr_gt=jtr_gt.view(T, B, -1, 3),
                body_gt=body_gt, verts=verts.view(T, B, -1, 3), faces=smplh["faces"].long(), obj_points=pts)


