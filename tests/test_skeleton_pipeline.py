"""The skeleton model end to end: conditioning encoder (model/diffusion_skeleton.py:194-215), the sampling loop with the
fused correction hook (eval_skeleton.py:80-135) and the evaluation metrics (eval_skeleton.py:46-68,
train_diffusion_skeleton.py:65-87).  CPU cases pin oracle.skeleton_restated to the reference's own code through tests/golden/skeleton_*.npz
(`python -m oracle.make_golden_skeleton`); GPU cases run the library against the restatement with both GEMM backends."""
import os
from argparse import Namespace

import numpy as np
import pytest
import torch

from interdiff_b200 import synthetic as S
from interdiff_b200 import weights as W
from oracle import restate as R
from oracle import skeleton_restated as SR
from oracle import transforms as tf
from oracle.export_ref_weights import OUT_DIR as REF_WEIGHTS
from tests.helpers import mdm_weights, projector_skeleton_weights, rel

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
METRIC_NAMES = ("mpjpe_h", "mpjpe_o", "translation_error", "rotation_error", "rotation_error_l2")


def skeleton_encoder_weights(source="auto", seed=236):
    """mdm_weights('skeleton') + the conditioning path's tensors (encoder.layers.*, shapeEmbedding.*): exported checkpoint
    weights ('ref', skips if absent) or seeded init ('random'); 'auto' = ref if present."""
    sd = dict(mdm_weights("skeleton", source))
    enc = None
    if source in ("ref", "auto"):
        enc = W.load_ref_weights("diffusion_skeleton_encoder", REF_WEIGHTS)
        if enc is None and source == "ref":
            pytest.skip("exported encoder weights not present (oracle/export_skeleton_weights.py)")
    if enc is None:
        enc = W.random_state_dict(W.mdm_skeleton_encoder_shapes(), seed)
    sd.update({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in enc.items()})
    return sd


def skeleton_batch(B, T, seed=233):
    """(body (T,B,21,3), obj (T,B,12,3), pose (T,B,7), zero_pose_obj (B,12,3)) as the reference's data loader hands them to
    _get_embeddings (after the transpose of eval_skeleton.py:115-118)"""
    b = S.make_skeleton_batch(B=B, T=T, seed=seed)
    xs = torch.from_numpy(b["gt"]).squeeze(1).permute(2, 0, 1)
    return (xs[..., :63].reshape(T, B, 21, 3).contiguous(), xs[..., 63:99].reshape(T, B, 12, 3).contiguous(), xs[..., 99:].contiguous(),
            torch.from_numpy(b["zero_pose_obj"]))


def _golden(name):
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, name)).items()}


# ------------------------------------------------------------------------------------------------------------------
# CPU: the restatement against the reference's own code
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("faithful", [True, False])
@pytest.mark.parametrize("source", ["random", "ref"])
def test_restated_skeleton_encoder(source, faithful):
    g = _golden("skeleton_encoder_%s.npz" % source)
    sd = skeleton_encoder_weights(source)
    T, B = g["body"].shape[:2]
    assert torch.equal(g["gt"], torch.cat([g["body"].reshape(T, B, -1), g["obj"].reshape(T, B, -1), g["pose"]], dim=2))
    past = g["gt"][: int(g["past_len"])].permute(1, 2, 0).unsqueeze(1).contiguous()
    with torch.no_grad():
        cond = SR.mdm_skeleton_condition(sd, past, g["zero_pose_obj"], faithful=faithful)
    assert cond.shape == g["cond"].shape
    assert rel(cond, g["cond"]) < 2e-5


def test_restated_skeleton_metrics():
    g = _golden("skeleton_metrics.npz")
    pred, gt = g["pred"], g["gt"]
    # the inputs exercise both branches of the quaternion sign-min
    qp, qg = pred[:, 0, -4:, 10:], gt[:, 0, -4:, 10:]
    plus_wins = (qp + qg).abs().sum(dim=1) < (qp - qg).abs().sum(dim=1)
    assert plus_wins.any() and (~plus_wins).any()
    m = SR.skeleton_metrics(pred, gt, 10)
    for k in METRIC_NAMES:
        assert m[k].shape == (pred.shape[0],)
    for k in ("mpjpe_h", "mpjpe_o", "translation_error", "rotation_error"):
        assert abs(m[k].mean().item() - g["single_" + k].item()) <= 1e-6 * abs(g["single_" + k].item()), k
    for k in ("mpjpe_h", "mpjpe_o", "translation_error"):
        assert abs(m[k].mean().item() - g["train_" + k].item()) <= 1e-6 * abs(g["train_" + k].item()), k
    assert abs(m["rotation_error_l2"].mean().item() - g["train_rotation_error"].item()) <= 1e-6 * g["train_rotation_error"].item()
    # dtype-generic: float64 agrees to float32 rounding
    m64 = SR.skeleton_metrics(pred.double(), gt.double(), 10)
    assert all(m64[k].dtype == torch.float64 and rel(m[k], m64[k]) < 1e-5 for k in METRIC_NAMES)


def test_skeleton_encoder_table_matches_checkpoint():
    """weights.mdm_skeleton_encoder_shapes covers the shipped checkpoint's encoder.* and shapeEmbedding.* tensors exactly"""
    from tests.test_host_api import reference_checkpoint
    _, sd = reference_checkpoint("diffusion_skeleton")
    want = {k: tuple(v.shape) for k, v in sd.items() if k.startswith(("encoder.", "shapeEmbedding."))}
    assert {k: tuple(v) for k, v in W.mdm_skeleton_encoder_shapes().items()} == want


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["simt", "tcgen05"])
def eng(request):
    """Every case runs with both GEMM backends (fp32 SIMT and tcgen05 split-precision)."""
    from interdiff_b200.engine import Engine
    e = Engine("cuda:0")
    e.set_gemm_backend(request.param)
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["random", "ref"])
@pytest.mark.parametrize("B,Tp", [(5, 10), (3, 16), (64, 10)])
def test_encode_condition_skeleton(eng, B, Tp, source):
    """skeleton conditioning encoder against the oracle, then straight into bind + forward"""
    sd = skeleton_encoder_weights(source)
    eng.load_denoiser(sd, "skeleton")
    T = 20
    b = S.make_skeleton_batch(B=B, T=max(T, Tp), seed=B)
    past = torch.from_numpy(b["gt"])[..., :Tp].contiguous()
    zp = torch.from_numpy(b["zero_pose_obj"])
    cond = eng.encode_condition_skeleton(past.cuda(), zp.cuda())
    with torch.no_grad():
        ref = SR.mdm_skeleton_condition(sd, past, zp, faithful=False)
    assert rel(cond.cpu(), ref) < 2e-4
    eng.bind(cond, T, zero_pose_obj=zp)
    x = torch.from_numpy(S.noise_tape((B, 1, 106, T), 0)[0])
    t = torch.full((B,), 321)
    got = eng.forward(x.cuda(), t.cuda()).cpu()
    with torch.no_grad():
        want = R.mdm_skeleton_forward(sd, x, t, zp, ref, faithful=False)
    assert rel(got, want) < 3e-4


def _mirror_model(steps, source):
    from interdiff_b200.model.diffusion_skeleton import create_model_and_diffusion
    from tests.test_host_api import reference_checkpoint
    hp, _ = reference_checkpoint("diffusion_skeleton")
    model, diffusion = create_model_and_diffusion(Namespace(**{**hp, "diffusion_steps": steps, "dropout": 0.0}))
    sd = skeleton_encoder_weights(source)
    own = model.state_dict()
    model.load_state_dict({k: (sd[k].reshape(own[k].shape) if k in sd else v) for k, v in own.items()})
    return model.cuda().eval(), diffusion


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["random", "ref"])
def test_mirror_get_embeddings_skeleton(source):
    """MDM._get_embeddings of the skeleton mirror on the reference's inputs: gt is the reference's concatenation exactly, the
    embedding matches the reference's own encoder (golden) and the oracle"""
    g = _golden("skeleton_encoder_%s.npz" % source)
    model, _ = _mirror_model(1000, source)
    with torch.no_grad():
        cond, gt = model._get_embeddings(g["body"].cuda(), g["obj"].cuda(), g["pose"].cuda(), g["zero_pose_obj"].cuda())
    assert torch.equal(gt.cpu(), g["gt"])
    msd = {k: v.cpu() for k, v in model.state_dict().items()}
    past = g["gt"][: int(g["past_len"])].permute(1, 2, 0).unsqueeze(1).contiguous()
    with torch.no_grad():
        ref = SR.mdm_skeleton_condition(msd, past, g["zero_pose_obj"], faithful=False)
    assert rel(cond.cpu(), ref) < 2e-4 and rel(cond.cpu(), g["cond"]) < 2e-4


@pytest.mark.gpu
def test_skeleton_metrics(eng):
    g = _golden("skeleton_metrics.npz")
    got = eng.skeleton_metrics(g["pred"].cuda(), g["gt"].cuda(), 10)
    want = SR.skeleton_metrics(g["pred"], g["gt"], 10)
    for k in METRIC_NAMES:
        assert rel(got[k], want[k]) < 1e-5, k
    for k in ("mpjpe_h", "mpjpe_o", "translation_error", "rotation_error"):
        assert abs(got[k].mean().item() - g["single_" + k].item()) < 1e-5 * g["single_" + k].item(), k
    assert abs(got["rotation_error_l2"].mean().item() - g["train_rotation_error"].item()) < 1e-5 * g["train_rotation_error"].item()
    # other past lengths: the same per-sample means over the frames t >= past_len
    for P in (0, 19):
        got = eng.skeleton_metrics(g["pred"].cuda(), g["gt"].cuda(), P)
        want = SR.skeleton_metrics(g["pred"], g["gt"], P)
        assert all(rel(got[k], want[k]) < 1e-5 for k in METRIC_NAMES), P


class _ObjModel:            # the reference passes the Lightning module; the hook reads `.model` (eval_skeleton.py:104)
    def __init__(self, m):
        self.model = m


def _python_denoised_fn(n_joints=21, n_points=12):
    """eval_skeleton.py:80-111 transcribed onto the MIRRORED skeleton ObjProjector (and pytorch3d's pure-torch
    quaternion_to_matrix from oracle.transforms); body_obj_to_contact is left out because upstream never uses its result."""
    J, P = n_joints, n_points

    def denoised_fn(x, t, model_kwargs):
        if t[0] > 500 or t[0] % 50 != 0:
            return x
        xs = x.squeeze(1).permute(2, 0, 1).contiguous()
        body = xs[..., :3 * J]
        T, B, _ = body.shape
        pose_gt = model_kwargs["y"]["inpainted_motion"].squeeze(1).permute(2, 0, 1).contiguous()[..., 3 * (J + P):]
        q, tr = model_kwargs["y"]["obj_model"].model.sample(pose_gt[..., 3:], pose_gt[..., :3], body.view(T, B, J, 3))
        pose = torch.cat([tr, q], dim=2)
        rot = tf.quaternion_to_matrix(torch.cat([pose[:, :, -1, None], pose[:, :, -4:-1]], dim=2))[:, :, None]
        obj = (rot.matmul(model_kwargs["zero_pose_obj"][None, :, :, :, None]) + pose[:, :, None, :3, None])[..., 0]
        x_ = torch.cat([body, obj.reshape(T, B, -1), pose], dim=2).permute(1, 2, 0).unsqueeze(1).contiguous()
        return t[0] / 1000 * x + (1 - t[0] / 1000) * x_
    return denoised_fn


@pytest.mark.gpu
@pytest.mark.parametrize("steps", [12, 52])
def test_veneer_sample_once_proj_skeleton(steps):
    """eval_skeleton.py sample_once_proj (:113-143) through the mirrored API only:
       embedding, gt = model._get_embeddings(body, obj, pose, zero_pose_obj) -> diffusion.p_sample_loop(model, shape,
       clip_denoised=False, noise, model_kwargs, denoised_fn) -> metrics.
    (a) denoised_fn = FusedSkeletonCorrection: the whole loop in the library, BIT FOR BIT the Engine path on the same tape;
    (b) the hook as a plain-Python callback on the mirrored projector (step by step): same sample to rounding;
    (c) end to end against the oracle.  12 steps: hook at i = 0 only; 52 steps: i = 50 and 0 (random weights: a
    well-conditioned chain, so the comparison with the oracle means something)."""
    from interdiff_b200.model.correction_skeleton import ObjProjector
    from interdiff_b200.sampling import FusedSkeletonCorrection, draw_tape
    B, past, fut = 3, 10, 10
    T = past + fut
    source = "auto" if steps == 12 else "random"
    model, diffusion = _mirror_model(steps, source)
    proj = ObjProjector(Namespace(num_joints=21, dropout=0.0, past_len=past, future_len=fut, embedding_dim=128))
    psd = projector_skeleton_weights("auto")
    own = proj.state_dict()
    proj.load_state_dict({k: (psd[k].reshape(own[k].shape) if k in psd else v) for k, v in own.items()})
    proj = proj.cuda().eval()
    body, obj, pose, zp = (a.cuda() for a in skeleton_batch(B, T, seed=17))
    with torch.no_grad():
        embedding, gt = model._get_embeddings(body, obj, pose, zp)
    gt = gt.permute(1, 2, 0).unsqueeze(1).contiguous()
    mask = torch.ones_like(gt, dtype=torch.bool)
    mask[..., past:] = False
    kw = lambda: {"y": {"cond": embedding, "inpainted_motion": gt, "inpainting_mask": mask, "obj_model": _ObjModel(proj)}, "zero_pose_obj": zp}
    x_T = torch.randn(gt.shape, generator=torch.Generator().manual_seed(3)).cuda()
    torch.manual_seed(11)
    fused = diffusion.p_sample_loop(model, gt.shape, clip_denoised=False, noise=x_T, model_kwargs=kw(),
                                    denoised_fn=FusedSkeletonCorrection()).clone()
    eng = model.engine_for(embedding.device)
    torch.manual_seed(11)
    tape = draw_tape(eng, x_T, steps)
    direct = eng.p_sample_loop(tape, gt, mask, correction=True).clone()
    assert torch.equal(fused, direct)
    # (b) plain-Python callback (arbitrary-callback path); the fused object called directly takes the same path
    for fn in (_python_denoised_fn(), FusedSkeletonCorrection().__call__):
        torch.manual_seed(11)
        py = diffusion.p_sample_loop(model, gt.shape, clip_denoised=False, noise=x_T, model_kwargs=kw(), denoised_fn=fn)
        assert rel(py, direct) < (1e-4 if steps == 12 else 1e-3)
    # (c) the oracle end to end (model weights = the mirrored module's own state dict)
    cpu_sd = {k: v.cpu() for k, v in model.state_dict().items()}
    ctx = dict(gt=gt.cpu(), zero_pose_obj=zp.cpu(), projector=psd, past_len=past, future_len=fut)
    with torch.no_grad():
        ref = R.p_sample_loop(lambda x, t: R.mdm_skeleton_forward(cpu_sd, x, t, zp.cpu(), embedding.cpu(), faithful=False),
                              R.diffusion_tables(R.named_beta_schedule("cosine", steps)), tape.cpu(), gt.cpu(), mask.cpu(),
                              denoised_fn=R.make_denoised_fn_skeleton(ctx))
    assert rel(direct, ref) < 1e-3
    # metrics of the sample, as sample() of eval_skeleton.py consumes them
    m = eng.skeleton_metrics(direct, gt, past)
    want = SR.skeleton_metrics(direct.cpu(), gt.cpu(), past)
    assert all(rel(m[k], want[k]) < 1e-5 for k in METRIC_NAMES)
