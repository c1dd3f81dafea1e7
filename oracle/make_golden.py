"""Generate tests/golden/* from the reference's OWN classes (imported from the reference tree via
oracle.shims, see oracle.ref_loader):  python -m oracle.make_golden [--reference-checks]
TEST INFRASTRUCTURE.  Inputs are the seeded synthetic generators of interdiff_b200.synthetic;
weights are either the seeded random init (portable: regenerated from the seed by the tests) or
the shipped checkpoints (tests using those need weights_ref, else skip).
"""
import ast
import gzip
import json
import os
import sys
from argparse import Namespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from interdiff_b200 import synthetic as S  # noqa: E402
from oracle import ref_loader as RL  # noqa: E402
from oracle import transforms as tf  # noqa: E402
from tests.helpers import encoder_weights, mdm_weights, projector_skeleton_weights, projector_weights  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def run_loop(diffusion, model, tape, kw, extra=None, denoised_fn=None):
    gd = RL.modules()["diffusion.gaussian_diffusion"]
    idx = [0]

    def fake(x):
        idx[0] += 1
        return tape[idx[0]].clone()
    old, gd.th.randn_like = gd.th.randn_like, fake
    try:
        with torch.no_grad():
            mk = dict(kw)
            if extra:
                mk.update(extra)
            return diffusion.p_sample_loop(model, tuple(tape[0].shape), noise=tape[0].clone(), clip_denoised=False,
                                           model_kwargs=mk, denoised_fn=denoised_fn)
    finally:
        gd.th.randn_like = old


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    for source in ("random", "ref"):
        # ---- SMPL denoiser forward + 5-step loop
        sd = mdm_weights("smpl", source)
        model, _, args = RL.build_mdm_smpl(state_dict=sd, diffusion_steps=1000)
        b = S.make_smpl_batch(B=2, T=30)
        x = torch.from_numpy(S.noise_tape(b["gt"].shape, 0)[0])
        t = torch.tensor([999, 3])
        cond = torch.from_numpy(b["cond"])
        with torch.no_grad():
            out = model(x, t, y={"cond": cond})
        steps = 5
        a = Namespace(**{**vars(args), "diffusion_steps": steps})
        diffusion = RL.modules()["model.diffusion_smpl"].create_gaussian_diffusion(a)
        tape = torch.from_numpy(S.noise_tape(b["gt"].shape, steps))
        kw = {"y": {"cond": cond, "inpainted_motion": torch.from_numpy(b["gt"]), "inpainting_mask": torch.from_numpy(b["mask"])}}
        loop = run_loop(diffusion, model, tape, kw)
        np.savez_compressed(os.path.join(OUT, "mdm_smpl_%s.npz" % source), forward=out.numpy(), t=t.numpy(), loop5=loop.numpy())
        # ---- conditioning encoder (the part of MDM._get_embeddings after the point-cloud encoder)
        esd = encoder_weights(source)
        emodel, _, eargs = RL.build_mdm_smpl(state_dict=esd, diffusion_steps=1000)
        past = torch.from_numpy(b["gt"])[..., : eargs.past_len].contiguous()
        pc = torch.randn(2, 256, generator=torch.Generator().manual_seed(7))
        xs = past.squeeze(1).permute(2, 0, 1)
        with torch.no_grad():
            emb = emodel.bodyEmbedding(xs[..., :135]) + emodel.objEmbedding(xs[..., 135:]) + pc[None]
            cond_out = emodel.encoder(emodel.PositionalEmbedding(emb))
        # point-cloud encoder: the reference's own PointNet2Encoder class on the restated pointnet2_ops operators
        op = torch.from_numpy(b["obj_points"])
        with torch.no_grad():
            pc_pts = emodel.pcEmbedding(torch.cat([op, op.norm(dim=2, keepdim=True)], dim=2).unsqueeze(0)).view(1, 2, -1)[0]
        np.savez_compressed(os.path.join(OUT, "cond_encoder_%s.npz" % source), pc=pc.numpy(), cond=cond_out.numpy(),
                            pc_from_points=pc_pts.numpy())
        # ---- skeleton denoiser, BASELINE config 1: 1 DDPM step, B=2, T=15
        sd = mdm_weights("skeleton", source)
        model, _, args = RL.build_mdm_skeleton(state_dict=sd, diffusion_steps=1000)
        b = S.make_skeleton_batch(B=2, T=15)
        x = torch.from_numpy(S.noise_tape(b["gt"].shape, 1)[0])
        zp = torch.from_numpy(b["zero_pose_obj"])
        with torch.no_grad():
            out = model(x, torch.tensor([999, 999]), zp, y={"cond": torch.from_numpy(b["cond"])})
        a = Namespace(**{**vars(args), "diffusion_steps": 1})
        # a 1-step schedule has posterior_variance[1] undefined in the reference; use the 1000-step
        # process and execute ONE p_sample at t=999 (config 1: "1 DDPM step")
        diffusion = RL.modules()["model.diffusion_skeleton"].create_gaussian_diffusion(Namespace(**{**vars(args), "diffusion_steps": 1000}))
        tape = torch.from_numpy(S.noise_tape(b["gt"].shape, 1))
        kw = {"y": {"cond": torch.from_numpy(b["cond"]), "inpainted_motion": torch.from_numpy(b["gt"]),
                    "inpainting_mask": torch.from_numpy(b["mask"])}, "zero_pose_obj": zp}
        gd = RL.modules()["diffusion.gaussian_diffusion"]
        old, gd.th.randn_like = gd.th.randn_like, (lambda x_: tape[1].clone())
        try:
            with torch.no_grad():
                st = diffusion.p_sample(model, tape[0].clone(), torch.tensor([999, 999]), clip_denoised=False, model_kwargs=kw)
        finally:
            gd.th.randn_like = old
        np.savez_compressed(os.path.join(OUT, "mdm_skeleton_%s.npz" % source), forward=out.numpy(), step_sample=st["sample"].numpy(),
                            step_x0=st["pred_xstart"].numpy())
        # ---- projector
        psd = projector_weights(source)
        proj, _ = RL.build_obj_projector(state_dict=psd, past_len=10, future_len=20)
        g = torch.Generator().manual_seed(3)
        T, B = 30, 4
        ang, tr, hv = torch.randn(T, B, 6, generator=g), torch.randn(T, B, 3, generator=g), torch.randn(T, B, 67, 3, generator=g)
        contact = (torch.rand(B, 67, generator=g) < 0.05).long() * torch.randint(1, 5, (B, 67), generator=g)
        contact[1] = 0
        with torch.no_grad():
            pout = proj.sample(ang, tr, hv, contact)
        np.savez_compressed(os.path.join(OUT, "projector_%s.npz" % source), ang=ang.numpy(), tr=tr.numpy(), hv=hv.numpy(),
                            contact=contact.numpy(), out=pout.numpy())

    # ---- geometry: LBS, normals, signed NN (synthetic SMPL-H, no learned weights)
    smplh = S.make_smplh_model(233)
    layer = RL.build_smpl_layer(smplh)
    g = torch.Generator().manual_seed(1)
    Fn = 5
    pose = 0.4 * torch.randn(Fn, 156, generator=g)
    pose[0, 3:6] = 0
    betas, trans = torch.randn(Fn, 10, generator=g), torch.randn(Fn, 3, generator=g)
    with torch.no_grad():
        verts, jtr, _, _ = layer(pose, th_betas=betas, th_trans=trans)
    mods = RL.modules()
    faces = torch.from_numpy(smplh["faces"])
    normals = mods["data.tools"].vertex_normals(verts, faces.unsqueeze(0).repeat(Fn, 1, 1))
    y = (verts[:, ::23][:, :256] * 1.03).contiguous()
    p2p = mods["tools"].point2point_signed(verts, y, x_normals=normals, return_vector=True)
    sub = slice(None, None, 53)
    np.savez_compressed(os.path.join(OUT, "geometry.npz"), pose=pose.numpy(), betas=betas.numpy(), trans=trans.numpy(),
                        verts_sub=verts[:, sub].numpy(), jtr=jtr.numpy(), normals_sub=normals[:, sub].numpy(), y=y.numpy(),
                        y2x_signed=p2p[0].numpy(), yidx=p2p[2].numpy().astype(np.int32), y2x=p2p[4].numpy())

    # ---- the reference's own denoised_fn source (eval_smpl_short.py:84-130), random projector weights
    psd = projector_weights("random")
    proj, _ = RL.build_obj_projector(state_dict=psd, past_len=10, future_len=20)
    T, B = 30, 2
    b = S.make_smpl_batch(B=B, T=T)
    path = os.path.join(RL.ref_root(), "interdiff", "eval_smpl_short.py")
    tree = ast.parse(open(path).read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "denoised_fn"][0]
    env = dict(torch=torch, args=Namespace(smpl_dim=132, past_len=10, future_len=20), rotation_6d_to_matrix=tf.rotation_6d_to_matrix,
               matrix_to_axis_angle=tf.matrix_to_axis_angle, markerset_ssm67_smplh=mods["data.utils"].markerset_ssm67_smplh,
               vertex_normals=mods["data.tools"].vertex_normals, point2point_signed=mods["tools"].point2point_signed)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), env)
    gt = torch.from_numpy(b["gt"])
    x = gt + 0.02 * torch.randn(gt.shape, generator=torch.Generator().manual_seed(4))
    kw = {"y": {"inpainted_motion": gt, "hand_pose": torch.from_numpy(b["hand_pose"]), "smpl": layer, "beta": torch.from_numpy(b["betas"]),
                "obj_model": Namespace(model=proj), "obj_points": torch.from_numpy(b["obj_points"])}}
    with torch.no_grad():
        o450 = env["denoised_fn"](x.clone(), torch.full((B,), 450), kw)
        o0 = env["denoised_fn"](x.clone(), torch.full((B,), 0), kw)
    # ---- evaluation metrics: the reference's own `metrics` function compiled out of eval_smpl_short.py
    from oracle import transforms as tfm
    from tests.helpers import metrics_inputs
    path = os.path.join(RL.ref_root(), "interdiff", "eval_smpl_short.py")
    fn = [n for n in ast.parse(open(path).read()).body if isinstance(n, ast.FunctionDef) and n.name == "metrics"][0]
    env = {"torch": torch, "axis_angle_to_matrix": tfm.axis_angle_to_matrix, "axis_angle_to_quaternion": tfm.axis_angle_to_quaternion,
           "vertex_normals": RL.modules()["data.tools"].vertex_normals, "point2point_signed": RL.modules()["tools"].point2point_signed}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), env)
    with torch.no_grad():
        mref = env["metrics"](**metrics_inputs(S.make_smplh_model(233)))
    np.savez_compressed(os.path.join(OUT, "metrics.npz"), **{k: v.numpy() for k, v in mref.items()})
    np.savez_compressed(os.path.join(OUT, "denoised_fn_random.npz"), x=x.numpy(), out450=o450.numpy(), out0=o0.numpy())
    reference_checks()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def _set_rotary(model, rotary):
    for m in model.modules():
        if hasattr(m, "rotary"):
            m.rotary = rotary


def _flat7(a):
    """fixed sample of a large output: every 7th element of the flattened array (7 is prime to every axis length sampled)"""
    return a.reshape(-1)[::7].numpy()


def reference_checks():
    """What tests/test_oracle_vs_reference.py and tests/test_host_api.py compare with, from the reference's own classes
    and functions on the seeded random-init weights (the inputs are regenerated by the tests from the same seeds):
      reference_checks.npz   outputs (large ones as a fixed strided sample), diffusion tables, timestep spacing
      checkpoints.json.gz    hyper-parameters and state_dict names / shapes of the shipped checkpoints"""
    mods = RL.modules()
    out = {}
    # ---- MDM forward, both rotary variants; conditioning encoder
    sd = mdm_weights("smpl", "random")
    model, _, args = RL.build_mdm_smpl(state_dict=sd, diffusion_steps=1000)
    b = S.make_smpl_batch(B=3, T=30)
    x = torch.from_numpy(S.noise_tape(b["gt"].shape, 0)[0])
    with torch.no_grad():
        for rotary in ("absolute", "bucketed"):
            _set_rotary(model, rotary)
            out["mdm_forward_%s_flat7" % rotary] = _flat7(model(x, torch.tensor([999, 500, 0]), y={"cond": torch.from_numpy(b["cond"])}))
    _set_rotary(model, "absolute")
    emodel, _, eargs = RL.build_mdm_smpl(state_dict=encoder_weights("random"), diffusion_steps=1000)
    past = torch.from_numpy(b["gt"])[..., : eargs.past_len].contiguous()
    pc = torch.randn(3, 256, generator=torch.Generator().manual_seed(4))
    xs = past.squeeze(1).permute(2, 0, 1)
    with torch.no_grad():
        emb = emodel.bodyEmbedding(xs[..., :135]) + emodel.objEmbedding(xs[..., 135:]) + pc[None]
        out["condition_encoder_flat7"] = _flat7(emodel.encoder(emodel.PositionalEmbedding(emb)))
    # ---- 6-step sampling loop and its diffusion tables
    steps = 6
    diffusion = mods["model.diffusion_smpl"].create_gaussian_diffusion(Namespace(**{**vars(args), "diffusion_steps": steps}))
    b = S.make_smpl_batch(B=2, T=30)
    tape = torch.from_numpy(S.noise_tape(b["gt"].shape, steps))
    kw = {"y": {"cond": torch.from_numpy(b["cond"]), "inpainted_motion": torch.from_numpy(b["gt"]), "inpainting_mask": torch.from_numpy(b["mask"])}}
    out["loop6_flat7"] = _flat7(run_loop(diffusion, model, tape, kw))
    for k in ("posterior_mean_coef1", "posterior_mean_coef2", "posterior_log_variance_clipped"):
        out["loop6_" + k] = getattr(diffusion, k)
    # ---- skeleton denoiser forward
    model, _, _ = RL.build_mdm_skeleton(state_dict=mdm_weights("skeleton", "random"), diffusion_steps=1000)
    b = S.make_skeleton_batch(B=2, T=15)
    x = torch.from_numpy(S.noise_tape(b["gt"].shape, 0)[0])
    with torch.no_grad():
        out["skeleton_forward"] = model(x, torch.tensor([999, 3]), torch.from_numpy(b["zero_pose_obj"]), y={"cond": torch.from_numpy(b["cond"])}).numpy()
    # ---- SMPL-H layer; vertex normals and signed nearest neighbours (vertex-sized outputs sampled)
    smplh = S.make_smplh_model(233)
    layer = RL.build_smpl_layer(smplh)
    g = torch.Generator().manual_seed(1)
    Fn = 7
    pose = 0.4 * torch.randn(Fn, 156, generator=g)
    pose[0, 3:6] = 0
    betas, trans = torch.randn(Fn, 10, generator=g), torch.randn(Fn, 3, generator=g)
    with torch.no_grad():
        v, j, _, _ = layer(pose, th_betas=betas, th_trans=trans)
    out["lbs_verts_sub53"], out["lbs_jtr"] = v[:, ::53].numpy(), j.numpy()
    g = torch.Generator().manual_seed(2)
    verts = torch.from_numpy(smplh["v_template"])[None].repeat(2, 1, 1) + 0.01 * torch.randn(2, 6890, 3, generator=g)
    faces = torch.from_numpy(smplh["faces"])
    n = mods["data.tools"].vertex_normals(verts, faces.unsqueeze(0).repeat(2, 1, 1))
    y = 0.3 * torch.randn(2, 300, 3, generator=g)
    p = mods["tools"].point2point_signed(verts, y, x_normals=n, return_vector=True)
    out["normals_sub53"] = n[:, ::53].numpy()
    out["y2x_signed"], out["yidx_near"] = p[0].numpy(), p[2].numpy().astype(np.int32)
    out["x2y_signed_sub7"], out["xidx_near_sub7"] = p[1][:, ::7].numpy(), p[3][:, ::7].numpy().astype(np.int32)
    # ---- correction networks
    proj, _ = RL.build_obj_projector(state_dict=projector_weights("random"), past_len=10, future_len=20)
    g = torch.Generator().manual_seed(3)
    T, B = 30, 5
    ang, tr, hv = torch.randn(T, B, 6, generator=g), torch.randn(T, B, 3, generator=g), torch.randn(T, B, 67, 3, generator=g)
    contact = (torch.rand(B, 67, generator=g) < 0.05).long() * torch.randint(1, 5, (B, 67), generator=g)
    contact[1] = 0
    with torch.no_grad():
        out["projector"] = proj.sample(ang, tr, hv, contact).numpy()
    sproj, sargs, _ = RL.build_obj_projector_skeleton(projector_skeleton_weights("random"))
    g = torch.Generator().manual_seed(8)
    T, B = sargs.past_len + sargs.future_len, 4
    quat = torch.nn.functional.normalize(torch.randn(T, B, 4, generator=g), dim=2)
    tr, hp = torch.randn(T, B, 3, generator=g), torch.randn(T, B, sargs.num_joints, 3, generator=g)
    with torch.no_grad():
        q, t = sproj.sample(quat, tr, hp)
    out["projector_skeleton_quat"], out["projector_skeleton_trans"] = q.numpy(), t.numpy()
    out["projector_skeleton_lens"] = np.array([sargs.past_len, sargs.future_len, sargs.num_joints])
    # ---- functions of the evaluation script: smooth, denoised_fn
    path = os.path.join(RL.ref_root(), "interdiff", "eval_smpl_short.py")
    fns = {f.name: f for f in ast.parse(open(path).read()).body if isinstance(f, ast.FunctionDef)}
    env = dict(torch=torch, args=Namespace(smpl_dim=132, past_len=10, future_len=20), rotation_6d_to_matrix=tf.rotation_6d_to_matrix,
               matrix_to_axis_angle=tf.matrix_to_axis_angle, markerset_ssm67_smplh=mods["data.utils"].markerset_ssm67_smplh,
               vertex_normals=mods["data.tools"].vertex_normals, point2point_signed=mods["tools"].point2point_signed)
    exec(compile(ast.Module(body=[fns["smooth"], fns["denoised_fn"]], type_ignores=[]), path, "exec"), env)
    g = torch.Generator().manual_seed(0)
    for i, a in enumerate(env["smooth"](*[torch.randn(30, 2, c, generator=g) for c in (6, 159, 12, 9, 3)])):
        out["smooth_%d_flat7" % i] = _flat7(a)
    b = S.make_smpl_batch(B=2, T=30)
    gt = torch.from_numpy(b["gt"])
    x = gt + 0.02 * torch.randn(gt.shape, generator=torch.Generator().manual_seed(4))
    kw = {"y": {"inpainted_motion": gt, "hand_pose": torch.from_numpy(b["hand_pose"]), "smpl": layer, "beta": torch.from_numpy(b["betas"]),
                "obj_model": Namespace(model=proj), "obj_points": torch.from_numpy(b["obj_points"])}}
    with torch.no_grad():
        out["denoised_fn_out7_flat7"] = _flat7(env["denoised_fn"](x.clone(), torch.full((2,), 7), kw))
    # ---- timestep spacing
    ref = mods["diffusion.respace"]
    gd = mods["diffusion.gaussian_diffusion"]
    out["space_1000_100"] = np.array(sorted(ref.space_timesteps(1000, [100])))
    out["space_300_10_15_20"] = np.array(sorted(ref.space_timesteps(300, "10,15,20")))
    from interdiff_b200.diffusion.gaussian_diffusion import get_named_beta_schedule
    rd = ref.SpacedDiffusion(use_timesteps=ref.space_timesteps(1000, [100]), betas=get_named_beta_schedule("cosine", 1000),
                             model_mean_type=gd.ModelMeanType.START_X, model_var_type=gd.ModelVarType.FIXED_SMALL, loss_type=gd.LossType.MSE)
    out["spaced_1000_100_betas"], out["spaced_1000_100_timestep_map"] = rd.betas, np.array(rd.timestep_map)
    np.savez_compressed(os.path.join(OUT, "reference_checks.npz"), **out)
    # ---- checkpoint tables
    tables = {}
    for ck in ("diffusion", "diffusion_skeleton", "correction", "obj_skeleton"):
        hp, csd = RL.load_ckpt(ck)
        tables[ck] = dict(hyper_parameters=dict(hp), state_dict={k: list(v.shape) for k, v in csd.items()})
    with gzip.GzipFile(os.path.join(OUT, "checkpoints.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(tables, sort_keys=True).encode())


if __name__ == "__main__":
    if "--reference-checks" in sys.argv:
        reference_checks()
    else:
        main()
