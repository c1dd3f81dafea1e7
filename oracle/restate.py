"""CPU restatement (torch, fp32 unless stated) of the reference's algorithm for every function
on the sampling hot path (SURVEY.md section 8a, rows A1-A13).  TEST INFRASTRUCTURE (see
oracle/__init__.py): this file is the parity checker for the CUDA path and the CPU baseline
that bench.py times; the product never imports it.

Every function cites the reference file:line it follows (paths relative to
/root/reference/interdiff).  Weights are passed as flat dicts {reference state_dict name:
tensor} so that the same dict feeds the reference module, this restatement and the CUDA path.

Pinned by the golden vectors under tests/golden/ (generated from the reference's own classes by
oracle/make_golden.py; tests/test_oracle_vs_reference.py and tests/test_golden.py).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from . import transforms as tf
from .local_attention_restated import LocalAttention, DEFAULT_ROTARY

# ----------------------------------------------------------------------------------------
# A3/A4/A5: denoiser
# ----------------------------------------------------------------------------------------


def layer_norm(x, sd, prefix, eps=1e-5):
    """torch.nn.LayerNorm, eps 1e-5 (model/sublayers.py:271-273 defaults)."""
    return F.layer_norm(x, (x.shape[-1],), sd[prefix + "weight"], sd[prefix + "bias"], eps)


def multihead_attention(sd, prefix, query, key, nhead):
    """torch.nn.MultiheadAttention forward, eval mode, no masks, seq-first (L,B,D);
    packed in_proj, scale 1/sqrt(head_dim) (built at model/diffusion_smpl.py:73-78 via
    torch.nn.TransformerDecoderLayer and at model/sublayers.py:261)."""
    W, bias = sd[prefix + "in_proj_weight"], sd[prefix + "in_proj_bias"]
    D = W.shape[1]
    hd = D // nhead
    L, B, _ = query.shape
    S = key.shape[0]
    q = F.linear(query, W[:D], bias[:D])
    k = F.linear(key, W[D:2 * D], bias[D:2 * D])
    v = F.linear(key, W[2 * D:], bias[2 * D:])
    q = q.reshape(L, B * nhead, hd).transpose(0, 1)
    k = k.reshape(S, B * nhead, hd).transpose(0, 1)
    v = v.reshape(S, B * nhead, hd).transpose(0, 1)
    attn = torch.softmax(torch.bmm(q * (1.0 / math.sqrt(hd)), k.transpose(1, 2)), dim=-1)
    out = torch.bmm(attn, v).transpose(0, 1).reshape(L, B, D)
    return F.linear(out, sd[prefix + "out_proj.weight"], sd[prefix + "out_proj.bias"])


def feed_forward(sd, prefix, x):
    """linear2(gelu(linear1(x))), exact-erf GELU (model/sublayers.py:373-375, :16)."""
    return F.linear(F.gelu(F.linear(x, sd[prefix + "linear1.weight"], sd[prefix + "linear1.bias"])),
                    sd[prefix + "linear2.weight"], sd[prefix + "linear2.bias"])


def normalize_queries(queries, nhead):
    """_normalize_and_reshape_query(unit_norm=True, depth_scale=True)
    (model/sublayers.py:18-35): per-head L2 normalisation (+1e-6) then / sqrt(head_dim)."""
    n, D = queries.shape
    q = queries.reshape(n, nhead, D // nhead)
    q = q / (torch.norm(q, dim=-1, keepdim=True) + 1e-6)
    q = q / math.sqrt(D // nhead)
    return q.reshape(n, D)


def qa_block_faithful(sd, prefix, x, nhead, rotary=None):
    """TransformerDecoderLayerQaN._qa_block (model/sublayers.py:343-352) exactly as the
    reference executes it: 10x replicated input, LocalAttention without projections,
    combine with wk.  x: (T,B,D)."""
    queries, wk = sd[prefix + "queries"], sd[prefix + "wk"]
    N = queries.shape[0]
    T, B, D = x.shape
    q = normalize_queries(queries, nhead)
    q = q.unsqueeze(0).unsqueeze(2).repeat(B, 1, T, 1).contiguous()  # B,N,T,D  (:295-304)
    xr = x.unsqueeze(0).repeat(N, 1, 1, 1).permute(2, 0, 1, 3).contiguous()  # B,N,T,D
    attn = LocalAttention(dim=D, window_size=1, causal=False, look_backward=1, look_forward=1,
                          dropout=0.0, exact_windowsize=False, autopad=True, rotary=rotary)
    mask = torch.ones(1, T).bool()
    y = attn(q.view(B * N, T, D), xr.view(B * N, T, D), xr.view(B * N, T, D), mask=mask).view(B, N, T, D)
    y = torch.einsum("bntd,nk->bktd", y, wk).squeeze(1).permute(1, 0, 2).contiguous()
    return y


ROTARY_OFFSETS = {"absolute": (1.0, 0.0, -1.0), "bucketed": (2.0, 1.0, 0.0)}  # q_pos - k_pos for key slots (t-1, t, t+1)


def qan_folded_queries(queries, nhead, rotary=None):
    """Algebraic form (SURVEY 8a note for A5): logits[t, n, slot] = x[t+slot-1] . Qt[slot, n]
    with Qt[slot, n] = R(-o_slot)^T-rotated, 1/16-scaled normalised query.  Returns
    (3, N, D) float32."""
    rotary = rotary or DEFAULT_ROTARY
    n, D = queries.shape
    q = normalize_queries(queries, nhead) * (D ** -0.5)
    inv_freq = (1.0 / (10000 ** (torch.arange(0, D, 2).float() / D))).to(q.dtype)
    out = []
    for o in ROTARY_OFFSETS[rotary]:
        # <R(a) q, R(b) k> = <R(a-b) q, k> = <q rotated by o = q_pos - k_pos, k>
        f = torch.cat((o * inv_freq, o * inv_freq))
        d = D // 2
        rot = torch.cat((-q[:, d:], q[:, :d]), dim=-1)
        out.append(q * f.cos() + rot * f.sin())
    return torch.stack(out)


def qa_block_algebraic(sd, prefix, x, nhead, rotary=None):
    """Same function as qa_block_faithful, restructured as one [M x 256] x [256 x 30] product
    + masked 3-way softmax + wk-combine + 3-tap filter (what the CUDA kernel computes)."""
    queries, wk = sd[prefix + "queries"], sd[prefix + "wk"]
    T, B, D = x.shape
    Qt = qan_folded_queries(queries, nhead, rotary)  # (3,N,D)
    P = torch.einsum("tbd,snd->tbsn", x, Qt)  # P[t', b, slot, n] = x[t'] . Qt[slot,n]
    neg = -torch.finfo(x.dtype).max
    logits = torch.full((T, B, 3, Qt.shape[1]), neg, dtype=x.dtype)
    logits[1:, :, 0] = P[:-1, :, 0]      # key t-1
    logits[:, :, 1] = P[:, :, 1]         # key t
    logits[:-1, :, 2] = P[1:, :, 2]      # key t+1
    a = torch.softmax(logits, dim=2)
    c = torch.einsum("tbsn,n->tbs", a, wk[:, 0])
    y = c[:, :, 1:2] * x
    y[1:] += c[1:, :, 0:1] * x[:-1]
    y[:-1] += c[:-1, :, 2:3] * x[1:]
    return y


def decoder_layer_std(sd, prefix, tgt, memory, nhead):
    """torch.nn.TransformerDecoderLayer(post-norm, gelu, eval) = layers 0 and 7
    (model/diffusion_smpl.py:73-78,115-120)."""
    x = layer_norm(tgt + multihead_attention(sd, prefix + "self_attn.", tgt, tgt, nhead), sd, prefix + "norm1.")
    x = layer_norm(x + multihead_attention(sd, prefix + "multihead_attn.", x, memory, nhead), sd, prefix + "norm2.")
    x = layer_norm(x + feed_forward(sd, prefix, x), sd, prefix + "norm3.")
    return x


def decoder_layer_qan(sd, prefix, tgt, memory, nhead, rotary=None, faithful=True):
    """TransformerDecoderLayerQaN.forward, norm_first=False, stochastic_depth p=0
    (model/sublayers.py:311-341)."""
    qa = qa_block_faithful if faithful else qa_block_algebraic
    x = tgt.clone()
    x = layer_norm(x + qa(sd, prefix, x, nhead, rotary), sd, prefix + "norm1.")
    x = layer_norm(x + multihead_attention(sd, prefix + "multihead_attn.", x, memory, nhead), sd, prefix + "norm2.")
    x = layer_norm(x + feed_forward(sd, prefix, x), sd, prefix + "norm3.")
    return tgt + (x - tgt)


def decoder(sd, tgt, memory, nhead, rotary=None, faithful=True, prefix="decoder.layers."):
    """TransformerDecoder layer loop (model/layers.py:258-264): layers 0,7 standard, 1-6 QaN."""
    n_layers = 1 + max(int(k[len(prefix):].split(".")[0]) for k in sd if k.startswith(prefix))
    x = tgt
    for i in range(n_layers):
        p = "%s%d." % (prefix, i)
        if (p + "queries") in sd:
            x = decoder_layer_qan(sd, p, x, memory, nhead, rotary, faithful)
        else:
            x = decoder_layer_std(sd, p, x, memory, nhead)
    return x


def encoder_layer_std(sd, prefix, x, nhead):
    """torch.nn.TransformerEncoderLayer(post-norm, gelu, eval) = encoder layers 0 and 7
    (model/diffusion_smpl.py:20-25, 62-67)."""
    x = layer_norm(x + multihead_attention(sd, prefix + "self_attn.", x, x, nhead), sd, prefix + "norm1.")
    return layer_norm(x + feed_forward(sd, prefix, x), sd, prefix + "norm2.")


def encoder_layer_qan(sd, prefix, src, nhead, rotary=None, faithful=True):
    """TransformerEncoderLayerQaN.forward, norm_first=False, stochastic_depth p=0
    (model/sublayers.py:137-161)."""
    qa = qa_block_faithful if faithful else qa_block_algebraic
    x = src.clone()
    x = layer_norm(x + qa(sd, prefix, x, nhead, rotary), sd, prefix + "norm1.")
    x = layer_norm(x + feed_forward(sd, prefix, x), sd, prefix + "norm2.")
    return src + (x - src)


def encoder(sd, src, nhead, rotary=None, faithful=True, prefix="encoder.layers."):
    """TransformerEncoder layer loop without final norm (model/layers.py:195-214): layers 0,7 standard, 1-6 QaN."""
    n_layers = 1 + max(int(k[len(prefix):].split(".")[0]) for k in sd if k.startswith(prefix))
    x = src
    for i in range(n_layers):
        p = "%s%d." % (prefix, i)
        x = encoder_layer_qan(sd, p, x, nhead, rotary, faithful) if (p + "queries") in sd else encoder_layer_std(sd, p, x, nhead)
    return x


def mdm_smpl_condition(sd, past, pc_embedding, nhead=4, rotary=None, faithful=True):
    """The part of MDM._get_embeddings after the point-cloud encoder (model/diffusion_smpl.py:217-221):
    embedding of the PAST frames + point-cloud embedding + positional encoding -> 8-layer encoder.
    past: (B,1,C,Tp) = the first past_len frames of the motion tensor (channels [body | object]),
    pc_embedding: (B,D) = pcEmbedding(...).view(1,B,-1)[0].  Returns cond (Tp,B,D)."""
    xs = past.squeeze(1).permute(2, 0, 1).contiguous()  # (Tp,B,C)
    nb = sd["bodyEmbedding.weight"].shape[1]
    emb = F.linear(xs[..., :nb], sd["bodyEmbedding.weight"], sd["bodyEmbedding.bias"]) \
        + F.linear(xs[..., nb:], sd["objEmbedding.weight"], sd["objEmbedding.bias"]) + pc_embedding[None]
    emb = emb + sd["PositionalEmbedding.pe"][: emb.shape[0]]
    return encoder(sd, emb, nhead, rotary, faithful)


def timestep_embed(sd, timesteps):
    """TimestepEmbedder.forward (model/layers.py:42-43): pe[t] -> Linear -> SiLU -> Linear,
    indexing the SAME sinusoid table as the positional encoding.  Returns (1,B,D)."""
    pe = sd["embedTimeStep.sequence_pos_encoder.pe"]
    h = F.linear(pe[timesteps], sd["embedTimeStep.time_embed.0.weight"], sd["embedTimeStep.time_embed.0.bias"])
    h = F.linear(F.silu(h), sd["embedTimeStep.time_embed.2.weight"], sd["embedTimeStep.time_embed.2.bias"])
    return h.permute(1, 0, 2)


def mdm_smpl_forward(sd, x, timesteps, cond, nhead=4, rotary=None, faithful=True):
    """MDM.forward/_decode for the SMPL model (model/diffusion_smpl.py:239-246, 226-237).
    x: (B,1,144,T), timesteps: (B,) long, cond: (Tm,B,D).  Returns (B,1,144,T)."""
    temb = timestep_embed(sd, timesteps)
    xs = x.squeeze(1).permute(2, 0, 1).contiguous()  # (T,B,C)
    nb = sd["bodyEmbedding.weight"].shape[1]
    body, obj = xs[..., :nb], xs[..., nb:]
    h = F.linear(body, sd["bodyEmbedding.weight"], sd["bodyEmbedding.bias"]) \
        + F.linear(obj, sd["objEmbedding.weight"], sd["objEmbedding.bias"]) + temb
    h = h + sd["PositionalEmbedding.pe"][: h.shape[0]]
    h = decoder(sd, h, cond, nhead, rotary, faithful)
    body = F.linear(h, sd["bodyFinalLinear.weight"], sd["bodyFinalLinear.bias"])
    obj = F.linear(h, sd["objFinalLinear.weight"], sd["objFinalLinear.bias"])
    pred = torch.cat([body, obj], dim=2)
    return pred.permute(1, 2, 0).unsqueeze(1).contiguous()


def skeleton_obj_from_pose(pose, zero_pose_obj):
    """MDM.calc_obj_pred (model/diffusion_skeleton.py:218-229): pose = [trans(3), quat xyzw];
    the quaternion is NOT normalised (two_s does it).  pose (T,B,7), zero_pose_obj (B,P,3)."""
    quat = torch.cat([pose[:, :, -1, None], pose[:, :, -4:-1]], dim=2)
    R = tf.quaternion_to_matrix(quat)[:, :, None]  # T,B,1,3,3
    p = zero_pose_obj[None, :, :, :, None]
    return (R.matmul(p) + pose[:, :, None, :3, None])[..., 0]


def mdm_skeleton_forward(sd, x, timesteps, zero_pose_obj, cond, nhead=4, rotary=None, faithful=True):
    """Skeleton MDM.forward/_decode (model/diffusion_skeleton.py:250-257, 231-248).
    x: (B,1,106,T) = 63 body + 36 object keypoints + 7 pose."""
    temb = timestep_embed(sd, timesteps)
    xs = x.squeeze(1).permute(2, 0, 1).contiguous()
    T, B, _ = xs.shape
    nb = sd["bodyEmbedding.weight"].shape[1]
    no = sd["objEmbedding.weight"].shape[1]
    body, obj = xs[..., :nb], xs[..., nb:nb + no]
    h = F.linear(body, sd["bodyEmbedding.weight"], sd["bodyEmbedding.bias"]) \
        + F.linear(obj, sd["objEmbedding.weight"], sd["objEmbedding.bias"]) + temb
    h = h + sd["PositionalEmbedding.pe"][:T]
    h = decoder(sd, h, cond, nhead, rotary, faithful)
    body = F.linear(h, sd["bodyFinalLinear.weight"], sd["bodyFinalLinear.bias"])
    pose = F.linear(h, sd["objFinalLinear.weight"], sd["objFinalLinear.bias"])
    obj = skeleton_obj_from_pose(pose, zero_pose_obj).reshape(T, B, -1)
    pred = torch.cat([body, obj, pose], dim=2)
    return pred.permute(1, 2, 0).unsqueeze(1).contiguous()


# ----------------------------------------------------------------------------------------
# A1/A2: diffusion process (ancestral DDPM, START_X, FIXED_SMALL)
# ----------------------------------------------------------------------------------------


def named_beta_schedule(name, n, scale=1.0):
    """get_named_beta_schedule / betas_for_alpha_bar (diffusion/gaussian_diffusion.py:20-64)."""
    if name == "linear":
        s = scale * 1000 / n
        return np.linspace(s * 0.0001, s * 0.02, n, dtype=np.float64)
    if name == "cosine":
        ab = lambda t: math.cos((t + 0.008) / 1.008 * math.pi / 2) ** 2
        return np.array([min(1 - ab((i + 1) / n) / ab(i / n), 0.999) for i in range(n)])
    raise NotImplementedError(name)


def diffusion_tables(betas):
    """Float64 coefficient tables of GaussianDiffusion.__init__ (gaussian_diffusion.py:160-197);
    SpacedDiffusion with use_timesteps = all steps re-derives the same betas (respace.py:64-87)."""
    betas = np.asarray(betas, dtype=np.float64)
    alphas = 1.0 - betas
    ac = np.cumprod(alphas, axis=0)
    ac_prev = np.append(1.0, ac[:-1])
    post_var = betas * (1.0 - ac_prev) / (1.0 - ac)
    return dict(
        betas=betas,
        alphas_cumprod=ac,
        sqrt_alphas_cumprod=np.sqrt(ac),
        sqrt_one_minus_alphas_cumprod=np.sqrt(1.0 - ac),
        posterior_variance=post_var,
        posterior_log_variance_clipped=np.log(np.append(post_var[1], post_var[1:])),
        posterior_mean_coef1=betas * np.sqrt(ac_prev) / (1.0 - ac),
        posterior_mean_coef2=(1.0 - ac_prev) * np.sqrt(alphas) / (1.0 - ac),
    )


def p_sample_step(model_fn, tables, x, i, noise, gt=None, mask=None, denoised_fn=None, model_kwargs=None,
                  clip_denoised=False):
    """One GaussianDiffusion.p_sample (gaussian_diffusion.py:496-548) for a uniform timestep i:
    model -> inpaint blend (:307-311) -> denoised_fn (:354-360) -> posterior mean (:253-275)
    -> mean + 1[t!=0] exp(0.5 logvar) noise (:532-547).  Coefficients: float64 table -> .float()
    exactly like _extract_into_tensor (:1611-1623).  Returns (sample, pred_xstart)."""
    B = x.shape[0]
    t = torch.full((B,), int(i), dtype=torch.long)
    out = model_fn(x, t)
    if mask is not None and gt is not None:
        out = (out * ~mask) + (gt * mask)
    if denoised_fn is not None:
        out = denoised_fn(out, t, model_kwargs)
    if clip_denoised:
        out = out.clamp(-1, 1)
    c1 = torch.tensor(tables["posterior_mean_coef1"][i]).float()
    c2 = torch.tensor(tables["posterior_mean_coef2"][i]).float()
    logvar = torch.tensor(tables["posterior_log_variance_clipped"][i]).float()
    mean = c1 * out + c2 * x
    nonzero = 0.0 if i == 0 else 1.0
    sample = mean + nonzero * torch.exp(0.5 * logvar) * noise
    return sample, out


def p_sample_loop(model_fn, tables, tape, gt=None, mask=None, denoised_fn=None, model_kwargs=None,
                  return_trajectory=False):
    """GaussianDiffusion.p_sample_loop(_progressive) with caller-provided initial noise
    (gaussian_diffusion.py:598-736; the eval scripts pass noise=, eval_smpl_short.py:152-153,
    so there is no initial inpaint blend).  tape[0] = x_T, tape[k] = eps of the k-th step."""
    n = len(tables["betas"])
    x = tape[0].clone()
    traj = []
    for k, i in enumerate(reversed(range(n))):
        x, x0 = p_sample_step(model_fn, tables, x, i, tape[k + 1], gt, mask, denoised_fn, model_kwargs)
        if return_trajectory:
            traj.append((x.clone(), x0.clone()))
    return (x, traj) if return_trajectory else x


# ----------------------------------------------------------------------------------------
# A6: SMPL-H linear blend skinning
# ----------------------------------------------------------------------------------------


def batch_rodrigues(aa):
    """rodrigues_layer.batch_rodrigues + quat2mat (libsmpl/smplpytorch/pytorch/
    rodrigues_layer.py:41-52, 13-38): angle = |aa + 1e-8|, quaternion route.  aa (N,3) -> (N,9)."""
    angle = torch.norm(aa + 1e-8, p=2, dim=1).unsqueeze(-1)
    n = aa / angle
    half = angle * 0.5
    quat = torch.cat([torch.cos(half), torch.sin(half) * n], dim=1)
    quat = quat / quat.norm(p=2, dim=1, keepdim=True)
    w, x, y, z = quat[:, 0], quat[:, 1], quat[:, 2], quat[:, 3]
    w2, x2, y2, z2 = w * w, x * x, y * y, z * z
    wx, wy, wz, xy, xz, yz = w * x, w * y, w * z, x * y, x * z, y * z
    return torch.stack([w2 + x2 - y2 - z2, 2 * xy - 2 * wz, 2 * wy + 2 * xz,
                        2 * wz + 2 * xy, w2 - x2 + y2 - z2, 2 * yz - 2 * wx,
                        2 * xz - 2 * wy, 2 * wx + 2 * yz, w2 - x2 - y2 + z2], dim=1)


def smplh_lbs(smplh, pose, betas, trans, scale=1.0):
    """SMPL_Layer.forward (libsmpl/smplpytorch/pytorch/smpl_layer.py:72-175), hands=True
    (52 joints), per-frame betas branch (:100-103), no root centring, + trans (:171-172).
    smplh: dict of tensors v_template (V,3), shapedirs (V,3,10), posedirs (V,3,459),
    J_regressor (52,V), weights (V,52), parents[52].  pose (F,156), betas (F,10), trans (F,3).
    Returns verts (F,V,3), jtr (F,52,3)."""
    Fn = pose.shape[0]
    J = len(smplh["parents"])
    dt = pose.dtype      # float32 as the reference; float64 gives the rounding-free yardstick for the precision tests
    R = batch_rodrigues(pose.reshape(Fn * J, 3)).reshape(Fn, J, 3, 3)
    pose_map = (R[:, 1:] - torch.eye(3, dtype=dt)).reshape(Fn, (J - 1) * 9)  # subtract_flat_id (tensutils.py:41-53)
    v_shaped = smplh["v_template"].unsqueeze(0) + torch.matmul(smplh["shapedirs"], betas.transpose(1, 0)).permute(2, 0, 1)
    jrest = torch.matmul(smplh["J_regressor"], v_shaped)  # (F,52,3)
    v_posed = v_shaped + torch.matmul(smplh["posedirs"], pose_map.transpose(0, 1)).permute(2, 0, 1)
    parents = [int(p) for p in smplh["parents"]]
    bottom = torch.tensor([0.0, 0.0, 0.0, 1.0], dtype=dt).view(1, 1, 4).repeat(Fn, 1, 1)
    G = [torch.cat([torch.cat([R[:, 0], jrest[:, 0].unsqueeze(2)], 2), bottom], 1)]
    for i in range(1, J):
        rel = torch.cat([torch.cat([R[:, i], (jrest[:, i] - jrest[:, parents[i]]).unsqueeze(2)], 2), bottom], 1)
        G.append(torch.matmul(G[parents[i]], rel))
    A = torch.zeros(Fn, 4, 4, J, dtype=dt)
    for i in range(J):
        jh = torch.cat([jrest[:, i], torch.zeros(Fn, 1, dtype=dt)], 1)
        tmp = torch.bmm(G[i], jh.unsqueeze(2))  # (F,4,1)
        A[:, :, :, i] = G[i] - torch.cat([torch.zeros(Fn, 4, 3, dtype=dt), tmp], 2)
    Tm = torch.matmul(A, smplh["weights"].transpose(0, 1))  # (F,4,4,V)
    vh = torch.cat([v_posed.transpose(2, 1), torch.ones(Fn, 1, v_posed.shape[1], dtype=dt)], 1)  # (F,4,V)
    verts = (Tm * vh.unsqueeze(1)).sum(2).transpose(2, 1)[:, :, :3]
    jtr = torch.stack(G, dim=1)[:, :, :3, 3]
    verts = verts * scale + trans.unsqueeze(1)
    jtr = jtr * scale + trans.unsqueeze(1)
    return verts, jtr


# ----------------------------------------------------------------------------------------
# A8/A9: geometry helpers
# ----------------------------------------------------------------------------------------


def vertex_normals(vertices, faces):
    """data/tools.py:4-39: area-weighted vertex normals via three index_add_ of face cross
    products, F.normalize(eps=1e-6).  vertices (N,V,3), faces (Fc,3) shared by all frames."""
    N, V = vertices.shape[:2]
    f = faces.long()
    v0, v1, v2 = vertices[:, f[:, 0]], vertices[:, f[:, 1]], vertices[:, f[:, 2]]
    normals = torch.zeros(N, V, 3)
    normals.index_add_(1, f[:, 1], torch.cross(v2 - v1, v0 - v1, dim=-1))
    normals.index_add_(1, f[:, 2], torch.cross(v0 - v2, v1 - v2, dim=-1))
    normals.index_add_(1, f[:, 0], torch.cross(v1 - v0, v2 - v0, dim=-1))
    return F.normalize(normals, eps=1e-6, dim=2)


def nearest_index(x, y, chunk=512):
    """chamfer_distance argmin (tools.py:45-47; third-party CUDA ext, PARITY UNPINNED):
    idx[n,i] = first argmin_j of (dx*dx + dy*dy) + dz*dz evaluated in fp32 without FMA."""
    N, P1, _ = x.shape
    out = torch.empty(N, P1, dtype=torch.long)
    for n in range(N):
        yx, yy, yz = y[n, :, 0][None], y[n, :, 1][None], y[n, :, 2][None]
        for s in range(0, P1, chunk):
            dx = x[n, s:s + chunk, 0:1] - yx
            dy = x[n, s:s + chunk, 1:2] - yy
            dz = x[n, s:s + chunk, 2:3] - yz
            d = (dx * dx + dy * dy) + dz * dz
            out[n, s:s + chunk] = d.argmin(dim=1)
    return out


def point2point_signed(x, y, x_normals):
    """tools.py:11-76 with x_normals given, y_normals None, return_vector=True.
    Returns y2x_signed (N,P2), x2y_signed (N,P1), yidx_near (N,P2), xidx_near (N,P1), y2x, x2y."""
    N, P1, D = x.shape
    P2 = y.shape[1]
    xidx = nearest_index(x, y)
    yidx = nearest_index(y, x)
    x_near = y.gather(1, xidx.view(N, P1, 1).expand(N, P1, D))
    y_near = x.gather(1, yidx.view(N, P2, 1).expand(N, P2, D))
    x2y = x - x_near
    y2x = y - y_near
    y_nn = x_normals.gather(1, yidx.view(N, P2, 1).expand(N, P2, D))
    in_out = torch.bmm(y_nn.view(-1, 1, 3), y2x.view(-1, 3, 1)).view(N, -1).sign()
    y2x_signed = y2x.norm(dim=2) * in_out
    x2y_signed = x2y.norm(dim=2)
    return y2x_signed, x2y_signed, yidx, xidx, y2x, x2y


# ----------------------------------------------------------------------------------------
# A10: ObjProjector (correction network)
# ----------------------------------------------------------------------------------------

MARKERSET_SSM67_SMPLH = [3470, 3171, 3327, 857, 1812, 628, 182, 3116, 3040, 239,
                         1666, 1725, 0, 2174, 1568, 1368, 3387, 2112, 1053, 1058,
                         3336, 3346, 1323, 2108, 3122, 3314, 1252, 1082, 1861, 1454,
                         850, 2224, 3233, 1769, 6728, 4343, 5273, 4116, 3694, 6399,
                         6540, 6488, 3749, 5135, 5194, 3512, 5635, 5210, 4360, 4841,
                         6786, 5573, 4538, 4544, 6736, 6747, 4804, 5568, 6544, 6682,
                         5322, 4927, 5686, 4598, 6633, 3506, 3508]  # data/utils.py:232-238
HAND_MARKERS = [10, 11, 14, 31, 13, 17, 23, 28, 27] + [60, 43, 44, 47, 62, 46, 51, 57]  # data/utils.py:252-253


def dct_matrices(N):
    """ObjProjector.get_dct_matrix (model/correction_smpl.py:55-67), float64."""
    dct_m = np.eye(N)
    for k in range(N):
        for i in range(N):
            w = np.sqrt(2 / N) if k != 0 else np.sqrt(1 / N)
            dct_m[k, i] = w * np.cos(np.pi * (i + 1 / 2) * k / N)
    return dct_m, np.linalg.inv(dct_m)


def _bn_eval(x, sd, p, eps=1e-5):
    shp = (1, -1, 1, 1)
    return (x - sd[p + "running_mean"].view(shp)) / torch.sqrt(sd[p + "running_var"].view(shp) + eps) \
        * sd[p + "weight"].view(shp) + sd[p + "bias"].view(shp)


def st_gcnn_layer(sd, p, x):
    """ST_GCNN_layer.forward (model/layers.py:338-345) in eval mode; gcn version inferred from
    the parameters present: version 0 = ConvTemporalGraphical (sublayers.py:414-419),
    version 2 = ConvSpatialTemporalGraphical (sublayers.py:510-515).  x: (N,C,T,V)."""
    if (p + "residual.0.weight") in sd:
        res = F.conv2d(x, sd[p + "residual.0.weight"], sd[p + "residual.0.bias"])
        res = _bn_eval(res, sd, p + "residual.1.")
    else:
        res = x
    Tm = sd[p + "gcn.T"]
    if Tm.dim() == 2:
        x = torch.einsum("nctv,tq->ncqv", x, Tm)
    else:
        x = torch.einsum("nctv,vtq->ncqv", x, Tm)
        x = torch.einsum("nctv,tvw->nctw", x, sd[p + "gcn.A"])
    x = F.conv2d(x.contiguous(), sd[p + "tcn.0.weight"], sd[p + "tcn.0.bias"])
    x = _bn_eval(x, sd, p + "tcn.1.")
    x = x + res
    return F.prelu(x, sd[p + "prelu.weight"])


def obj_projector_sample(sd, obj_angles, obj_trans, human_verts, contact, past_len, future_len, n_pre=10):
    """ObjProjector.sample, eval mode, initialize=False (model/correction_smpl.py:79-138).
    obj_angles (T,B,6), obj_trans (T,B,3), human_verts (T,B,67,>=3), contact (B,67)."""
    human_verts = human_verts[:, :, :, :3]
    T0 = past_len + future_len
    dct_m, idct_m = dct_matrices(T0)
    dct_m, idct_m = torch.from_numpy(dct_m).float(), torch.from_numpy(idct_m).float()
    idx_pad = list(range(past_len)) + [past_len - 1] * future_len
    rel_t = obj_trans.unsqueeze(2) - human_verts
    obj_rel = torch.cat([obj_angles.unsqueeze(2).repeat(1, 1, rel_t.shape[2], 1), rel_t], dim=3)[idx_pad]
    T, B, P, C = obj_rel.shape
    obj_rel = obj_rel.permute(1, 0, 3, 2).contiguous().view(B, T, C * P)
    obj_rel = torch.matmul(dct_m[:n_pre], obj_rel).view(B, -1, C, P).permute(0, 2, 1, 3).contiguous()
    x = obj_rel.clone()
    for i in range(4):
        x = st_gcnn_layer(sd, "st_gcnns_relative.%d." % i, x)
    obj_rel = obj_rel + x
    human_trans = human_verts.permute(1, 0, 3, 2).contiguous().view(B, T, -1)
    human_trans = torch.matmul(dct_m[:n_pre], human_trans).view(B, -1, 3, P).permute(0, 2, 1, 3).contiguous()
    obj_multi = torch.cat([obj_rel[:, :6], obj_rel[:, 6:9] + human_trans], dim=1)
    obj_gt = torch.cat([obj_angles, obj_trans], dim=2)
    obj = obj_gt[idx_pad].unsqueeze(2).permute(1, 0, 3, 2).contiguous().view(B, T, C)
    obj = torch.matmul(dct_m[:n_pre], obj).view(B, -1, C, 1).permute(0, 2, 1, 3).contiguous()
    x = obj.clone()
    for i in range(4):
        x = st_gcnn_layer(sd, "st_gcnns.%d." % i, x)
    obj = obj + x
    obj = torch.cat([obj, obj_multi], dim=3)
    x = obj.clone()
    for i in range(4):
        x = st_gcnn_layer(sd, "st_gcnns_all.%d." % i, x)
    obj = obj + x
    obj = obj.permute(0, 2, 1, 3).contiguous().view(B, -1, C * (P + 1))
    results = torch.matmul(idct_m[:, :n_pre], obj).view(B, T, C, P + 1).permute(1, 0, 3, 2)[:, :, :, :9]
    final = torch.zeros(T, B, 9)
    csum = contact.sum(dim=1)
    final[:, csum == 0] = results[:, csum == 0, 0, :]
    happen = contact[csum > 0].float()
    happen[:, HAND_MARKERS] = happen[:, HAND_MARKERS] + 0.5
    rch = results[:, csum > 0, 1:, :]
    idx = torch.argmax(happen, dim=1, keepdim=True).unsqueeze(0).unsqueeze(3).repeat(T, 1, 1, 9)
    final[:, csum > 0] = torch.gather(rch, 2, idx).squeeze(2)
    return final


def obj_projector_skeleton_sample(sd, obj_angles, obj_trans, human_points, past_len, future_len, n_pre=20):
    """Skeleton correction net, ObjProjector.sample in eval mode (model/correction_skeleton.py:84-135; SURVEY 8f rank 4,
    oracle only so far).  obj_angles (T,B,4) quaternion xyzw, obj_trans (T,B,3), human_points (T,B,J,3)
    -> (obj_angles_p (T,B,4) xyzw, obj_trans_p (T,B,3))."""
    quat = torch.cat([obj_angles[:, :, -1, None], obj_angles[:, :, -4:-1]], dim=2)
    ang6 = tf.matrix_to_rotation_6d(tf.quaternion_to_matrix(quat))
    T0 = past_len + future_len
    dct_m, idct_m = dct_matrices(T0)
    dct_m, idct_m = torch.from_numpy(dct_m).float(), torch.from_numpy(idct_m).float()
    idx_pad = list(range(past_len)) + [past_len - 1] * future_len
    rel_t = obj_trans.unsqueeze(2) - human_points
    obj_rel = torch.cat([ang6.unsqueeze(2).repeat(1, 1, rel_t.shape[2], 1), rel_t], dim=3)[idx_pad]
    T, B, P, C = obj_rel.shape
    obj_rel = obj_rel.permute(1, 0, 3, 2).contiguous().view(B, T, C * P)
    obj_rel = torch.matmul(dct_m[:n_pre], obj_rel).view(B, -1, C, P).permute(0, 2, 1, 3).contiguous()
    x = obj_rel.clone()
    for i in range(4):
        x = st_gcnn_layer(sd, "st_gcnns_relative.%d." % i, x)
    obj_rel = obj_rel + x
    human_trans = human_points.permute(1, 0, 3, 2).contiguous().view(B, T, -1)
    human_trans = torch.matmul(dct_m[:n_pre], human_trans).view(B, -1, 3, P).permute(0, 2, 1, 3).contiguous()
    obj_multi = torch.cat([obj_rel[:, :6], obj_rel[:, 6:9] + human_trans], dim=1)
    obj = torch.cat([ang6, obj_trans], dim=2)[idx_pad].unsqueeze(2).permute(1, 0, 3, 2).contiguous().view(B, T, C)
    obj = torch.matmul(dct_m[:n_pre], obj).view(B, -1, C, 1).permute(0, 2, 1, 3).contiguous()
    x = obj.clone()
    for i in range(4):
        x = st_gcnn_layer(sd, "st_gcnns.%d." % i, x)
    obj = torch.cat([obj + x, obj_multi], dim=3)
    x = obj.clone()
    for i in range(4):
        x = st_gcnn_layer(sd, "st_gcnns_all.%d." % i, x)
    obj = (obj + x).permute(0, 2, 1, 3).contiguous().view(B, -1, C * (P + 1))
    results = torch.matmul(idct_m[:, :n_pre], obj).view(B, T, C, P + 1).permute(1, 0, 3, 2)[:, :, 0, :9]
    q = tf.matrix_to_quaternion(tf.rotation_6d_to_matrix(results[:, :, :6]))
    return torch.cat([q[:, :, 1:4], q[:, :, 0, None]], dim=2), results[:, :, 6:9]


# ----------------------------------------------------------------------------------------
# A7: the correction hook (denoised_fn of eval_smpl_short.py:84-130)
# ----------------------------------------------------------------------------------------


def correction_observables(x, ctx):
    """The geometry half of denoised_fn (eval_smpl_short.py:87-125): returns a dict with
    markers (T,B,67,3), o2h_signed (T*B,2048), condition (B,) bool, contact (B,67) long, and the
    intermediates (verts, normals, obj_points_pred, nn indices)."""
    past_len, nb = ctx["past_len"], ctx["smpl_dim"] + 3
    xs = x.squeeze(1).permute(2, 0, 1).contiguous()
    body, obj = xs[..., :nb], xs[..., nb:]
    T, B, _ = body[:, :, :-3].shape
    obj_R = tf.rotation_6d_to_matrix(obj[:, :, :-3].reshape(T, B, 6))
    body_rot = tf.matrix_to_axis_angle(tf.rotation_6d_to_matrix(body[:, :, :-3].reshape(T, B, -1, 6))).reshape(T, B, -1)
    body_pred = torch.cat([body_rot, ctx["hand_pose"], body[:, :, -3:]], dim=2).reshape(T * B, -1)
    verts, jtr = smplh_lbs(ctx["smplh"], body_pred[:, :-3], ctx["betas"].reshape(T * B, -1), body_pred[:, -3:])
    markers = verts[:, MARKERSET_SSM67_SMPLH].view(T, B, -1, 3)
    obj_pts = torch.matmul(ctx["obj_points"].unsqueeze(0), obj_R.permute(0, 1, 3, 2)) + obj[:, :, -3:].unsqueeze(2)
    normals = vertex_normals(verts, ctx["smplh"]["faces"])
    o2h_signed, h2o_signed, o2h_idx, h2o_idx, o2h, h2o = point2point_signed(verts, obj_pts.view(T * B, -1, 3), normals)
    w = torch.zeros(T * B, o2h_signed.size(1))
    w[o2h_signed < 0] = 20
    loss_dist_o = (torch.abs(o2h_signed) * w).view(T, B, -1)
    # marker <-> object distances, chunked over frames (the reference materialises (T,B,2048,67,3))
    dmin = torch.empty(T, B)
    contact_lbl = torch.empty(T, B, markers.shape[2], dtype=torch.bool)
    for t in range(T):
        d = torch.norm(markers[t].unsqueeze(1) - obj_pts[t].unsqueeze(2), dim=3)  # (B,2048,67)
        dmin[t] = d.min(dim=2)[0].min(dim=1)[0]
        contact_lbl[t] = (d < 0.02).any(dim=1)
    distance = dmin.mean(dim=0)
    pen = loss_dist_o[past_len:].mean(dim=2).mean(dim=0)
    condition = torch.logical_not(torch.logical_and(pen < 0.002, distance < 0.02))
    contact = contact_lbl[past_len:].sum(dim=0)
    return dict(markers=markers, verts=verts, jtr=jtr, normals=normals, obj_points_pred=obj_pts,
                o2h_signed=o2h_signed, o2h_idx=o2h_idx, h2o_idx=h2o_idx, penetration=pen, distance=distance,
                condition=condition, contact=contact)


def make_denoised_fn(ctx):
    """Returns denoised_fn(x, t, model_kwargs) following eval_smpl_short.py:84-130.
    ctx keys: past_len, future_len, smpl_dim (132), gt (B,1,144,T), hand_pose (T,B,90),
    betas (T,B,10), obj_points (B,P,3), smplh (dict of tensors), projector (state dict)."""
    def denoised_fn(x, t, model_kwargs=None):
        if t[0] > 500 or t[0] % 50 != 0:
            return x
        obs = correction_observables(x, ctx)
        nb = ctx["smpl_dim"] + 3
        xs = x.squeeze(1).permute(2, 0, 1).contiguous()
        body = xs[..., :nb]
        gts = ctx["gt"].squeeze(1).permute(2, 0, 1).contiguous()
        obj_gt = gts[..., nb:]
        obj_proj = obj_projector_sample(ctx["projector"], obj_gt[:, :, :-3], obj_gt[:, :, -3:], obs["markers"],
                                        obs["contact"], ctx["past_len"], ctx["future_len"])
        x_ = torch.cat([body, obj_proj], dim=2).permute(1, 2, 0).unsqueeze(1).contiguous()
        x_ = t[0] / 1000 * x + (1 - t[0] / 1000) * x_
        x[obs["condition"]] = x_[obs["condition"]]
        return x
    return denoised_fn


def sample_postprocess(sample, ctx):
    """The tail of sample_once(_proj) (eval_smpl_short.py:154-173): 6D -> axis-angle, SMPL-H
    LBS on all T*B frames.  Returns body_pose (T,B,159), obj_pose (T,B,6), verts, jtr."""
    nb = ctx["smpl_dim"] + 3
    xs = sample.squeeze(1).permute(2, 0, 1).contiguous()
    body, obj = xs[..., :nb], xs[..., nb:]
    T, B, _ = body.shape
    body_rot = tf.matrix_to_axis_angle(tf.rotation_6d_to_matrix(body[:, :, :-3].reshape(T, B, -1, 6))).reshape(T, B, -1)
    obj_rot = tf.matrix_to_axis_angle(tf.rotation_6d_to_matrix(obj[:, :, :-3].reshape(T, B, 6))).reshape(T, B, -1)
    body_pred = torch.cat([body_rot, ctx["hand_pose"], body[:, :, -3:]], dim=2)
    bb = body_pred.reshape(T * B, -1)
    verts, jtr = smplh_lbs(ctx["smplh"], bb[:, :-3], ctx["betas"].reshape(T * B, -1), bb[:, -3:])
    return body_pred, torch.cat([obj_rot, obj[:, :, -3:]], dim=2), verts.view(T, B, -1, 3), jtr.view(T, B, -1, 3)


def metrics(obj_pred, body_jtr, body, obj_gt, body_jtr_gt, body_gt, verts, faces, obj_points):
    """eval_smpl_short.py:24-81 restated: per-sample evaluation metrics over the T predicted frames.
    obj_pred/obj_gt (T,B,6) = [axis-angle | translation], body_jtr(_gt) (T,B,J,3), body(_gt) (T,B,Db) with the
    translation in the last 3 channels, verts (T,B,V,3), faces (F,3) long, obj_points (B,P,3).
    Returns dict of (B,) tensors: global_mpjpe, local_mpjpe, body_translation, obj_translation, obj_rot_error, penetrate."""
    T, B = body_jtr_gt.shape[:2]
    Rm = tf.axis_angle_to_matrix(obj_pred[:, :, :3])
    pts = torch.matmul(obj_points.unsqueeze(0), Rm.permute(0, 1, 3, 2)) + obj_pred[:, :, 3:].unsqueeze(2)
    v = verts.reshape(T * B, -1, 3)
    normals = vertex_normals(v, faces)
    o2h = point2point_signed(v, pts.reshape(T * B, -1, 3), normals)[0]
    out = dict(penetrate=(o2h < 0).view(T, B, -1).float().mean(dim=2).mean(dim=0))
    out["global_mpjpe"] = (body_jtr - body_jtr_gt).norm(dim=3).mean(dim=2).mean(dim=0)
    out["local_mpjpe"] = ((body_jtr - body_jtr[:, :, 0:1]) - (body_jtr_gt - body_jtr_gt[:, :, 0:1])).norm(dim=3).mean(dim=2).mean(dim=0)
    out["body_translation"] = (body[:, :, -3:] - body_gt[:, :, -3:]).norm(dim=2).mean(dim=0)
    out["obj_translation"] = (obj_pred[:, :, -3:] - obj_gt[:, :, -3:]).norm(dim=2).mean(dim=0)
    q, qg = tf.axis_angle_to_quaternion(obj_pred[:, :, :3]), tf.axis_angle_to_quaternion(obj_gt[:, :, :3])
    out["obj_rot_error"] = torch.minimum((q - qg).norm(dim=2, p=1), (q + qg).norm(dim=2, p=1)).mean(dim=0)
    return out


# ----------------------------------------------------------------------------------------
# 8f rank 2: the step between two windows of the autoregressive rollout (eval_smpl_long.py:26-84, :247-285)
# ----------------------------------------------------------------------------------------


def rollout_next_window(body, obj, jtr, T, past_len):
    """Restated INTENT of get_batch (eval_smpl_long.py:26-84) followed by MDM._get_embeddings' gt assembly
    (model/diffusion_smpl.py:195-214) - PARITY UNPINNED: upstream get_batch raises for every batch size
    (`.unsqueeze(0).repeat(B, 1)` on a (B,3) tensor, :46) and `denormalize` / `correct` (:278, :285) are undefined.
    What the function visibly means: `rotation` stays the identity (:39-40), `centroid` = pelvis of the first of the last
    past_len frames (:38), translations of body and object are taken relative to it (:43-46, :58-59), rotations are
    unchanged (:52-55, :60-64), the future_len inputs repeat the last past frame (:78).
    body (Tw,B,159) = [66 axis-angle | 90 hand | 3 trans], obj (Tw,B,6) = [axis-angle | trans], jtr (Tw,B,J,3).
    Returns gt (B,1,144,T) and centroid (B,3); `denormalize` = add the centroid back."""
    P = past_len
    b, o, pel = body[-P:], obj[-P:], jtr[-P:, :, 0]
    B = b.shape[1]
    centroid = pel[0]
    r6 = lambda aa: tf.matrix_to_rotation_6d(tf.axis_angle_to_matrix(aa))
    frames = torch.cat([r6(b[..., :66].reshape(P, B, 22, 3)).reshape(P, B, 132), b[..., -3:] - centroid,
                        r6(o[..., :3].reshape(P, B, 1, 3)).reshape(P, B, 6), o[..., 3:6] - centroid], dim=2)
    frames = torch.cat([frames, frames[-1:].repeat(T - P, 1, 1)], dim=0)
    return frames.permute(1, 2, 0).unsqueeze(1).contiguous(), centroid


def make_denoised_fn_skeleton(ctx):
    """denoised_fn of eval_skeleton.py:80-111 restated.  ctx: gt (B,1,106,T), zero_pose_obj (B,12,3), projector (state dict of the
    skeleton correction net), past_len, future_len.  (body_obj_to_contact (:96) is evaluated upstream but its result is unused.)"""
    def denoised_fn(x, t, model_kwargs=None):
        if t[0] > 500 or t[0] % 50 != 0:
            return x
        xs = x.squeeze(1).permute(2, 0, 1).contiguous()
        body_pred = xs[..., :63]
        gts = ctx["gt"].squeeze(1).permute(2, 0, 1).contiguous()
        pose_gt = gts[..., 99:106]
        T, B, _ = body_pred.shape
        q, tr = obj_projector_skeleton_sample(ctx["projector"], pose_gt[..., 3:7], pose_gt[..., :3], body_pred.reshape(T, B, -1, 3),
                                              ctx["past_len"], ctx["future_len"])
        pose_proj = torch.cat([tr, q], dim=2)
        obj_proj = skeleton_obj_from_pose(pose_proj, ctx["zero_pose_obj"]).reshape(T, B, -1)
        x_ = torch.cat([body_pred, obj_proj, pose_proj], dim=2).permute(1, 2, 0).unsqueeze(1).contiguous()
        return t[0] / 1000 * x + (1 - t[0] / 1000) * x_
    return denoised_fn
