"""Parameter-name/shape tables of the reference's hot-path modules (state_dict names without the
'model.' prefix), used for seeded random-init weights (no network for checkpoints) and for
exporting/loading real weights.  Names follow reference checkpoints/diffusion.ckpt,
diffusion_skeleton.ckpt and correction.ckpt (SURVEY.md section 8b)."""
import os

import numpy as np

from . import synthetic


def decoder_layer_shapes(prefix, qan, D=256, F=1024, N=10):
    s = {}
    if qan:
        s[prefix + "queries"] = (N, D)
        s[prefix + "wk"] = (N, 1)
        s[prefix + "self_attn.rel_pos.inv_freq"] = (D // 2,)
    else:
        s[prefix + "self_attn.in_proj_weight"] = (3 * D, D)
        s[prefix + "self_attn.in_proj_bias"] = (3 * D,)
        s[prefix + "self_attn.out_proj.weight"] = (D, D)
        s[prefix + "self_attn.out_proj.bias"] = (D,)
    s[prefix + "multihead_attn.in_proj_weight"] = (3 * D, D)
    s[prefix + "multihead_attn.in_proj_bias"] = (3 * D,)
    s[prefix + "multihead_attn.out_proj.weight"] = (D, D)
    s[prefix + "multihead_attn.out_proj.bias"] = (D,)
    s[prefix + "linear1.weight"] = (F, D)
    s[prefix + "linear1.bias"] = (F,)
    s[prefix + "linear2.weight"] = (D, F)
    s[prefix + "linear2.bias"] = (D,)
    for i in (1, 2, 3):
        s[prefix + "norm%d.weight" % i] = (D,)
        s[prefix + "norm%d.bias" % i] = (D,)
    return s


def mdm_hot_shapes(variant="smpl", D=256, F=None, n_layers=8, N=10, pe_rows=5000):
    """Tensors the sampling hot path reads (decoder + embeddings + heads + timestep MLP + pe)."""
    if variant == "smpl":
        c_body, c_obj, c_head2 = 135, 9, 9
        F = F or 1024
    else:
        c_body, c_obj, c_head2 = 63, 36, 7
        F = F or 256
    s = {
        "bodyEmbedding.weight": (D, c_body), "bodyEmbedding.bias": (D,),
        "objEmbedding.weight": (D, c_obj), "objEmbedding.bias": (D,),
        "PositionalEmbedding.pe": (pe_rows, 1, D),
        "embedTimeStep.sequence_pos_encoder.pe": (pe_rows, 1, D),
        "embedTimeStep.time_embed.0.weight": (D, D), "embedTimeStep.time_embed.0.bias": (D,),
        "embedTimeStep.time_embed.2.weight": (D, D), "embedTimeStep.time_embed.2.bias": (D,),
        "bodyFinalLinear.weight": (c_body, D), "bodyFinalLinear.bias": (c_body,),
        "objFinalLinear.weight": (c_head2, D), "objFinalLinear.bias": (c_head2,),
    }
    for l in range(n_layers):
        s.update(decoder_layer_shapes("decoder.layers.%d." % l, qan=0 < l < n_layers - 1, D=D, F=F, N=N))
    return s


def mdm_encoder_shapes(variant="smpl", D=256, F=None, n_layers=8, N=10):
    """Tensors of the conditioning encoder (MDM.encoder, model/diffusion_smpl.py:20-70): like the decoder
    layers without the cross-attention block and norm3."""
    F = F or (1024 if variant == "smpl" else 256)
    s = {}
    for l in range(n_layers):
        d = decoder_layer_shapes("encoder.layers.%d." % l, qan=0 < l < n_layers - 1, D=D, F=F, N=N)
        s.update({k: v for k, v in d.items() if "multihead_attn" not in k and "norm3" not in k})
    return s


def mdm_skeleton_encoder_shapes(D=256, F=256, n_layers=8, N=10, n_points=12):
    """Conditioning path of the skeleton model (model/diffusion_skeleton.py:194-215): the 8 encoder layers (d_ff 256) and
    shapeEmbedding, the Linear on the flattened canonical object keypoints."""
    s = mdm_encoder_shapes("skeleton", D=D, F=F, n_layers=n_layers, N=N)
    s["shapeEmbedding.weight"] = (D, 3 * n_points)
    s["shapeEmbedding.bias"] = (D,)
    return s


def pointnet_shapes(prefix="pcEmbedding."):
    """PointNet2Encoder(c_in=1, c_out=256, num_keypoints=1) (model/layers.py:111-141): two MSG set-abstraction
    modules (Conv2d 1x1 without bias + BatchNorm2d + ReLU, three times per scale) and the Linear head."""
    s = {}
    for m, specs in enumerate(([[4, 16, 16, 32], [4, 32, 32, 64]], [[99, 64, 64, 128], [99, 64, 96, 128]])):
        for k, spec in enumerate(specs):
            for l in range(3):
                p = "%sSA_modules.%d.mlps.%d." % (prefix, m, k)
                s[p + "%d.weight" % (3 * l)] = (spec[l + 1], spec[l], 1, 1)
                for leaf in ("weight", "bias", "running_mean", "running_var"):
                    s[p + "%d.%s" % (3 * l + 1, leaf)] = (spec[l + 1],)
    s[prefix + "Linear.weight"] = (253, 256)
    s[prefix + "Linear.bias"] = (253,)
    return s


def projector_shapes(P=67, n_pre=10):
    s = {}
    chans = [9, 32, 16, 32, 9]
    for stack, nodes, ver in (("st_gcnns_relative", P, 0), ("st_gcnns", 1, 0), ("st_gcnns_all", P + 1, 2)):
        for i in range(4):
            p = "%s.%d." % (stack, i)
            cin, cout = chans[i], chans[i + 1]
            if ver == 0:
                s[p + "gcn.T"] = (n_pre, n_pre)
            else:
                s[p + "gcn.A"] = (n_pre, nodes, nodes)
                s[p + "gcn.T"] = (nodes, n_pre, n_pre)
            for blk in ("tcn", "residual"):
                s[p + blk + ".0.weight"] = (cout, cin, 1, 1)
                s[p + blk + ".0.bias"] = (cout,)
                for leaf in ("weight", "bias", "running_mean", "running_var"):
                    s[p + blk + ".1." + leaf] = (cout,)
            s[p + "prelu.weight"] = (1,)
    return s


def projector_skeleton_shapes(P=21, n_pre=20):
    """skeleton correction net (reference model/correction_skeleton.py:13-50): joint stack 9-64-32-64-9"""
    s = {}
    for stack, nodes, ver, chans in (("st_gcnns_relative", P, 0, [9, 32, 16, 32, 9]), ("st_gcnns", 1, 0, [9, 32, 16, 32, 9]),
                                     ("st_gcnns_all", P + 1, 2, [9, 64, 32, 64, 9])):
        for i in range(4):
            p = "%s.%d." % (stack, i)
            cin, cout = chans[i], chans[i + 1]
            if ver == 0:
                s[p + "gcn.T"] = (n_pre, n_pre)
            else:
                s[p + "gcn.A"] = (n_pre, nodes, nodes)
                s[p + "gcn.T"] = (nodes, n_pre, n_pre)
            for blk in ("tcn", "residual"):
                s[p + blk + ".0.weight"] = (cout, cin, 1, 1)
                s[p + blk + ".0.bias"] = (cout,)
                for leaf in ("weight", "bias", "running_mean", "running_var"):
                    s[p + blk + ".1." + leaf] = (cout,)
            s[p + "prelu.weight"] = (1,)
    return s


def random_state_dict(shapes, seed=233):
    return synthetic.fill_state_dict(shapes, seed)


# ---- real weights exported from the reference checkpoints (git-ignored, travels with gpurun) --
# plain .npz files of tensors keyed by the reference's state_dict names; INTERDIFF_B200_WEIGHTS overrides the directory
REF_WEIGHT_DIR = os.environ.get("INTERDIFF_B200_WEIGHTS") or os.path.join(
    os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "weights_ref")


def ref_weights_path(name, directory=None):
    return os.path.join(directory or REF_WEIGHT_DIR, name + ".npz")


def load_ref_weights(name, directory=None):
    """Returns {name: ndarray} exported by oracle/export_ref_weights.py into `directory` (default REF_WEIGHT_DIR),
    or None if absent."""
    p = ref_weights_path(name, directory)
    if not os.path.exists(p):
        return None
    with np.load(p) as z:
        return {k: z[k] for k in z.files}


def bench_weights(name, seed=233):
    """{state_dict name: torch tensor} for the benchmarks / probes / smoke run: the exported checkpoint tensors when
    weights_ref/<name>.npz exists, else seeded random init of the same shapes (the sinusoid tables are always rebuilt).
    name: diffusion_smpl | diffusion_skeleton | correction_smpl | correction_skeleton | diffusion_smpl_encoder |
    diffusion_skeleton_encoder (the encoder names only; merge with diffusion_skeleton for a whole model)."""
    import torch
    sd = load_ref_weights(name)
    if sd is None:
        if name == "correction_smpl":
            shapes = projector_shapes()
        elif name == "correction_skeleton":
            shapes = projector_skeleton_shapes()
        elif name == "diffusion_smpl_encoder":
            shapes = {**mdm_encoder_shapes("smpl"), **pointnet_shapes()}
        elif name == "diffusion_skeleton_encoder":
            shapes = mdm_skeleton_encoder_shapes()
        else:
            variant = name[len("diffusion_"):]
            shapes = {k: v for k, v in mdm_hot_shapes(variant, F=1024 if variant == "smpl" else 256).items() if not k.endswith(".pe")}
        sd = random_state_dict(shapes, seed)
    sd = dict(sd)
    if name.startswith("diffusion_") and not name.endswith("_encoder"):
        pe = synthetic.sinusoid_table(5000, 256).reshape(5000, 1, 256)
        sd["PositionalEmbedding.pe"] = pe
        sd["embedTimeStep.sequence_pos_encoder.pe"] = pe
    return {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()}


def have_ref_weights(name="diffusion_smpl"):
    return os.path.exists(ref_weights_path(name))
