"""Import the reference's own Python classes (from /root/reference, read-only) through the
shims, for validating oracle.restate and generating golden vectors in THIS container.
TEST INFRASTRUCTURE (see oracle/__init__.py).  /root/reference does not exist on the GPU
box: nothing that runs there may call into this module (callers check `available()`).
"""
import os
import sys
from argparse import Namespace

import numpy as np
import torch

from . import shims


def ref_root():
    for cand in (os.environ.get("INTERDIFF_REF"), "/root/reference"):
        if cand and os.path.isdir(os.path.join(cand, "interdiff", "model")):
            return cand
    return None


def available():
    return ref_root() is not None


_IMPORTED = {}


def _prepare():
    root = ref_root()
    if root is None:
        raise RuntimeError("reference tree not found (INTERDIFF_REF or /root/reference)")
    shims.install()
    p = os.path.join(root, "interdiff")
    if p not in sys.path:
        sys.path.insert(0, p)
    return root


def modules():
    """Returns a dict of the reference modules on the hot path."""
    if _IMPORTED:
        return _IMPORTED
    _prepare()
    import importlib
    for name in ("diffusion.gaussian_diffusion", "diffusion.respace", "model.sublayers", "model.layers",
                 "model.diffusion_smpl", "model.diffusion_skeleton", "model.correction_smpl", "model.correction_skeleton",
                 "data.tools", "data.utils", "tools",
                 "libsmpl.smplpytorch.pytorch.smpl_layer"):
        _IMPORTED[name] = importlib.import_module(name)
    return _IMPORTED


def ckpt_path(name):
    return os.path.join(ref_root(), "interdiff", "checkpoints", name + ".ckpt")


def load_ckpt(name):
    ck = torch.load(ckpt_path(name), map_location="cpu", weights_only=False)
    sd = {k[len("model."):]: v for k, v in ck["state_dict"].items() if k.startswith("model.")}
    return ck["hyper_parameters"], sd


def smpl_args(diffusion_steps=None, **over):
    hp, _ = load_ckpt("diffusion")
    hp = dict(hp)
    if diffusion_steps is not None:
        hp["diffusion_steps"] = diffusion_steps
    hp.update(over)
    return Namespace(**hp)


def build_mdm_smpl(state_dict=None, diffusion_steps=None, **over):
    """Reference MDM + SpacedDiffusion (interdiff/model/diffusion_smpl.py:286-289) with the
    shipped weights (state_dict=None) or a caller-provided state dict."""
    m = modules()["model.diffusion_smpl"]
    args = smpl_args(diffusion_steps, **over)
    model, diffusion = m.create_model_and_diffusion(args)
    if state_dict is None:
        _, state_dict = load_ckpt("diffusion")
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    # a caller-provided state dict may omit tensors that are not on the restated hot path
    missing = [k for k in missing if not k.startswith(("pcEmbedding", "encoder", "finalLinear"))
               and "FutureEmbedding" not in k]
    assert not missing and not unexpected, (missing, unexpected)
    model.eval()
    return model, diffusion, args


def skeleton_args(diffusion_steps=None, **over):
    hp, _ = load_ckpt("diffusion_skeleton")
    hp = dict(hp)
    if diffusion_steps is not None:
        hp["diffusion_steps"] = diffusion_steps
    hp.update(over)
    return Namespace(**hp)


def build_mdm_skeleton(state_dict=None, diffusion_steps=None, **over):
    m = modules()["model.diffusion_skeleton"]
    args = skeleton_args(diffusion_steps, **over)
    model, diffusion = m.create_model_and_diffusion(args)
    if state_dict is None:
        _, state_dict = load_ckpt("diffusion_skeleton")
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    missing = [k for k in missing if not k.startswith("encoder") and not k.startswith("shapeEmbedding")]
    assert not missing and not unexpected, (missing, unexpected)
    model.eval()
    return model, diffusion, args


def correction_args(past_len=10, future_len=20, **over):
    hp, _ = load_ckpt("correction")
    hp = dict(hp)
    hp.update(dict(dct=10, num_verts=67, past_len=past_len, future_len=future_len))
    hp.update(over)
    return Namespace(**hp)


def build_obj_projector(state_dict=None, past_len=10, future_len=20):
    m = modules()["model.correction_smpl"]
    args = correction_args(past_len, future_len)
    model = m.ObjProjector(args)
    if state_dict is None:
        _, state_dict = load_ckpt("correction")
    model.load_state_dict(state_dict, strict=True)
    model.eval()
    return model, args


def build_obj_projector_skeleton(state_dict=None):
    """Reference skeleton correction net (model/correction_skeleton.py:8-135) with checkpoints/obj_skeleton.ckpt
    (state_dict=None) or a caller-provided state dict (BatchNorm batch counters may be omitted)."""
    m = modules()["model.correction_skeleton"]
    hp, sd = load_ckpt("obj_skeleton")
    model = m.ObjProjector(Namespace(**hp))
    if state_dict is None:
        model.load_state_dict(sd, strict=True)
    else:
        sd = state_dict
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected and all(k.endswith("num_batches_tracked") for k in missing), (missing, unexpected)
    model.eval()
    return model, Namespace(**hp), sd


def build_smpl_layer(smplh):
    """Reference SMPL_Layer (libsmpl/smplpytorch/pytorch/smpl_layer.py:19-70) constructed
    without the licensed .pkl: __new__ + the buffers its __init__ would register, filled from
    a dict of arrays (see interdiff_b200.synthetic.make_smplh_model)."""
    SMPL_Layer = modules()["libsmpl.smplpytorch.pytorch.smpl_layer"].SMPL_Layer
    layer = SMPL_Layer.__new__(SMPL_Layer)
    torch.nn.Module.__init__(layer)
    layer.center_idx = None
    layer.gender = "male"
    layer.hands = True
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    layer.register_buffer("th_betas", torch.zeros(1, 10))
    layer.register_buffer("th_shapedirs", f32(smplh["shapedirs"]))
    layer.register_buffer("th_posedirs", f32(smplh["posedirs"]))
    layer.register_buffer("th_v_template", f32(smplh["v_template"]).unsqueeze(0))
    layer.register_buffer("th_J_regressor", f32(smplh["J_regressor"]))
    layer.register_buffer("th_weights", f32(smplh["weights"]))
    layer.register_buffer("th_faces", torch.from_numpy(np.asarray(smplh["faces"], dtype=np.int64)))
    layer.kintree_parents = [int(p) for p in smplh["parents"]]
    layer.num_joints = len(layer.kintree_parents)
    return layer
