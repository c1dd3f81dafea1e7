"""CPU-side checks of the drop-in boundary: the C ABI exports every symbol the header declares,
the mirrored modules load the reference checkpoints strictly, the diffusion tables equal the
reference's, and the product path refuses to run without a GPU (no CPU fallback)."""
import gzip
import json
import os
import re
from argparse import Namespace

import numpy as np
import pytest
import torch

from interdiff_b200 import _lib
from interdiff_b200 import weights as W
from oracle import restate as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def reference_checkpoint(name):
    """(hyper_parameters, {state_dict name: zero tensor of the stored shape}) of the reference's shipped checkpoint `name`
    (tests/golden/checkpoints.json.gz, written by `python -m oracle.make_golden --reference-checks`)"""
    with gzip.open(os.path.join(GOLDEN, "checkpoints.json.gz")) as f:
        ck = json.load(f)[name]
    return ck["hyper_parameters"], {k: torch.zeros(shape) for k, shape in ck["state_dict"].items()}


SMPL_ARGS = dict(embedding_dim=256, smpl_dim=132, use_pointnet2=1, dropout=0.0, num_heads=4, ff_size=1024, activation="gelu",
                 latent_usage="memory", future_len=25, past_len=10, cond_mask_prob=0, diffusion_steps=1000, noise_schedule="cosine",
                 sigma_small=True, weight_v=0.2)


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    lib = _lib.lib()
    header = open(os.path.join(ROOT, "include", "interdiff_b200.h")).read()
    declared = set(re.findall(r"\b(idb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.EXPORTS)
    assert lib.idb_version() >= 100


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from interdiff_b200.engine import Engine, EngineError
    with pytest.raises(EngineError):
        Engine()
    from interdiff_b200.model.diffusion_smpl import MDM
    m = MDM(Namespace(**SMPL_ARGS))
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 1, 144, 30), torch.zeros(1, dtype=torch.long), y={"cond": torch.zeros(10, 1, 256)})


def test_mirror_state_dict_names_match_tables():
    from interdiff_b200.model.diffusion_smpl import MDM
    sd = MDM(Namespace(**SMPL_ARGS)).state_dict()
    for k, shp in W.mdm_hot_shapes("smpl", F=1024).items():
        assert k in sd and tuple(sd[k].shape) == tuple(shp), k
    for k, shp in {**W.mdm_encoder_shapes("smpl", F=1024), **W.pointnet_shapes()}.items():
        assert k in sd and tuple(sd[k].shape) == tuple(shp), k
    from interdiff_b200.model.correction_smpl import ObjProjector
    psd = ObjProjector(Namespace(dct=10, num_verts=67, dropout=0.1, past_len=10, future_len=20, embedding_dim=64)).state_dict()
    for k, shp in W.projector_shapes().items():
        assert k in psd and tuple(psd[k].shape) == tuple(shp), k


def test_mirrors_load_reference_checkpoints_strictly():
    from interdiff_b200.model import correction_smpl, diffusion_skeleton, diffusion_smpl
    hp, sd = reference_checkpoint("diffusion")
    m, d = diffusion_smpl.create_model_and_diffusion(Namespace(**hp))
    m.load_state_dict(sd, strict=True)
    assert d.num_timesteps == 1000
    hp, sd = reference_checkpoint("diffusion_skeleton")
    m, _ = diffusion_skeleton.create_model_and_diffusion(Namespace(**hp))
    m.load_state_dict(sd, strict=True)
    hp, sd = reference_checkpoint("correction")
    p = correction_smpl.ObjProjector(Namespace(**{**hp, "dct": 10}))
    p.load_state_dict(sd, strict=True)


def test_diffusion_tables_and_spacing():
    from interdiff_b200.diffusion import gaussian_diffusion as gd
    from interdiff_b200.diffusion.respace import SpacedDiffusion, space_timesteps
    for steps in (100, 1000):
        betas = gd.get_named_beta_schedule("cosine", steps)
        d = SpacedDiffusion(use_timesteps=space_timesteps(steps, [steps]), betas=betas, model_mean_type=gd.ModelMeanType.START_X,
                            model_var_type=gd.ModelVarType.FIXED_SMALL, loss_type=gd.LossType.MSE)
        t = R.diffusion_tables(R.named_beta_schedule("cosine", steps))
        for k in ("posterior_mean_coef1", "posterior_mean_coef2", "posterior_log_variance_clipped"):
            assert np.allclose(getattr(d, k), t[k], rtol=1e-12, atol=0)
        assert d.timestep_map == list(range(steps))
    d = SpacedDiffusion(use_timesteps=space_timesteps(1000, [100]), betas=gd.get_named_beta_schedule("cosine", 1000),
                        model_mean_type=gd.ModelMeanType.START_X, model_var_type=gd.ModelVarType.FIXED_SMALL, loss_type=gd.LossType.MSE)
    assert d.num_timesteps == 100 and d.timestep_map[0] == 0 and d.timestep_map[-1] == 999
    # the reference's diffusion.respace on the same arguments (tests/golden/reference_checks.npz)
    ref = np.load(os.path.join(GOLDEN, "reference_checks.npz"))
    assert space_timesteps(1000, [100]) == set(ref["space_1000_100"].tolist())
    assert space_timesteps(300, "10,15,20") == set(ref["space_300_10_15_20"].tolist())
    assert np.array_equal(ref["spaced_1000_100_betas"], d.betas) and ref["spaced_1000_100_timestep_map"].tolist() == d.timestep_map


def test_skeleton_projector_mirror_loads_checkpoint_strictly():
    """interdiff_b200.model.correction_skeleton.ObjProjector carries the reference's state_dict names (obj_skeleton.ckpt)"""
    from interdiff_b200.model.correction_skeleton import ObjProjector
    hp, sd = reference_checkpoint("obj_skeleton")
    m = ObjProjector(Namespace(**hp))
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    from interdiff_b200 import weights as W2
    assert set(W2.projector_skeleton_shapes()) == {k for k in sd if "num_batches_tracked" not in k}
