"""Export the hot-path tensors of the reference's shipped checkpoints as <name>.npz files.
TEST INFRASTRUCTURE: gives the parity tests the trained weights' value distribution.  build() writes them to
oracle/_ref/weights/ (git-ignored, like every artefact built from the reference tree) when the reference tree is
readable; the tests load them from there.  bench.py keeps its seeded random init unless INTERDIFF_B200_WEIGHTS (or
weights_ref/) names such a directory:  python -m oracle.export_ref_weights [DIR]
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from interdiff_b200 import weights as W  # noqa: E402
from oracle import ref_loader as RL  # noqa: E402

OUT_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "weights")


def main(out_dir=OUT_DIR):
    os.makedirs(out_dir, exist_ok=True)
    jobs = (("diffusion", "diffusion_smpl", W.mdm_hot_shapes("smpl", F=1024)),
            ("diffusion_skeleton", "diffusion_skeleton", W.mdm_hot_shapes("skeleton", F=256)),
            ("correction", "correction_smpl", W.projector_shapes()),
            ("obj_skeleton", "correction_skeleton", W.projector_skeleton_shapes()),
            # conditioning encoder: its own file, only the encoder tests load it
            ("diffusion", "diffusion_smpl_encoder", {**W.mdm_encoder_shapes("smpl", F=1024), **W.pointnet_shapes()}))
    for ck, out, shapes in jobs:
        _, sd = RL.load_ckpt(ck)
        sel = {}
        for k, shp in shapes.items():
            if k.endswith(".pe"):
                continue  # recomputed (model/layers.py:14-19)
            v = sd[k].numpy()
            assert tuple(v.shape) == tuple(shp), (k, v.shape, shp)
            sel[k] = v
        np.savez(W.ref_weights_path(out, out_dir), **sel)
        print(out, len(sel), "tensors", sum(v.size for v in sel.values()) * 4 / 1e6, "MB")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else OUT_DIR)
