"""Export the skeleton model's conditioning-path tensors (encoder.layers.*, shapeEmbedding.*) of the shipped
checkpoints/diffusion_skeleton.ckpt as diffusion_skeleton_encoder.npz, next to the files oracle/export_ref_weights.py writes.
TEST INFRASTRUCTURE; build() runs it where the reference tree is readable:  python -m oracle.export_skeleton_weights [DIR]
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from interdiff_b200 import weights as W  # noqa: E402
from oracle import ref_loader as RL  # noqa: E402
from oracle.export_ref_weights import OUT_DIR  # noqa: E402

NAME = "diffusion_skeleton_encoder"


def main(out_dir=OUT_DIR):
    os.makedirs(out_dir, exist_ok=True)
    _, sd = RL.load_ckpt("diffusion_skeleton")
    sel = {}
    for k, shp in W.mdm_skeleton_encoder_shapes().items():
        v = sd[k].numpy()
        assert tuple(v.shape) == tuple(shp), (k, v.shape, shp)
        sel[k] = v
    np.savez(W.ref_weights_path(NAME, out_dir), **sel)
    print(NAME, len(sel), "tensors", sum(v.size for v in sel.values()) * 4 / 1e6, "MB")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else OUT_DIR)
