"""Host-side mirror of reference model/diffusion_skeleton.py (skeleton MDM :15-257; factory
:259-299): 21 body joints + 12 object keypoints + 7-D object pose (106 channels).  The object
keypoints of the prediction are re-derived from the predicted pose inside the library
(calc_obj_pred :218-229).  _get_embeddings (:194-215) assembles `gt` on the host and runs the
conditioning encoder (shape embedding, past-frame embeddings, positional encoding, 8 layers) in
the library (`idb_encode_condition_skeleton`)."""
import torch
import torch.nn as nn

from .diffusion_smpl import _EngineHost, _layer_stack, create_gaussian_diffusion  # noqa: F401
from .layers import PositionalEncoding, TimestepEmbedder, TransformerDecoder, TransformerEncoder
from .sublayers import TransformerDecoderLayerQaN, TransformerEncoderLayerQaN


class MDM(_EngineHost, nn.Module):
    variant = "skeleton"

    def __init__(self, args):
        super().__init__()
        self.args = args
        D = args.embedding_dim
        self.bodyEmbedding = nn.Linear(args.smpl_dim, D)
        self.shapeEmbedding = nn.Linear(args.num_points * 3, D)
        self.objEmbedding = nn.Linear(args.num_points * 3, D)
        self.PositionalEmbedding = PositionalEncoding(d_model=D, dropout=args.dropout)
        self.embedTimeStep = TimestepEmbedder(D, self.PositionalEmbedding)
        self.encoder = TransformerEncoder(_layer_stack(nn.TransformerEncoderLayer, TransformerEncoderLayerQaN, args, D))
        if args.latent_usage != "memory":
            raise NotImplementedError("only latent_usage='memory' (the shipped configuration) is built")
        self.decoder = TransformerDecoder(_layer_stack(nn.TransformerDecoderLayer, TransformerDecoderLayerQaN, args, D))
        self.bodyFinalLinear = nn.Linear(D, args.smpl_dim)
        self.objFinalLinear = nn.Linear(D, 7)

    def encode_condition(self, past, zero_pose_obj):
        """cond (past_len,B,D) from the past frames (B,1,106,past_len) and the canonical object keypoints (B,12,3), on the
        device (the part of `_get_embeddings` after the `gt` concatenation, reference :203-213)."""
        return self.engine_for(past.device).encode_condition_skeleton(past, zero_pose_obj)

    def _get_embeddings(self, body_gt, obj_gt, pose_gt, zero_pose_obj):
        """Reference :194-215: body_gt (T,B,21,3) joints, obj_gt (T,B,12,3) keypoints, pose_gt (T,B,7), zero_pose_obj (B,12,3)
        -> (embedding (past_len,B,D), gt (T,B,106)).  gt is the reference's concatenation; the encoder runs in the library."""
        T, B, n_joints, _ = body_gt.shape
        n_points = obj_gt.shape[2]
        gt = torch.cat([body_gt.reshape(T, B, n_joints * 3), obj_gt.reshape(T, B, n_points * 3), pose_gt], dim=2)
        past = gt[: self.args.past_len].permute(1, 2, 0).unsqueeze(1).contiguous()          # (B,1,106,past_len)
        return self.encode_condition(past, zero_pose_obj), gt

    def forward(self, x, timesteps, zero_pose_obj, y=None):
        """x (B,1,106,T); zero_pose_obj (B,12,3) (reference :250-257)."""
        if y is None:
            raise ValueError("y={'cond': ...} is required")
        eng = self.engine_for(x.device)
        self.bind_kwargs(eng, {"y": y, "zero_pose_obj": zero_pose_obj}, T=x.shape[-1])
        return eng.forward(x, timesteps)


def create_model_and_diffusion(args):
    return MDM(args), create_gaussian_diffusion(args)
