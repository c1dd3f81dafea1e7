"""Host-side mirror of reference model/diffusion_smpl.py: MDM (:8-246), create_gaussian_diffusion
(:251-284), create_model_and_diffusion (:286-289).

The module tree reproduces the reference's state_dict names exactly (strict checkpoint loading,
SURVEY.md section 8b) but only holds parameters: forward() runs the sm_100a decoder in
libinterdiff_b200.so.  There is no eager/CPU fallback.
"""
import torch
import torch.nn as nn

from ..diffusion import gaussian_diffusion as gd
from ..diffusion.respace import SpacedDiffusion, space_timesteps
from ..engine import Engine
from .layers import PointNet2Encoder, PositionalEncoding, TimestepEmbedder, TransformerDecoder, TransformerEncoder
from .sublayers import TransformerDecoderLayerQaN, TransformerEncoderLayerQaN


def _layer_stack(std_cls, qan_cls, args, D):
    kw = dict(d_model=D, nhead=args.num_heads, dim_feedforward=args.ff_size, dropout=args.dropout,
              activation=args.activation, batch_first=False)
    # layers 1 and 8 are the stock torch layers, 2..7 the query-and-attend ones
    return nn.ModuleList([(std_cls if i in (0, 7) else qan_cls)(**kw) for i in range(8)])


class _EngineHost:
    """Shared by the SMPL and skeleton MDM mirrors: lazily creates one Engine per device, keeps
    its packed weights in sync with the module's parameters and binds the conditioning."""
    variant = "smpl"
    rotary = "absolute"   # local-attention <= 1.5 rotary placement; 'bucketed' for >= 1.6 (SURVEY 8c)

    def _hot_state(self):
        keep = ("decoder.", "encoder.", "pcEmbedding.", "shapeEmbedding.", "bodyEmbedding.", "objEmbedding.", "bodyFinalLinear.",
                "objFinalLinear.", "embedTimeStep.time_embed.", "PositionalEmbedding.pe")
        return {k: v for k, v in self.state_dict().items() if k.startswith(keep)}

    def _signature(self):
        return tuple((k, v._version, v.data_ptr()) for k, v in self._hot_state().items())

    def engine_for(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("interdiff_b200.MDM runs on a CUDA (sm_100a) device only: no CPU fallback")
        engines = self.__dict__.setdefault("_engines", {})
        ent = engines.get(device)
        sig = self._signature()
        if ent is None or ent[1] != sig:
            eng = ent[0] if ent else Engine(device)
            eng.load_denoiser(self._hot_state(), self.variant, rotary=self.rotary, n_heads=self.args.num_heads)
            engines[device] = ent = (eng, sig)
            self.__dict__["_bound"] = None
        return ent[0]

    def bind_kwargs(self, eng, model_kwargs, T=None):
        y = model_kwargs["y"]
        cond = self.mask_cond(y["cond"])
        zp = model_kwargs.get("zero_pose_obj")
        T = T if T is not None else y["inpainted_motion"].shape[-1] if "inpainted_motion" in y else None
        key = (id(eng), cond.data_ptr(), cond._version, tuple(cond.shape), T, None if zp is None else (zp.data_ptr(), zp._version))
        if self.__dict__.get("_bound") != key:
            if T is None:
                raise ValueError("cannot infer the number of frames; call forward() first or pass inpainted_motion")
            eng.bind(cond, T, zero_pose_obj=zp)
            self.__dict__["_bound"] = key

    def mask_cond(self, cond, force_mask=False):
        if force_mask:
            return torch.zeros_like(cond)
        if self.training and self.args.cond_mask_prob > 0.0:
            raise NotImplementedError("condition dropout is a training-time feature (model/diffusion_smpl.py:185-193)")
        return cond


class MDM(_EngineHost, nn.Module):
    variant = "smpl"

    def __init__(self, args):
        super().__init__()
        self.args = args
        D = args.embedding_dim
        self.bodyEmbedding = nn.Linear(args.smpl_dim + 3, D)
        self.pcEmbedding = PointNet2Encoder(c_in=1, c_out=D, num_keypoints=1) if args.use_pointnet2 else nn.Linear(6, D)
        self.objEmbedding = nn.Linear(9, D)
        self.PositionalEmbedding = PositionalEncoding(d_model=D, dropout=args.dropout)
        self.embedTimeStep = TimestepEmbedder(D, self.PositionalEmbedding)
        self.objPooling = nn.MaxPool1d(1)
        self.encoder = TransformerEncoder(_layer_stack(nn.TransformerEncoderLayer, TransformerEncoderLayerQaN, args, D))
        if args.latent_usage == "memory":
            self.decoder = TransformerDecoder(_layer_stack(nn.TransformerDecoderLayer, TransformerDecoderLayerQaN, args, D))
        else:
            raise NotImplementedError("only latent_usage='memory' (the shipped configuration) is built")
        self.finalLinear = nn.Linear(D, args.smpl_dim + 9)
        self.bodyFinalLinear = nn.Linear(D, args.smpl_dim + 3)
        self.objFinalLinear = nn.Linear(D, 9)
        self.bodyFutureEmbedding = nn.Parameter(torch.empty(args.future_len, 1, D).uniform_(-1, 1))
        self.objFutureEmbedding = nn.Parameter(torch.empty(args.future_len, 1, D).uniform_(-1, 1))

    @staticmethod
    def _axis_angle_to_rot6d(aa):
        """matrix_to_rotation_6d(axis_angle_to_matrix(aa)) (pytorch3d convention: first two ROWS), aa (...,3)."""
        th = aa.norm(dim=-1, keepdim=True)
        k = aa / th.clamp_min(1e-12)
        kx, ky, kz = k[..., 0], k[..., 1], k[..., 2]
        c, s_ = torch.cos(th[..., 0]), torch.sin(th[..., 0])
        C = 1 - c
        return torch.stack([c + kx * kx * C, kx * ky * C - kz * s_, kx * kz * C + ky * s_,
                            ky * kx * C + kz * s_, c + ky * ky * C, ky * kz * C - kx * s_], dim=-1)

    def encode_condition(self, past, pc_embedding):
        """cond (past_len,B,D) from the past frames (B,1,144,past_len) and the point-cloud embedding (B,D): the part
        of `_get_embeddings` after `pcEmbedding` (reference :217-221), on the device."""
        return self.engine_for(past.device).encode_condition(past, pc_embedding)

    def _get_embeddings(self, data, device=None):
        """Reference :195-223, on the device: PointNet++ point-cloud embedding (`idb_pointcloud_embed`), past-frame
        embeddings + positional encoding + 8-layer encoder (`idb_encode_condition`).  data['pc_embedding'] (B,D),
        when present, replaces the point-cloud encoder (e.g. cached per object)."""
        dev = torch.device(device) if device else data["frames"][0]["smplfit_params"]["pose"].device
        cat = lambda key, sub, sl=slice(None): torch.cat([f[key][sub][:, sl].unsqueeze(0) for f in data["frames"]], dim=0).float().to(dev)
        body_pose, body_trans = cat("smplfit_params", "pose", slice(0, 66)), cat("smplfit_params", "trans")
        obj_angles, obj_trans = cat("objfit_params", "angle"), cat("objfit_params", "trans")
        T, B, _ = body_pose.shape
        body_pose = self._axis_angle_to_rot6d(body_pose.view(T, B, -1, 3)).view(T, B, -1)
        obj_angles = self._axis_angle_to_rot6d(obj_angles.view(T, B, -1, 3)).view(T, B, -1)
        gt = torch.cat([body_pose, body_trans, obj_angles, obj_trans], dim=2)                  # (T,B,144)
        past = gt[: self.args.past_len].permute(1, 2, 0).unsqueeze(1).contiguous()              # (B,1,144,past_len)
        if "pc_embedding" in data:
            pc = data["pc_embedding"].to(dev).float().view(B, -1)
        else:
            if not self.args.use_pointnet2:
                raise NotImplementedError("use_pointnet2=0 (a Linear on 6 channels) is not a shipped configuration")
            pc = self.engine_for(dev).pointcloud_embed(data["obj_points"][:, :, :3].float().to(dev))
        return self.encode_condition(past, pc), gt

    def forward(self, x, timesteps, y=None):
        """x (B,1,144,T), timesteps (B,) long, y={'cond': (Tm,B,D)} -> predicted x_0 (B,1,144,T)
        (reference :239-246)."""
        if y is None:
            raise ValueError("y={'cond': ...} is required")
        eng = self.engine_for(x.device)
        self.bind_kwargs(eng, {"y": y}, T=x.shape[-1])
        return eng.forward(x, timesteps)


def create_gaussian_diffusion(args):
    steps = args.diffusion_steps
    betas = gd.get_named_beta_schedule(args.noise_schedule, steps, 1.0)
    return SpacedDiffusion(
        use_timesteps=space_timesteps(steps, [steps]), betas=betas, model_mean_type=gd.ModelMeanType.START_X,
        model_var_type=gd.ModelVarType.FIXED_SMALL if args.sigma_small else gd.ModelVarType.FIXED_LARGE,
        loss_type=gd.LossType.MSE, rescale_timesteps=False, lambda_vel=args.weight_v)


def create_model_and_diffusion(args):
    return MDM(args), create_gaussian_diffusion(args)
