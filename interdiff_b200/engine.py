"""Thin host wrapper over the C ABI: one Engine = one idb_handle on one GPU.

PyTorch is used for device memory and streams only (tensor.data_ptr() in, tensor out); all
arithmetic on the hot path runs in libinterdiff_b200.so.  Nothing here falls back to torch ops.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

ROTARY_OFFSETS = {"absolute": (1.0, 0.0, -1.0), "bucketed": (2.0, 1.0, 0.0)}

# reference data/utils.py:232-238, 252-253 (constants of the correction hook)
MARKERSET_SSM67_SMPLH = [3470, 3171, 3327, 857, 1812, 628, 182, 3116, 3040, 239,
                         1666, 1725, 0, 2174, 1568, 1368, 3387, 2112, 1053, 1058,
                         3336, 3346, 1323, 2108, 3122, 3314, 1252, 1082, 1861, 1454,
                         850, 2224, 3233, 1769, 6728, 4343, 5273, 4116, 3694, 6399,
                         6540, 6488, 3749, 5135, 5194, 3512, 5635, 5210, 4360, 4841,
                         6786, 5573, 4538, 4544, 6736, 6747, 4804, 5568, 6544, 6682,
                         5322, 4927, 5686, 4598, 6633, 3506, 3508]
HAND_MARKERS = [10, 11, 14, 31, 13, 17, 23, 28, 27] + [60, 43, 44, 47, 62, 46, 51, 57]


class EngineError(RuntimeError):
    pass


def _shape_arr(shape):
    return (C.c_int64 * max(len(shape), 1))(*[int(s) for s in shape])


class Engine:
    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise EngineError("interdiff_b200 needs a CUDA (sm_100a) device; there is no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.lib = _lib.lib()
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            rc = self.lib.idb_create(C.byref(self._h))
        if rc:
            msg = self.lib.idb_last_error(self._h).decode() if self._h else "idb_create failed"
            raise EngineError(msg)
        self._keep = []       # tensors the library may still read asynchronously
        self.variant = None
        self.C = None
        self.n_steps = 0

    def close(self):
        if self._h:
            torch.cuda.synchronize(self.device)
            self.lib.idb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _chk(self, rc):
        if rc:
            raise EngineError("%s (status %d)" % (self.lib.idb_last_error(self._h).decode(), rc))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _f32(self, t):
        if isinstance(t, np.ndarray):
            t = torch.from_numpy(t)
        return t.to(device=self.device, dtype=torch.float32).contiguous()

    @staticmethod
    def _ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p()

    @property
    def launch_count(self):
        return int(self.lib.idb_launch_count(self._h))

    def set_dependent_launch(self, on):
        """Programmatic dependent launch between the kernels of a step (default on; identical results)."""
        self._chk(self.lib.idb_set_dependent_launch(self._h, 1 if on else 0))

    def set_nn_pruning(self, on):
        """Cluster-pruned nearest-neighbour search for body-mesh targets (default on; identical results)."""
        self._chk(self.lib.idb_set_nn_pruning(self._h, 1 if on else 0))

    def set_gemm_multicast(self, on):
        """SMPL-H blend GEMM with / without TMA-multicast row-tile pairs (identical results; bisecting / A-B timing)."""
        self._chk(self.lib.idb_debug_set_gemm_multicast(self._h, 1 if on else 0))

    def set_fused_mlp(self, on):
        """Feed-forward block as one cluster kernel (default on) vs two GEMM launches."""
        self._chk(self.lib.idb_set_fused_mlp(self._h, int(on)))

    def mlp(self, x, w1, b1, w2, b2, res, iters=1, trace=None, ln_w=None, ln_b=None):
        """gelu(x @ w1.T + b1) @ w2.T + b2 + res through the fused feed-forward kernel (tests / probes).
        iters > 1: self.last_ms() is the mean time of launches 2..iters; trace: int64 [ctas,16] device tensor."""
        x, w1, b1, w2, b2, res = (self._f32(t) for t in (x, w1, b1, w2, b2, res))
        out = torch.empty_like(x)
        ln_w = self._f32(ln_w) if ln_w is not None else None
        ln_b = self._f32(ln_b) if ln_b is not None else None
        self._chk(self.lib.idb_debug_mlp(self._h, self._ptr(x), self._ptr(w1), self._ptr(b1), self._ptr(w2), self._ptr(b2), self._ptr(res),
                                         self._ptr(out), x.shape[0], int(iters), self._ptr(trace), self._ptr(ln_w), self._ptr(ln_b),
                                         self._stream()))
        return out

    def last_ms(self):
        return float(self.lib.idb_debug_last_ms(self._h))

    def set_gemm_backend(self, backend):
        self._chk(self.lib.idb_set_gemm_backend(self._h, {"simt": 0, "tcgen05": 1}.get(backend, backend)))

    # ------------------------------------------------------------------ kernel-level hooks
    def gemm(self, A, W, bias=None, res=None, gelu=False, silu=False, split_k=False):
        """epi(A @ W.T) through the handle's GEMM backend (tests / roofline leg).  split_k: the tensor path's
        2-way split-K variant (two partial tiles reduced onto a zeroed C), as the denoiser runs ff2."""
        A, W = self._f32(A), self._f32(W)
        bias = self._f32(bias) if bias is not None else None
        res = self._f32(res) if res is not None else None
        M, K = A.shape
        N = W.shape[0]
        out = torch.empty(M, N, device=self.device)
        epi = (1 if bias is not None else 0) | (2 if gelu else 0) | (4 if res is not None else 0) | (8 if silu else 0)
        epi |= 128 if split_k else 0
        self._chk(self.lib.idb_debug_gemm(self._h, self._ptr(A), self._ptr(W), self._ptr(bias), self._ptr(res), self._ptr(out),
                                          M, N, K, epi, self._stream()))
        return out

    def gemm_microbench(self, M, N, K, iters=200, gelu=True, split_k=False):
        """Mean device time of one tensor-core GEMM launch (fp16-pair operands as the denoiser feeds them,
        bias + optional GELU epilogue) over `iters` back-to-back launches issued from C on the current
        stream, CUDA events, after warm-up."""
        g = torch.Generator(device="cpu").manual_seed(0)
        A = torch.randn(M, K, generator=g).to(self.device)
        W = (torch.randn(N, K, generator=g) / K ** 0.5).to(self.device)
        bias = torch.randn(N, generator=g).to(self.device)
        out = torch.empty(M, N, device=self.device)
        Ah, Al, Wh, Wl = (torch.empty_like(t, dtype=torch.float16) for t in (A, A, W, W))
        P = self._ptr
        self._chk(self.lib.idb_debug_split(self._h, P(A), P(Ah), P(Al), M, K, K, self._stream()))
        self._chk(self.lib.idb_debug_split(self._h, P(W), P(Wh), P(Wl), N, K, K, self._stream()))
        epi = 1 | (2 if gelu else 0) | (128 if split_k else 0)
        call = lambda n: self._chk(self.lib.idb_debug_gemm_presplit(self._h, P(Ah), P(Al), P(Wh), P(Wl), P(bias), P(out), M, N, K, epi, n,
                                                                    C.c_void_p(), self._stream()))
        call(10)
        torch.cuda.synchronize(self.device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call(iters)
        e1.record()
        torch.cuda.synchronize(self.device)
        return dict(M=M, N=N, K=K, iters=iters, ms=e0.elapsed_time(e1) / iters, kernel="gemm_split_f16_kernel<128> (ff1: bias+GELU)")

    # ------------------------------------------------------------------ denoiser
    def load_denoiser(self, state_dict, variant="smpl", rotary="absolute", n_heads=4, n_queries=10):
        """state_dict: reference names without the 'model.' prefix (tensors or arrays)."""
        sd = {k: v for k, v in state_dict.items()}
        D = int(sd["bodyEmbedding.weight"].shape[0])
        layers = sorted({int(k.split(".")[2]) for k in sd if k.startswith("decoder.layers.")})
        qan_mask = 0
        for l in layers:
            if "decoder.layers.%d.queries" % l in sd:
                qan_mask |= 1 << l
        cfg = _lib.DenoiserConfig()
        cfg.variant = 0 if variant == "smpl" else 1
        cfg.d_model, cfg.n_heads, cfg.n_layers, cfg.n_queries = D, n_heads, len(layers), n_queries
        cfg.d_ff = int(sd["decoder.layers.0.linear1.weight"].shape[0])
        cfg.c_body = int(sd["bodyEmbedding.weight"].shape[1])
        cfg.c_obj = int(sd["objEmbedding.weight"].shape[1])
        cfg.c_extra = 0 if variant == "smpl" else 7
        cfg.n_points = 0 if variant == "smpl" else cfg.c_obj // 3
        cfg.qan_mask = qan_mask
        for i, o in enumerate(ROTARY_OFFSETS[rotary]):
            cfg.rotary_offsets[i] = o
        self._chk(self.lib.idb_denoiser_init(self._h, C.byref(cfg)))
        for name, w in sd.items():
            if not torch.is_tensor(w):
                w = torch.as_tensor(np.asarray(w))
            if not w.dtype.is_floating_point:
                continue
            w = w.detach().to(dtype=torch.float32).contiguous()
            self._chk(self.lib.idb_denoiser_load(self._h, name.encode(), C.c_void_p(w.data_ptr()),
                                                 _shape_arr(w.shape), w.dim()))
        self._chk(self.lib.idb_denoiser_commit(self._h))
        self.variant = variant
        self.C = cfg.c_body + cfg.c_obj + cfg.c_extra
        self.D = D

    def bind(self, cond, T, zero_pose_obj=None):
        """cond (Tm,B,D) as in model_kwargs['y']['cond']."""
        cond = self._f32(cond)
        Tm, B, _ = cond.shape
        zp = self._f32(zero_pose_obj) if zero_pose_obj is not None else None
        self._chk(self.lib.idb_denoiser_bind(self._h, B, T, Tm, self._ptr(cond), self._ptr(zp), self._stream()))
        self._keep = [cond, zp]
        self.B, self.T = B, T

    def forward(self, x, timesteps):
        x = self._f32(x)
        t = timesteps.to(device=self.device, dtype=torch.int64).contiguous()
        out = torch.empty_like(x)
        self._chk(self.lib.idb_denoiser_forward(self._h, self._ptr(x), self._ptr(t), self._ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ diffusion
    def init_diffusion(self, betas, timestep_map=None):
        betas = np.ascontiguousarray(betas, dtype=np.float64)
        n = len(betas)
        tm = None
        if timestep_map is not None:
            tm = (C.c_int64 * n)(*[int(v) for v in timestep_map])
        self._chk(self.lib.idb_diffusion_init(self._h, betas.ctypes.data_as(C.POINTER(C.c_double)), tm, n))
        self.n_steps = n

    @staticmethod
    def _mask_u8(mask, device):
        """bool and uint8 masks share one byte layout: a device-resident bool mask is reinterpreted, not copied."""
        if mask is None:
            return None
        mask = mask.to(device=device)
        if mask.dtype == torch.bool:
            return mask.contiguous().view(torch.uint8)
        return mask.to(torch.uint8).contiguous()

    def p_sample(self, i, x_t, noise, gt=None, mask=None):
        x_t, noise = self._f32(x_t), self._f32(noise)
        gt = self._f32(gt) if gt is not None else None
        m = self._mask_u8(mask, self.device)
        out, x0 = torch.empty_like(x_t), torch.empty_like(x_t)
        self._chk(self.lib.idb_p_sample(self._h, int(i), self._ptr(x_t), self._ptr(noise), self._ptr(gt), self._ptr(m),
                                        self._ptr(out), self._ptr(x0), self._stream()))
        return out, x0

    def p_sample_predict(self, i, x_t, gt=None, mask=None):
        x_t = self._f32(x_t)
        gt = self._f32(gt) if gt is not None else None
        m = self._mask_u8(mask, self.device)
        x0 = torch.empty_like(x_t)
        self._chk(self.lib.idb_p_sample_predict(self._h, int(i), self._ptr(x_t), self._ptr(gt), self._ptr(m), self._ptr(x0), self._stream()))
        return x0

    def p_sample_finish(self, i, x0, x_t, noise):
        x0, x_t, noise = self._f32(x0), self._f32(x_t), self._f32(noise)
        out = torch.empty_like(x_t)
        self._chk(self.lib.idb_p_sample_finish(self._h, int(i), self._ptr(x0), self._ptr(x_t), self._ptr(noise), self._ptr(out), self._stream()))
        return out

    default_graph_mode = 2     # use_graph=True -> this mode: 1 = one captured graph per step, 2 = the whole loop as one graph (+1.4 %)

    def _graph_mode(self, use_graph):
        if isinstance(use_graph, str):
            return {"off": 0, "step": 1, "loop": 2}[use_graph]
        if use_graph is True:
            return self.default_graph_mode
        return int(use_graph)

    def p_sample_loop(self, tape, gt=None, mask=None, correction=False, use_graph=True, out=None):
        """tape: (n_steps+1, B,1,C,T) device tensor; tape[0] = x_T.  use_graph: False / True / 'off' / 'step' / 'loop'.
        gt / mask are copied into the handle's own buffers and the tape is reached through a device slot, so the
        captured graphs are reused across calls with fresh tensors."""
        assert tape.is_cuda and tape.dtype == torch.float32 and tape.is_contiguous()
        assert tape.shape[0] == self.n_steps + 1
        gt = self._f32(gt) if gt is not None else None
        m = self._mask_u8(mask, self.device)
        if out is None:
            out = torch.empty_like(tape[0])
        mode = self._graph_mode(use_graph)
        self._chk(self.lib.idb_p_sample_loop(self._h, self._ptr(tape), self._ptr(gt), self._ptr(m), int(bool(correction)),
                                             int(mode), self._ptr(out), self._stream()))
        self._keep_loop = [tape, gt, m]   # read asynchronously by the enqueued work
        return out

    def pointcloud_embed(self, obj_points):
        """pc_embedding (B,256) = the reference's pcEmbedding (PointNet++ MSG) on obj_points (B,P,3); needs the
        pcEmbedding.* weights loaded."""
        p = self._f32(obj_points)
        B, P, _ = p.shape
        out = torch.empty(B, 256, device=self.device)
        self._chk(self.lib.idb_pointcloud_embed(self._h, B, P, self._ptr(p), self._ptr(out), self._stream()))
        return out

    def encode_condition(self, past, pc_embedding):
        """cond (Tp,B,256) = conditioning encoder on the past frames (B,1,C,Tp) + point-cloud embedding (B,256)
        (reference MDM._get_embeddings after pcEmbedding); needs the encoder.layers.* weights loaded."""
        past, pc = self._f32(past), self._f32(pc_embedding)
        B, Tp = past.shape[0], past.shape[-1]
        out = torch.empty(Tp, B, 256, device=self.device)
        self._chk(self.lib.idb_encode_condition(self._h, B, Tp, self._ptr(past), self._ptr(pc), self._ptr(out), self._stream()))
        return out

    def encode_condition_skeleton(self, past, zero_pose_obj):
        """cond (Tp,B,256) of the skeleton model = conditioning encoder on the past frames (B,1,106,Tp) + the shape embedding
        of zero_pose_obj (B,12,3) (reference skeleton MDM._get_embeddings); needs encoder.layers.* and shapeEmbedding.* loaded."""
        past, zp = self._f32(past), self._f32(zero_pose_obj)
        B, Tp = past.shape[0], past.shape[-1]
        out = torch.empty(Tp, B, 256, device=self.device)
        self._chk(self.lib.idb_encode_condition_skeleton(self._h, B, Tp, self._ptr(past), self._ptr(zp), self._ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ body model / geometry
    def load_body(self, smplh):
        f = lambda k: np.ascontiguousarray(np.asarray(smplh[k]), dtype=np.float32)
        vt, sd, pd, jr, w = f("v_template"), f("shapedirs"), f("posedirs"), f("J_regressor"), f("weights")
        parents = np.ascontiguousarray(np.asarray(smplh["parents"]), dtype=np.int32)
        faces = np.ascontiguousarray(np.asarray(smplh["faces"]), dtype=np.int32)
        V, J, NB = vt.shape[0], jr.shape[0], sd.shape[2]
        assert pd.shape == (V, 3, (J - 1) * 9) and w.shape == (V, J)
        p = lambda a: C.c_void_p(a.ctypes.data)
        self._chk(self.lib.idb_body_init(self._h, V, J, NB, faces.shape[0], p(vt), p(sd), p(pd), p(jr), p(w), p(parents), p(faces)))
        self.V, self.J = V, J
        self._body_owner = None      # set by SMPL_Layer.load_into (which module's arrays this engine holds)

    def lbs(self, pose, betas, trans, want_verts=True, want_jtr=True):
        pose, betas, trans = self._f32(pose), self._f32(betas), self._f32(trans)
        F = pose.shape[0]
        verts = torch.empty(F, self.V, 3, device=self.device) if want_verts else None
        jtr = torch.empty(F, self.J, 3, device=self.device) if want_jtr else None
        self._chk(self.lib.idb_smplh_lbs(self._h, F, self._ptr(pose), self._ptr(betas), self._ptr(trans),
                                         self._ptr(verts), self._ptr(jtr), self._stream()))
        return verts, jtr

    def vertex_normals(self, verts):
        verts = self._f32(verts)
        out = torch.empty_like(verts)
        self._chk(self.lib.idb_vertex_normals(self._h, verts.shape[0], self._ptr(verts), self._ptr(out), self._stream()))
        return out

    def signed_nn(self, query, target, target_normals=None):
        query, target = self._f32(query), self._f32(target)
        tn = self._f32(target_normals) if target_normals is not None else None
        F, Pq, _ = query.shape
        Pt = target.shape[1]
        d = torch.empty(F, Pq, device=self.device)
        idx = torch.empty(F, Pq, device=self.device, dtype=torch.int32)
        vec = torch.empty(F, Pq, 3, device=self.device)
        self._chk(self.lib.idb_signed_nn(self._h, F, Pq, Pt, self._ptr(query), self._ptr(target), self._ptr(tn),
                                         self._ptr(d), self._ptr(idx), self._ptr(vec), self._stream()))
        return d, idx, vec

    def rot6d_to_axis_angle(self, d6):
        d6 = self._f32(d6)
        out = torch.empty(d6.shape[:-1] + (3,), device=self.device)
        self._chk(self.lib.idb_rot6d_to_axis_angle(self._h, d6.numel() // 6, self._ptr(d6), self._ptr(out), self._stream()))
        return out

    METRIC_NAMES = ("global_mpjpe", "local_mpjpe", "body_translation", "obj_translation", "obj_rot_error", "penetrate")

    def metrics(self, obj_pred, body_jtr, body, obj_gt, body_jtr_gt, body_gt, verts, obj_points):
        """The reference's `metrics` (eval_smpl_short.py:24-81) on the device -> dict of (B,) tensors; the body model
        (with faces) must be loaded."""
        a = [self._f32(t) for t in (obj_pred, body_jtr, body, obj_gt, body_jtr_gt, body_gt, verts, obj_points)]
        T, B, J = a[1].shape[:3]
        out = torch.empty(6, B, device=self.device)
        self._chk(self.lib.idb_metrics(self._h, T, B, J, a[7].shape[1], a[2].shape[2], *[self._ptr(t) for t in a], self._ptr(out),
                                       self._stream()))
        return {k: out[i] for i, k in enumerate(self.METRIC_NAMES)}

    SKELETON_METRIC_NAMES = ("mpjpe_h", "mpjpe_o", "translation_error", "rotation_error", "rotation_error_l2")

    def skeleton_metrics(self, pred, gt, past_len, n_joints=21):
        """The skeleton model's metrics (eval_skeleton.py:46-68; rotation_error_l2 = train_diffusion_skeleton.py:65-87) per sample
        on the device: pred / gt (B,1,3 n_joints + 3 n_points + 7,T) -> dict of (B,) tensors, means over the frames t >= past_len."""
        pred, gt = self._f32(pred), self._f32(gt)
        B, _, Cn, T = pred.shape
        if gt.shape != pred.shape or (Cn - 7 - 3 * n_joints) % 3 or Cn - 7 - 3 * n_joints <= 0:
            raise EngineError("pred / gt must both be (B,1,3 n_joints + 3 n_points + 7,T)")
        out = torch.empty(5, B, device=self.device)
        self._chk(self.lib.idb_skeleton_metrics(self._h, B, T, int(past_len), int(n_joints), (Cn - 7 - 3 * n_joints) // 3, self._ptr(pred),
                                                self._ptr(gt), self._ptr(out), self._stream()))
        return {k: out[i] for i, k in enumerate(self.SKELETON_METRIC_NAMES)}

    def rollout_next_window(self, body, obj, jtr, T, past_len):
        """get_batch of eval_smpl_long.py:26-84 on the device: (gt (B,1,144,T), centroid (B,3)) of the next window from the
        finished window's body (Tw,B,159), obj (Tw,B,6), jtr (Tw,B,J,3)."""
        body, obj, jtr = self._f32(body), self._f32(obj), self._f32(jtr)
        Tw, B, Db = body.shape
        gt = torch.empty(B, 1, 144, T, device=self.device)
        cen = torch.empty(B, 3, device=self.device)
        if Tw != T:
            raise EngineError("rollout windows share one length T")
        self._chk(self.lib.idb_rollout_next_window(self._h, T, B, jtr.shape[2], Db, int(past_len), self._ptr(body), self._ptr(obj),
                                                   self._ptr(jtr), self._ptr(gt), self._ptr(cen), self._stream()))
        return gt, cen

    def add_offset_(self, x, offset, col0=0, K=None, sign=1.0):
        """x (T,B,...) contiguous float32, in place: the 3-vectors x[t,b,col0+3k : col0+3k+3], k < K, += sign * offset[b]."""
        assert x.is_cuda and x.is_contiguous() and x.dtype == torch.float32
        T, B = x.shape[:2]
        ld = x.numel() // (T * B)
        K = (ld - col0) // 3 if K is None else K
        offset = self._f32(offset)
        self._chk(self.lib.idb_add_offset(self._h, T, B, int(K), ld, int(col0), self._ptr(x), self._ptr(offset), float(sign), self._stream()))
        return x

    def smooth_(self, x, future_len):
        """In place on a contiguous float32 device tensor (T, ...): the reference's `smooth` for one tensor."""
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
        T = x.shape[0]
        self._chk(self.lib.idb_smooth(self._h, T, int(future_len), x.numel() // T, self._ptr(x), self._stream()))
        return x

    def metric_min_(self, acc, cur):
        """acc = min(acc, cur) element-wise, in place (the best-of-N reduction over diverse samples)."""
        assert acc.is_cuda and acc.is_contiguous() and acc.dtype == torch.float32 and acc.shape == cur.shape
        cur = self._f32(cur)
        self._chk(self.lib.idb_metric_min(self._h, acc.numel(), self._ptr(acc), self._ptr(cur), self._stream()))
        return acc

    # ------------------------------------------------------------------ correction
    def load_projector(self, state_dict, past_len, future_len, n_pre=10, n_markers=67):
        self._chk(self.lib.idb_projector_init(self._h, past_len, future_len, n_pre, n_markers))
        for name, w in state_dict.items():
            if not torch.is_tensor(w):
                w = torch.as_tensor(np.asarray(w))
            if not w.dtype.is_floating_point:
                continue
            w = w.detach().to(dtype=torch.float32).contiguous()
            self._chk(self.lib.idb_projector_load(self._h, name.encode(), C.c_void_p(w.data_ptr()), _shape_arr(w.shape), w.dim()))
        self._chk(self.lib.idb_projector_commit(self._h))
        hm = np.asarray(HAND_MARKERS, dtype=np.int32)
        self._chk(self.lib.idb_projector_set_hand_markers(self._h, C.c_void_p(hm.ctypes.data), len(hm)))
        self.past_len, self.future_len = past_len, future_len
        self._projector_owner = None

    def load_projector_skeleton(self, state_dict, past_len, future_len, n_joints=21):
        """the skeleton correction net (reference model/correction_skeleton.py, checkpoints/obj_skeleton.ckpt)"""
        self._chk(self.lib.idb_projector_init_skeleton(self._h, past_len, future_len, n_joints))
        for name, w in state_dict.items():
            if not torch.is_tensor(w):
                w = torch.as_tensor(np.asarray(w))
            if not w.dtype.is_floating_point:
                continue
            w = w.detach().to(dtype=torch.float32).contiguous()
            self._chk(self.lib.idb_projector_load(self._h, name.encode(), C.c_void_p(w.data_ptr()), _shape_arr(w.shape), w.dim()))
        self._chk(self.lib.idb_projector_commit(self._h))
        self.past_len, self.future_len = past_len, future_len
        self._projector_owner = None

    def projector_sample_skeleton(self, obj_quat, obj_trans, joints):
        """ObjProjector.sample of the skeleton net: (T,B,4) xyzw, (T,B,3), (T,B,J,3) -> (quat (T,B,4), trans (T,B,3))"""
        q, t, j = self._f32(obj_quat), self._f32(obj_trans), self._f32(joints)
        T, B, _ = q.shape
        qo, to = torch.empty(T, B, 4, device=self.device), torch.empty(T, B, 3, device=self.device)
        self._chk(self.lib.idb_projector_sample_skeleton(self._h, T, B, self._ptr(q), self._ptr(t), self._ptr(j), self._ptr(qo), self._ptr(to), self._stream()))
        return qo, to

    def skeleton_correction_apply(self, x0, gt, zero_pose_obj, t):
        """In place on x0 (B,1,106,T): the body of the skeleton denoised_fn (eval_skeleton.py:80-111) for an active step."""
        assert x0.is_cuda and x0.is_contiguous() and x0.dtype == torch.float32
        gt, zp = self._f32(gt), self._f32(zero_pose_obj)
        B, _, _, T = x0.shape
        self._chk(self.lib.idb_skeleton_correction_apply(self._h, B, T, zp.shape[1], self._ptr(x0), self._ptr(gt), self._ptr(zp), int(t), self._stream()))
        return x0

    def bind_correction(self, hand_pose, betas, obj_points, past_len=None, marker_ids=None, hand_marker_ids=None):
        hand_pose, betas, obj_points = self._f32(hand_pose), self._f32(betas), self._f32(obj_points)
        T, B, _ = hand_pose.shape
        mk = np.asarray(marker_ids if marker_ids is not None else MARKERSET_SSM67_SMPLH, dtype=np.int32)
        hm = np.asarray(hand_marker_ids if hand_marker_ids is not None else HAND_MARKERS, dtype=np.int32)
        self._chk(self.lib.idb_correction_bind(self._h, B, T, past_len if past_len is not None else self.past_len,
                                               obj_points.shape[1], self._ptr(hand_pose), self._ptr(betas), self._ptr(obj_points),
                                               C.c_void_p(mk.ctypes.data), C.c_void_p(hm.ctypes.data), len(hm), self._stream()))
        self._keep_corr = [hand_pose, betas, obj_points]     # copied asynchronously on the stream
        self.n_markers = len(mk)
        self.n_obj = obj_points.shape[1]
        self.corr_B = B

    def projector_sample(self, obj_angles, obj_trans, markers, contact):
        a, t, m = self._f32(obj_angles), self._f32(obj_trans), self._f32(markers)
        c = contact.to(device=self.device, dtype=torch.int32).contiguous()
        T, B, _ = a.shape
        out = torch.empty(T, B, 9, device=self.device)
        self._chk(self.lib.idb_projector_sample(self._h, T, B, self._ptr(a), self._ptr(t), self._ptr(m), self._ptr(c), self._ptr(out), self._stream()))
        return out

    def correction_log(self, capacity):
        """Parity hook: returns (cond_log [capacity,B] uint8, contact_log [capacity,B,P] int32) device tensors that the next
        `capacity` correction steps enqueued (in-loop or stand-alone) fill in order; capacity 0 switches the log off."""
        if not capacity:
            self._chk(self.lib.idb_correction_set_log(self._h, None, None, 0))
            self._corr_log = None
            return None
        B = self.corr_B
        cond = torch.zeros(capacity, B, dtype=torch.uint8, device=self.device)
        contact = torch.zeros(capacity, B, self.n_markers, dtype=torch.int32, device=self.device)
        self._chk(self.lib.idb_correction_set_log(self._h, self._ptr(cond), self._ptr(contact), int(capacity)))
        self._corr_log = (cond, contact)
        return cond, contact

    def correction_apply(self, x0, gt, t, debug=False):
        """In-place denoised_fn body on x0 (B,1,144,T) for an active step; returns x0 (and the
        decision tensors when debug=True)."""
        assert x0.is_cuda and x0.is_contiguous() and x0.dtype == torch.float32
        gt = self._f32(gt)
        B, _, _, T = x0.shape
        dbg = {}
        cond = contact = markers = o2h = None
        if debug:
            cond = torch.empty(B, dtype=torch.uint8, device=self.device)
            contact = torch.empty(B, self.n_markers, dtype=torch.int32, device=self.device)
            markers = torch.empty(T, B, self.n_markers, 3, device=self.device)
            o2h = torch.empty(T * B, self.n_obj, device=self.device)
        self._chk(self.lib.idb_correction_apply(self._h, self._ptr(x0), self._ptr(gt), int(t), self._ptr(cond), self._ptr(contact),
                                                self._ptr(markers), self._ptr(o2h), self._stream()))
        if debug:
            dbg = dict(condition=cond.bool(), contact=contact, markers=markers, o2h_signed=o2h)
            return x0, dbg
        return x0
