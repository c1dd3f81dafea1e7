"""Sampling drivers on top of the Engine (the L4 layer of SURVEY section 1).

sample_smpl_host is the end-to-end call bench.py times: host (pinned) buffers in, host buffer
out, everything in between on the device.  Mirrors reference eval_smpl_short.py:179-192
(sample_once) up to the final sample: model_kwargs = {cond, inpainted_motion, inpainting_mask},
noise = x_T, diffusion.p_sample_loop(model, shape, clip_denoised=False, noise, model_kwargs).
"""
import torch


def draw_tape(engine, x_T, n_steps, seed=None):
    """(n_steps+1, *shape) device tensor: tape[0] = x_T, tape[1:] = per-step eps drawn on the
    device (the reference draws th.randn_like(x) every step, gaussian_diffusion.py:532)."""
    tape = torch.empty((n_steps + 1,) + tuple(x_T.shape), device=engine.device)
    tape[0].copy_(x_T, non_blocking=True)
    g = None
    if seed is not None:
        g = torch.Generator(device=engine.device)
        g.manual_seed(int(seed))
    tape[1:].normal_(generator=g)
    return tape


def draw_tape_indexed(engine, sample_shape, n_steps, global_ids, seed=233):
    """(n_steps+1, B, *sample_shape) device tape whose column j depends ONLY on (seed, global_ids[j]): the noise of a
    sample is keyed by its index in the GLOBAL batch, so a multi-GPU run that slices one global batch reproduces the
    single-GPU trajectories (SURVEY 8e).  sample_shape = (1, C, T)."""
    B = len(global_ids)
    tape = torch.empty((n_steps + 1, B) + tuple(sample_shape), device=engine.device)
    g = torch.Generator(device=engine.device)
    for j, gid in enumerate(global_ids):
        g.manual_seed(int(seed) * 1000003 + int(gid))
        tape[:, j] = torch.randn((n_steps + 1,) + tuple(sample_shape), generator=g, device=engine.device)
    return tape


def sample_smpl_host(engine, h_xT, h_gt, h_mask, h_cond, h_out, seed=None, correction=False, use_graph=True):
    """One sampling call with host tensors (pinned for async copies).  The engine must have its
    denoiser loaded and its diffusion initialised.  correction: False, or the hook's per-batch context as HOST tensors
    dict(hand_pose (T,B,90), betas (T,B,10), obj_points (B,P,3), past_len) - body model and projector already loaded -
    which is uploaded and bound inside the call like the rest of the inputs."""
    dev = engine.device
    gt = h_gt.to(dev, non_blocking=True)
    mask = h_mask.to(dev, non_blocking=True)
    cond = h_cond.to(dev, non_blocking=True)
    xT = h_xT.to(dev, non_blocking=True)
    T = gt.shape[-1]
    engine.bind(cond, T)
    if correction:
        engine.bind_correction(correction["hand_pose"].to(dev, non_blocking=True), correction["betas"].to(dev, non_blocking=True),
                               correction["obj_points"].to(dev, non_blocking=True), past_len=correction["past_len"])
    # keep the tape buffer across calls (same shape) so the captured graph stays valid
    key = (tuple(gt.shape), engine.n_steps)
    cache = getattr(engine, "_host_loop_cache", None)
    if cache is None or cache[0] != key:
        cache = (key, torch.empty((engine.n_steps + 1,) + tuple(gt.shape), device=dev), torch.empty_like(gt), torch.empty_like(mask),
                 torch.empty_like(gt))
        engine._host_loop_cache = cache
    _, tape, gt_buf, mask_buf, out = cache
    gt_buf.copy_(gt)
    mask_buf.copy_(mask)
    tape[0].copy_(xT)
    g = None
    if seed is not None:
        g = torch.Generator(device=dev)
        g.manual_seed(int(seed))
    tape[1:].normal_(generator=g)
    engine.p_sample_loop(tape, gt_buf, mask_buf, correction=bool(correction), use_graph=use_graph, out=out)
    h_out.copy_(out, non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    return h_out


class FusedCorrection:
    """The reference's denoised_fn hook (eval_smpl_short.py:84-130) as an object the diffusion
    recognises: with it p_sample_loop keeps the whole loop, including the correction steps, inside
    the library.  Called directly (x, t, model_kwargs) it applies the same gate and runs the fused
    correction kernels on x in place, so it also works as a plain denoised_fn callback.

    model_kwargs['y'] must carry what the reference's hook reads: inpainted_motion, hand_pose
    (T,B,90), smpl (interdiff_b200 SMPL_Layer), beta (T,B,10), obj_model (object with .model =
    interdiff_b200 ObjProjector) and obj_points (B,P,3)."""
    is_fused_correction = True

    def __init__(self, past_len):
        self.past_len = past_len
        self._bound = None

    def bind(self, eng, model_kwargs):
        y = model_kwargs["y"]
        y["smpl"].load_into(eng)
        y["obj_model"].model.load_into(eng)
        hp, beta, pts = y["hand_pose"], y["beta"], y["obj_points"]
        key = (id(eng), hp.data_ptr(), hp._version, beta.data_ptr(), beta._version, pts.data_ptr(), pts._version)
        if self._bound != key:
            eng.bind_correction(hp, beta, pts, past_len=self.past_len)
            self._bound = key
        return eng

    def __call__(self, x, t, model_kwargs):
        ti = int(t[0])
        if ti > 500 or ti % 50 != 0:
            return x
        y = model_kwargs["y"]
        eng = y["smpl"].engine_for(x.device) if not hasattr(self, "_eng") else self._eng
        self.bind(eng, model_kwargs)
        return eng.correction_apply(x, y["inpainted_motion"], ti)


class FusedSkeletonCorrection:
    """The skeleton model's denoised_fn hook (eval_skeleton.py:80-111) as an object the diffusion recognises, the counterpart
    of FusedCorrection: with it p_sample_loop keeps eval_skeleton's whole loop, including the correction steps, inside the
    library.  Called directly (x, t, model_kwargs) it applies the same gate and runs the fused hook on x in place, so it also
    works as a plain denoised_fn callback.

    model_kwargs must carry what the reference's hook reads: y['inpainted_motion'] (B,1,106,T), y['obj_model'] (object with
    .model = interdiff_b200 skeleton ObjProjector) and zero_pose_obj (B,12,3), which is bound together with the denoiser."""
    is_fused_correction = True

    def bind(self, eng, model_kwargs):
        model_kwargs["y"]["obj_model"].model.load_into(eng)
        return eng

    def __call__(self, x, t, model_kwargs):
        ti = int(t[0])
        if ti > 500 or ti % 50 != 0:
            return x
        proj = model_kwargs["y"]["obj_model"].model
        eng = proj.engine_for(x.device)
        return eng.skeleton_correction_apply(x, model_kwargs["y"]["inpainted_motion"], model_kwargs["zero_pose_obj"], ti)


def sample_postprocess(engine, sample, hand_pose, betas, past_len=10, future_len=None):
    """Tail of sample_once(_proj) (eval_smpl_short.py:154-173): 6D -> axis-angle and SMPL-H LBS of
    all T*B frames.  Returns body pose (T,B,159), object pose (T,B,6), verts (T,B,V,3), joints."""
    B, _, C, T = sample.shape
    xs = sample.squeeze(1).permute(2, 0, 1).contiguous()            # (T,B,144)
    body_rot = engine.rot6d_to_axis_angle(xs[..., :132].reshape(T, B, 22, 6)).reshape(T, B, 66)
    obj_rot = engine.rot6d_to_axis_angle(xs[..., 135:141].reshape(T, B, 1, 6)).reshape(T, B, 3)
    body = torch.cat([body_rot, hand_pose, xs[..., 132:135]], dim=2)
    bb = body.reshape(T * B, -1)
    verts, jtr = engine.lbs(bb[:, :-3], betas.reshape(T * B, -1), bb[:, -3:])
    return body, torch.cat([obj_rot, xs[..., 141:144]], dim=2), verts.view(T, B, -1, 3), jtr.view(T, B, -1, 3)


def smooth(obj, body, verts, jtrs, pelvis, future_len, engine=None):
    """Reference eval_smpl_short.py:217-223: shift every predicted future frame by the second-difference jump at the
    past/future seam, x[-F:] += 2 x[-F-1] - x[-F-2] - x[-F]; in place on (T, ...) tensors.  Device tensors go through the
    library (`idb_smooth`; pass the engine, or one is looked up for the tensor's device); host tensors (e.g. unit tests of
    the formula) take the same expression in torch."""
    F = int(future_len)
    for x in (obj, body, verts, jtrs, pelvis):
        if x.is_cuda:
            eng = engine if engine is not None else _engine_for(x.device)
            if x.is_contiguous() and x.dtype == torch.float32:
                eng.smooth_(x, F)
            else:
                y = x.float().contiguous()
                eng.smooth_(y, F)
                x.copy_(y)
        else:
            x[-F:] = x[-F:] + (2 * x[-F - 1] - x[-F - 2] - x[-F])
    return obj, body, verts, jtrs, pelvis


_ENGINES = {}


def _engine_for(device):
    from .engine import Engine
    device = torch.device(device)
    if device not in _ENGINES:
        _ENGINES[device] = Engine(device)
    return _ENGINES[device]


def gather_metrics(block):
    """The path's only collective (SURVEY 8e): ONE all_gather of the (6, B/G) per-sample metric block of every rank
    (the six (B,) vectors `metrics` returns, eval_smpl_short.py:73-80) -> (6, B) in global sample order on every rank.
    nccl (device tensors) and gloo (CPU tensors) both work; without a process group the block is returned as is."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return block
    parts = [torch.empty_like(block) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, block.contiguous())
    return torch.cat(parts, dim=1)


class BestOfSamples:
    """The diverse-sample reduction of the reference's evaluation loop (eval_smpl_short.py:268-296): per batch every
    metric starts at 1e10, each of the `diverse_samples` draws contributes its per-sample metric vector, the
    element-wise minimum over the draws is averaged over the batch and accumulated over batches.  Device metric vectors
    are reduced in the library (`idb_metric_min`) on one (6, B) block; with `gather=True` the block of every rank is
    exchanged with one all_gather before the batch mean (multi-GPU evaluation of a sliced batch)."""

    def __init__(self, names=("global_mpjpe", "local_mpjpe", "body_translation", "obj_translation", "obj_rot_error", "penetrate"),
                 engine=None, gather=False):
        self.names = tuple(names)
        self.totals = {k: 0.0 for k in self.names}
        self.batches = 0
        self._cur = None
        self.engine, self.gather = engine, gather

    def start_batch(self):
        self._cur = None

    def add(self, metric):
        """metric: {name: (B,) tensor} of one draw (Engine.metrics output)."""
        block = torch.stack([metric[k].float() for k in self.names]).contiguous()
        if self._cur is None:
            self._cur = torch.full_like(block, 1e10)
        if block.is_cuda:
            (self.engine if self.engine is not None else _engine_for(block.device)).metric_min_(self._cur, block)
        else:
            self._cur = torch.minimum(self._cur, block)

    def end_batch(self):
        cur = gather_metrics(self._cur) if self.gather else self._cur
        means = cur.mean(dim=1).tolist()
        for k, v in zip(self.names, means):
            self.totals[k] += v
        self.batches += 1
        self._cur = None

    def averages(self):
        return {k: v / max(self.batches, 1) for k, v in self.totals.items()}
