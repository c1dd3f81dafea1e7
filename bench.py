#!/usr/bin/env python
"""bench.py -- HOI denoising-steps/sec on synthetic BEHAVE-shape sequences (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W                      # this repo's CUDA path, BASELINE configs[1]
  python bench.py --config 3|4|5 [--scaling strong] ...              # the other BASELINE configs (see CONFIGS)
  python bench.py --impl reference --gpus N --steps K ...            # the reference's CPU path on the host cores
  python bench.py ... --dump-outputs DIR                             # also write the arrays the last timed step returned
                                                                     # (the sample; for config 5 also the trajectories) to
                                                                     # DIR/<name>.npy, float32; the inputs are seeded

One bench "step" = one full sampling call of the workload on every rank (config 2: SMPL diffusion, 100 DDPM steps,
B=64, T=30, inpainted past of 10 frames); the metric counts the DENOISING steps executed.

  scaling "weak"   (default; the driver's 1/2/4/8 run): every rank samples its own batch of B sequences, no data-path
                   collective (SURVEY 8e);  value = N_ranks * K * n_steps / max-over-ranks time
  scaling "strong" (--scaling strong, and always for configs 4 / 5): ONE global batch sliced into contiguous B/G
                   samples per rank, noise keyed by the global sample index (rank outputs concatenate to the 1-GPU
                   result bit for bit, tests/test_gpu_configs.py::test_batch_slices_bit_identical);
                   value = K * n_steps / max-over-ranks time (one denoising step advances the whole global batch);
                   after the timed region the six per-sample metric vectors of eval_smpl_short.py:73-80 are computed
                   per rank (idb_metrics) and exchanged with ONE all_gather (the path's only collective)

  value : inputs (noise tape, gt, mask, cond, correction context) already resident in HBM, device time (CUDA events)
  e2e   : the same loop through the public Python API with HOST (pinned) buffers: H2D of x_T, gt, mask, cond (and the
          correction context) and D2H of the sample inside the timed region; per-step noise is drawn on the device
          like the reference does (th.randn_like)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs[1..4] (configs[0] is the CPU-runnable skeleton smoke case: a parity test, not a bench line)
CONFIGS = {
    2: dict(name="SMPL diffusion, 100 DDPM steps, B=64, T=30 (past 10 + future 20), 144 channels, inpainting mask on the past, "
                 "no correction (BASELINE configs[1])", B=64, T=30, past=10, steps=100, correction=False, windows=1, strong=False),
    3: dict(name="SMPL diffusion + correction predictor (hook active at t=50 and t=0), 100 DDPM steps, B=64, T=30 (BASELINE configs[2])",
            B=64, T=30, past=10, steps=100, correction=True, windows=1, strong=False),
    4: dict(name="SMPL diffusion + correction (11 hook steps), 1000 DDPM steps, global B=256 sharded over the GPUs, T=30 "
                 "(BASELINE configs[3])", B=256, T=30, past=10, steps=1000, correction=True, windows=1, strong=True),
    5: dict(name="SMPL long-horizon autoregressive rollout (eval_smpl_long), 1 + 10 windows of 100 DDPM steps with correction, "
                 "global B=128 sharded over the GPUs, T=30 (BASELINE configs[4])", B=128, T=30, past=10, steps=100, correction=True,
            windows=11, strong=True),
}
# dram__bytes_read.sum + dram__bytes_write.sum of ONE mlp_fused_kernel launch (ncu --set full, cold caches:
# profiles/r1_ncu_full_mlp.txt)
MLP_DRAM_TRAFFIC_BYTES = 6072576
METRIC = "HOI denoising-steps/sec (B=64,T=30)"
UNIT = "denoising steps/s"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="MEASURED_PEAKS.json")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def workload_config(cfg_id, scaling, world):
    """the `config` object of the JSON line: identical for the product arm and the reference arm"""
    from interdiff_b200.weights import have_ref_weights
    c = CONFIGS[cfg_id]
    strong = c["strong"] or scaling == "strong"
    return dict(workload=c["name"], baseline_config=cfg_id, batch=("global B=%d" % c["B"]) if strong else ("B=%d per GPU" % c["B"]),
                T=c["T"], diffusion_steps=c["steps"], correction=c["correction"], windows=c["windows"],
                scaling="strong" if strong else "weak",
                weights="reference checkpoint (exported)" if have_ref_weights() else "seeded random init")


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own classes when its tree is reachable, else the oracle port
# ------------------------------------------------------------------------------------------------------------------
def _reference_tree():
    for cand in (os.environ.get("INTERDIFF_REF"), os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if cand and os.path.isdir(os.path.join(cand, "interdiff", "model")):
            return cand
    return None


def cpu_reference_rate(cfg_id, n_plain, threads=None, seed=233):
    """Times the reference's CPU path for the workload on a bounded sample: `n_plain` plain p_sample steps of the full
    B x T batch after one untimed step, and - for the correction configs - ONE hook step.  The hook's nearest-neighbour
    search has no CPU implementation upstream (chamfer_distance is CUDA-only, tools.py:9,45): the oracle's restated hook
    (torch argmin over chunked distance matrices) stands in, timed on a 4-sample slice and scaled by the frame count (the
    hook is per-frame work), and reported separately (SURVEY 8d "CPU caveat").
    Returns dict(rate, plain_s, corr_s, cores, kind, sample)."""
    import torch
    from interdiff_b200 import synthetic as S
    from interdiff_b200.weights import bench_weights
    from oracle import restate as R
    c = CONFIGS[cfg_id]
    cores = threads or int(os.environ.get("IDB_CPU_THREADS", "0")) or min(os.cpu_count(), 32)
    torch.set_num_threads(cores)
    B, T, n = c["B"] if not c["strong"] else min(c["B"], 64), c["T"], c["steps"]
    b = S.make_smpl_batch(B=B, T=T, past_len=c["past"], seed=seed)
    gt, mask, cond = torch.from_numpy(b["gt"]), torch.from_numpy(b["mask"]), torch.from_numpy(b["cond"])
    tape = torch.from_numpy(S.noise_tape(b["gt"].shape, n_plain + 1, seed))
    tree = _reference_tree()
    kind = "port"
    if tree:
        try:
            os.environ.setdefault("INTERDIFF_REF", tree)
            from oracle import ref_loader as RL
            model, diffusion, _ = RL.build_mdm_smpl(diffusion_steps=n)
            kw = {"y": {"cond": cond, "inpainted_motion": gt, "inpainting_mask": mask}}

            def step(x, i, k):
                t = torch.full((B,), i, dtype=torch.long)
                return diffusion.p_sample(model, x, t, clip_denoised=False, model_kwargs=kw)["sample"]
            kind = "reference"
        except Exception as e:      # fall back to the port (and say so)
            sys.stderr.write("reference classes unavailable (%r): timing the oracle port\n" % (e,))
            tree = None
    if not tree:
        sd = bench_weights("diffusion_smpl")
        tables = R.diffusion_tables(R.named_beta_schedule("cosine", n))
        fn = lambda x, t: R.mdm_smpl_forward(sd, x, t, cond, faithful=True)   # faithful: 10x replicated LocalAttention input, as upstream

        def step(x, i, k):
            return R.p_sample_step(fn, tables, x, i, tape[1 + k], gt, mask)[0]
    x = tape[0]
    with torch.no_grad():
        x = step(x, n - 1, 0)       # untimed
        t0 = time.perf_counter()
        for k in range(n_plain):
            x = step(x, n - 2 - k, 1 + k)
        plain_s = (time.perf_counter() - t0) / n_plain
    corr_s = 0.0
    n_corr = len([i for i in range(n) if i <= 500 and i % 50 == 0]) if c["correction"] else 0
    if n_corr:
        Bs = 4
        smplh = {k: torch.from_numpy(np.asarray(v)) for k, v in S.make_smplh_model(233, sparse_weights=True).items()}
        bs = S.make_smpl_batch(B=Bs, T=T, past_len=c["past"], seed=seed)
        ctx = dict(past_len=c["past"], future_len=T - c["past"], smpl_dim=132, gt=torch.from_numpy(bs["gt"]), hand_pose=torch.from_numpy(bs["hand_pose"]),
                   betas=torch.from_numpy(bs["betas"]), obj_points=torch.from_numpy(bs["obj_points"]), smplh=smplh,
                   projector=bench_weights("correction_smpl"))
        hook = R.make_denoised_fn(ctx)
        with torch.no_grad():
            t0 = time.perf_counter()
            hook(ctx["gt"].clone(), torch.zeros(Bs, dtype=torch.long), None)
            corr_s = (time.perf_counter() - t0) * (B / Bs)
    total = n * c["windows"]
    n_hook = n_corr * c["windows"]
    loop_s = (total - n_hook) * plain_s + n_hook * (plain_s + corr_s)
    sample = "%d plain p_sample steps of the B=%d, T=%d batch (%.2f s each, %s)" % (
        n_plain, B, T, plain_s, "the reference's own MDM + SpacedDiffusion through oracle/shims.py" if kind == "reference"
        else "oracle.restate faithful port, torch CPU fp32")
    if n_corr:
        sample += "; hook step = plain step + %.1f s (restated hook on a 4-sample slice x %d; argmin stand-in for the CUDA-only chamfer search)" % (corr_s, B // 4)
    if c["strong"] and B != c["B"]:
        sample += "; timed at B=%d and scaled to the global B=%d" % (B, c["B"])
        loop_s *= c["B"] / B
    return dict(rate=total / loop_s, plain_s=plain_s, corr_s=corr_s, cores=cores, kind=kind, sample=sample)


def aggregate_max(values, device=None):
    """max over ranks of per-rank timings (device time of the slowest rank decides); works with the
    nccl (GPU tensors) and gloo (CPU tensors) backends, and without a process group (N = 1)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def rank_seed(rank, base=233):
    """weak scaling: every rank samples its own batch of sequences (distinct, reproducible seeds)"""
    return base + rank


def rank_slice(B, rank, world):
    """strong scaling: contiguous B/G samples of the global batch per rank (SURVEY 8e); B must divide evenly"""
    if B % world:
        raise ValueError("global batch %d does not divide over %d ranks" % (B, world))
    n = B // world
    return slice(rank * n, (rank + 1) * n)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per = 3  # plain denoising steps timed per bench "step" (bounded sample of the workload's loop)
    total = max(1, args.steps) * per
    r = cpu_reference_rate(args.config, total)
    world = args.gpus
    line = dict(impl="reference", metric=METRIC, value=r["rate"], unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1000.0 * r["plain_s"] * per, higher_is_better=True, scaling=workload_config(args.config, args.scaling, world)["scaling"],
                vs_baseline=None, dtype="f32", data="synthetic", config=workload_config(args.config, args.scaling, world),
                cpu_baseline=dict(value=r["rate"], unit=UNIT, cores=r["cores"], kind=r["kind"], sample=r["sample"],
                                  plain_step_s=r["plain_s"], correction_step_extra_s=r["corr_s"]),
                e2e=dict(value=r["rate"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from interdiff_b200 import synthetic as S
    from interdiff_b200.diffusion.gaussian_diffusion import get_named_beta_schedule
    from interdiff_b200.engine import Engine
    from interdiff_b200.sampling import draw_tape_indexed, gather_metrics, sample_postprocess, sample_smpl_host
    from interdiff_b200.weights import bench_weights

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    c = CONFIGS[args.config]
    strong = c["strong"] or args.scaling == "strong"
    n, T = c["steps"], c["T"]
    eng = Engine(dev)
    if args.backend:
        eng.set_gemm_backend(args.backend)
    eng.load_denoiser(bench_weights("diffusion_smpl"), "smpl")
    if strong:
        sl = rank_slice(c["B"], rank, world)
        gb = S.make_smpl_batch(B=c["B"], T=T, past_len=c["past"], seed=233)       # ONE global batch, sliced
        b = {k: np.ascontiguousarray(v[sl] if k in ("gt", "mask", "obj_points") else v[:, sl]) for k, v in gb.items() if isinstance(v, np.ndarray)}
        ids = list(range(sl.start, sl.stop))
    else:
        b = S.make_smpl_batch(B=c["B"], T=T, past_len=c["past"], seed=rank_seed(rank))   # each rank its own sequences
        ids = [rank * c["B"] + j for j in range(c["B"])]
    Bl = b["gt"].shape[0]
    eng.init_diffusion(get_named_beta_schedule("cosine", n))
    shape = b["gt"].shape
    if c["correction"]:
        smplh = S.make_smplh_model(233, sparse_weights=True)       # <= 4 non-zero skinning weights per vertex, as SMPL-H is painted
        eng.load_body(smplh)
        eng.load_projector(bench_weights("correction_smpl"), c["past"], T - c["past"])
    # ---- device-resident leg
    gt_d, mask_d, cond_d = torch.from_numpy(b["gt"]).to(dev), torch.from_numpy(b["mask"]).to(dev), torch.from_numpy(b["cond"]).to(dev)
    eng.bind(cond_d, T)
    if c["correction"]:
        eng.bind_correction(b["hand_pose"], b["betas"], b["obj_points"], past_len=c["past"])
    tape_d = draw_tape_indexed(eng, shape[1:], n, ids, seed=233)              # noise keyed by the GLOBAL sample index
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)  # > 126 MB L2
    out = torch.empty(shape, device=dev)
    rollout = None
    if c["windows"] > 1:
        from interdiff_b200.rollout import RolloutDriver
        rollout = RolloutDriver(eng, past_len=c["past"], n_windows=c["windows"] - 1)

    def one_call():
        """one sampling call; returns what its caller receives: the sample, and for the rollout the world-coordinate
        trajectories as well"""
        if rollout is None:
            return dict(sample=eng.p_sample_loop(tape_d, gt_d, mask_d, correction=c["correction"], use_graph=True, out=out))
        traj = rollout.run(tape_d, gt_d, mask_d, torch.from_numpy(b["hand_pose"]).to(dev), torch.from_numpy(b["betas"]).to(dev), out)
        return dict(sample=out, **traj)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(3, args.warmup)):
        one_call()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = eng.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for s, e in ev:
        flush.fill_(1.0)  # evict L2 between timed iterations (outside the event pair)
        s.record()
        result = one_call()
        e.record()
    barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs:
        # host copies now: the legs below reuse the device buffers
        dump = {k: v.detach().cpu().numpy() for k, v in result.items()}
    launches = eng.launch_count - l0
    dev_ms = sum(s.elapsed_time(e) for s, e in ev)
    # ---- end-to-end leg through the public API with host buffers
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_gt, h_mask, h_cond, h_xT = pin(b["gt"]), pin(b["mask"]), pin(b["cond"]), pin(S.noise_tape(shape, 0, 233 + rank)[0])
    h_ctx = dict(hand_pose=pin(b["hand_pose"]), betas=pin(b["betas"]), obj_points=pin(b["obj_points"]), past_len=c["past"]) if c["correction"] else None
    h_out = torch.empty(shape).pin_memory()
    e2e_ms = None
    if rollout is None:
        for _ in range(2):
            sample_smpl_host(eng, h_xT, h_gt, h_mask, h_cond, h_out, seed=1, correction=h_ctx)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for it in range(args.steps):
            sample_smpl_host(eng, h_xT, h_gt, h_mask, h_cond, h_out, seed=2 + it, correction=h_ctx)
        e1.record()
        barrier()
        e2e_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    # ---- metric collection: the path's only collective (strong scaling / multi-GPU): six (B/G,) vectors per rank, one all_gather
    gathered = None
    if c["correction"] and rollout is None:
        hp, bt = torch.from_numpy(b["hand_pose"]).to(dev), torch.from_numpy(b["betas"]).to(dev)
        body, obj, verts, jtr = sample_postprocess(eng, out, hp, bt)
        body_g, obj_g, _, jtr_g = sample_postprocess(eng, gt_d, hp, bt)
        P = c["past"]
        m = eng.metrics(obj[P:], jtr[P:], body[P:], obj_g[P:], jtr_g[P:], body_g[P:], verts[P:], torch.from_numpy(b["obj_points"]).to(dev))
        block = torch.stack([m[k] for k in eng.METRIC_NAMES])          # (6, B/G)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        allm = gather_metrics(block)
        g1.record()
        torch.cuda.synchronize(dev)
        gathered = dict(names=list(eng.METRIC_NAMES), mean=[float(v) for v in allm.mean(dim=1)], samples=int(allm.shape[1]),
                        all_gather_ms=g0.elapsed_time(g1), collective="all_gather of a (6, %d) fp32 block per rank" % block.shape[1])
    # ---- roofline of the dominant kernel: the fused feed-forward block (8 launches per step), timed alone: mean of 200
    # back-to-back launches, CUDA events on its stream; rows = this rank's token count
    M = Bl * T
    g = torch.Generator().manual_seed(0)
    rx, rw1, rb1 = torch.randn(M, 256, generator=g), torch.randn(1024, 256, generator=g) / 16, torch.randn(1024, generator=g) * 0.1
    rw2, rb2, rres = torch.randn(256, 1024, generator=g) / 32, torch.randn(256, generator=g) * 0.1, torch.randn(M, 256, generator=g)
    eng.mlp(rx, rw1, rb1, rw2, rb2, rres, iters=5)
    eng.mlp(rx, rw1, rb1, rw2, rb2, rres, iters=201)
    roof = dict(ms=eng.last_ms(), flops=2.0 * M * (256 * 1024 + 1024 * 256), iters=200,
                kernel="mlp_fused_kernel (gelu(X W1^T + b1) W2^T + b2 + R, M=%d, d_model 256, d_ff 1024)" % M)
    lbs = None
    if c["correction"]:
        F = T * Bl
        gg = torch.Generator().manual_seed(0)
        pose, betas, trans = (0.3 * torch.randn(F, 156, generator=gg)).to(dev), torch.randn(F, 10, generator=gg).to(dev), torch.randn(F, 3, generator=gg).to(dev)
        for _ in range(3):
            eng.lbs(pose, betas, trans, want_jtr=False)
        tot = 0.0
        for _ in range(10):
            flush.fill_(1.0)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            eng.lbs(pose, betas, trans, want_jtr=False)
            a1.record()
            torch.cuda.synchronize(dev)
            tot += a0.elapsed_time(a1)
        lbs = dict(ms=tot / 10, F=F, bytes=41.7e6 + F * 84.0e3, flops=F * 33.2e6)

    agg = aggregate_max([dev_ms, e2e_ms if e2e_ms is not None else 0.0], device=dev)
    dev_ms, e2e_ms = agg[0], (agg[1] if e2e_ms is not None else None)
    if rank == 0:
        peaks = _peaks()
        per_call = n * c["windows"]
        total_steps = (1 if strong else world) * args.steps * per_call
        value = total_steps / (dev_ms / 1000.0)
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(3, args.warmup),
                    ms_per_step=dev_ms / args.steps, higher_is_better=True, scaling="strong" if strong else "weak", vs_baseline=None,
                    dtype="f32 (fp32 SIMT GEMMs)" if args.backend == "simt" else "f32-grade (GEMMs: fp16 hi/lo split pairs on tcgen05, fp32 TMEM accumulate; rest fp32)",
                    data="synthetic", config=workload_config(args.config, args.scaling, world),
                    run=dict(l2="flushed between timed iterations (256 MB fill outside the event pair)", cuda_graph="whole loop as one graph",
                             gemm_backend=args.backend or "tcgen05", batch_per_gpu=Bl, us_per_denoising_step=1000.0 * dev_ms / args.steps / per_call,
                             sample_steps_per_s=value * (c["B"] if strong else Bl),
                             body_model="synthetic SMPL-H-shaped model, <= 4 non-zero skinning weights per vertex" if c["correction"] else None),
                    gpu_launches=int(launches), clocks=clocks, wall_s=wall)
        if e2e_ms is not None:
            h2d = int(h_gt.numel() * 4 + h_mask.numel() + h_cond.numel() * 4 + h_xT.numel() * 4)
            if h_ctx:
                h2d += int(sum(h_ctx[k].numel() * 4 for k in ("hand_pose", "betas", "obj_points")))
            line["e2e"] = dict(value=total_steps / (e2e_ms / 1000.0), unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=int(h_out.numel() * 4))
        else:
            line["e2e"] = dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0,
                               note="rollout driver: the device-resident loop IS the public call (no separate host-buffer leg)")
        if gathered:
            line["metrics"] = gathered
        if roof and roof["ms"] > 0:
            ach = roof["flops"] / (roof["ms"] * 1e-3) / 1e12
            line["roofline"] = dict(bound="tensor", kernel=roof["kernel"], achieved=ach, peak=peaks["bf16_tflops"], unit="TFLOP/s",
                                    frac=ach / peaks["bf16_tflops"], traffic=MLP_DRAM_TRAFFIC_BYTES, us_per_launch=roof["ms"] * 1e3,
                                    peak_source=peaks["source"] + " (burst bf16)",
                                    issue_ceiling=peaks["bf16_tflops"] / 3.0, frac_of_issue_ceiling=ach / (peaks["bf16_tflops"] / 3.0),
                                    note="algorithmic flops 2*M*(256*1024 + 1024*256) = %.3f GFLOP per launch / mean time of %d back-to-back "
                                         "launches (CUDA events); the split-precision kernel issues 3 fp16 MMAs per algorithmic MAC, so its "
                                         "ceiling is 1/3 of the fp16/bf16 peak; at M=%d the launch is one wave of %d CTAs bound by "
                                         "fixed latencies (DESIGN.md 4.1b timeline), not by the tensor pipe; traffic = dram bytes per "
                                         "launch from the ncu --set full capture in profiles/ (operands are L2 resident in the loop)"
                                         % (roof["flops"] / 1e9, roof["iters"], M, 8 * ((M + 127) // 128)))
        if lbs:
            gbs = lbs["bytes"] / (lbs["ms"] * 1e-3) / 1e9
            tf = lbs["flops"] / (lbs["ms"] * 1e-3) / 1e12
            line["roofline_lbs"] = dict(bound="hbm", kernel="SMPL-H LBS (k_lbs_pose + tcgen05 blend GEMM + k_lbs_skin_sparse), F=%d frames" % lbs["F"],
                                        achieved=gbs, peak=peaks["hbm_gbs"], unit="GB/s", frac=gbs / peaks["hbm_gbs"], ms=lbs["ms"],
                                        algorithmic_bytes=lbs["bytes"], tflops=tf, tflops_frac_of_bf16_peak=tf / peaks["bf16_tflops"],
                                        note="algorithmic bytes = constants once (41.7 MB) + 84.0 KB per frame (SURVEY 8d); 33.2 MFLOP per frame; "
                                             "L2 flushed before each of 10 timed calls")
        if world == 1 and not args.no_cpu:
            r = cpu_reference_rate(args.config, args.cpu_steps)
            line["cpu_baseline"] = dict(value=r["rate"], unit=UNIT, cores=r["cores"], kind=r["kind"], sample=r["sample"],
                                        plain_step_s=r["plain_s"], correction_step_extra_s=r["corr_s"])
        print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dump, rank if world > 1 else None)
    if world > 1:
        dist.destroy_process_group()
    eng.close()


def dump_outputs(directory, arrays, rank=None):
    """<directory>/<name>.npy (float32) of each array of the last timed step, <name>_rank<r>.npy for multi-rank runs:
    two builds run with the same arguments sample the same inputs, so their files compare output for output"""
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "outputs above 64 MB: dump a sample instead"
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ("" if rank is None else "_rank%d" % rank) + ".npy"), a.astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed sampling calls (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--backend", default=None, choices=[None, "simt", "tcgen05"])
    ap.add_argument("--cpu-steps", type=int, default=6)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step returned to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
