#!/usr/bin/env python
"""Headline benchmark: V-JEPA pre-training step, clips/sec, ViT-L/16 16x224x224 synthetic, B=32 per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config vitl16|vith16|vith16_384|tiny]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is everything inside the reference's train_step() (app/vjepa/train.py:414-498) minus the three
logging helpers (grad_logger x2, adamw_logger): LR/WD schedule, target forward + LN + gather, context
encoder + predictor forward/backward, L1 loss, GradScaler, AdamW, zero_grad, EMA; N>1 adds the DDP gradient
all-reduce.  `value` times K such steps with inputs resident in HBM (CUDA events, max over ranks); `e2e`
repeats them through the public module API with HOST inputs: pinned clips + masks copied to the device and
the loss read back every step.  `--impl reference` times the UNMODIFIED reference's CPU path (baseline/_ref, its own
app.vjepa.train.main, fp32) on the host cores; if baseline/_ref is absent it falls back to the CPU oracle port.
`--dump-outputs DIR` writes what the last timed step computed to DIR (see dump_outputs).
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

VITL16_MASKS = [
    dict(aspect_ratio=[0.75, 1.5], num_blocks=8, spatial_scale=[0.15, 0.15], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
    dict(aspect_ratio=[0.75, 1.5], num_blocks=2, spatial_scale=[0.7, 0.7], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
]
CONFIGS = {
    # name: (model_name, embed D, depth L, heads, crop, frames, batch/GPU)
    "vitl16": ("vit_large", 1024, 24, 16, 224, 16, 32),
    "vith16": ("vit_huge", 1280, 32, 16, 224, 16, 24),
    "vith16_384": ("vit_huge", 1280, 32, 16, 384, 16, 10),
    "tiny": ("vit_tiny", 192, 12, 3, 224, 8, 2),
}
PRED_DIM, PRED_DEPTH = 384, 12
OPT = dict(wd=0.04, final_wd=0.4, start_lr=0.0002, lr=0.000625, final_lr=1e-6, warmup=40, epochs=300, ipe=300,
           ipe_scale=1.25, ema=(0.998, 1.0))


def flops_per_clip(D, L, N, Ke, Kp, Dp=PRED_DIM, Lp=PRED_DEPTH, P=1536):
    """SURVEY.md section 8d / BASELINE.md section 2: algorithmic FLOPs of one clip's train step."""
    blk = lambda S, d: 24 * d * d * S + 4 * S * S * d
    f_tgt = L * blk(N, D) + 2 * P * D * N
    f_ctx = sum(L * blk(k, D) for k in Ke)
    f_pe = 2 * P * D * sum(Ke)
    f_pred = sum(Lp * blk(ke + kp, Dp) for ke, kp in zip(Ke, Kp)) + 2 * D * Dp * sum(k1 + k2 for k1, k2 in zip(Ke, Kp))
    return f_tgt + 3 * (f_ctx + f_pred) + 2 * f_pe


def gemm_flops_per_clip(D, L, N, Ke, Kp, Dp=PRED_DIM, Lp=PRED_DEPTH, P=1536):
    """Same accounting restricted to the Linear / patch-embed GEMMs (what gemm_kernel executes)."""
    lin = lambda S, d: 24 * d * d * S
    f_tgt = L * lin(N, D) + 2 * P * D * N
    f_ctx = sum(L * lin(k, D) for k in Ke)
    f_pe = 2 * P * D * sum(Ke)
    f_pred = sum(Lp * lin(ke + kp, Dp) for ke, kp in zip(Ke, Kp)) + 2 * D * Dp * sum(k1 + k2 for k1, k2 in zip(Ke, Kp))
    return f_tgt + 3 * (f_ctx + f_pred) + 2 * f_pe


def seeded_masks(crop, frames, B, seed=0):
    from src.masks.multiblock3d import MaskCollator
    torch.manual_seed(seed)
    coll = MaskCollator(cfgs_mask=VITL16_MASKS, crop_size=crop, num_frames=frames, patch_size=16, tubelet_size=2)
    _, me, mp = coll([torch.zeros(1) for _ in range(B)])
    return me, mp


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(bf16_burst=d.get("bf16_tflops"), bf16_sustained=d.get("bf16_tflops_sustained"),
                    hbm_gbs=d.get("hbm_gbs"), source="measured")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def build_training_state(cfg_name, device, world, rank):
    from app.vjepa.utils import init_opt, init_video_model
    import copy
    model_name, D, L, heads, crop, frames, B = CONFIGS[cfg_name]
    torch.manual_seed(0)
    encoder, predictor = init_video_model(device=device, patch_size=16, num_frames=frames, tubelet_size=2,
                                          model_name=model_name, crop_size=crop, pred_depth=PRED_DEPTH,
                                          pred_embed_dim=PRED_DIM, uniform_power=True, use_mask_tokens=True,
                                          num_mask_tokens=2, zero_init_mask_tokens=True, use_sdpa=True)
    target = copy.deepcopy(encoder)
    optimizer, scaler, scheduler, wd_scheduler = init_opt(
        encoder=encoder, predictor=predictor, wd=OPT["wd"], final_wd=OPT["final_wd"], start_lr=OPT["start_lr"],
        ref_lr=OPT["lr"], final_lr=OPT["final_lr"], iterations_per_epoch=OPT["ipe"], warmup=OPT["warmup"],
        num_epochs=OPT["epochs"], ipe_scale=OPT["ipe_scale"], mixed_precision=True)
    if world > 1:
        if os.environ.get("VJ_TORCH_DDP"):   # A/B: torch's reducer buckets instead of the flat-buffer exchange
            from torch.nn.parallel import DistributedDataParallel as DDP
        else:
            from jepa_b200.distributed import DistributedDataParallel as DDP
        encoder = DDP(encoder, static_graph=True)
        predictor = DDP(predictor, static_graph=True)
        target = DDP(target)
    for p in target.parameters():
        p.requires_grad = False
    total = int(OPT["ipe"] * OPT["epochs"] * OPT["ipe_scale"])
    momentum = (OPT["ema"][0] + i * (OPT["ema"][1] - OPT["ema"][0]) / total for i in range(total + 1))
    return dict(encoder=encoder, predictor=predictor, target=target, optimizer=optimizer, scaler=scaler,
                scheduler=scheduler, wd_scheduler=wd_scheduler, momentum=momentum)


def train_step(st, clips, masks_enc, masks_pred, loggers=False, outputs=None):
    """train_step() of app/vjepa/train.py:414-498; returns the loss (device scalar).  loggers=False is SURVEY 8d's (A)
    math step (grad_logger x2 / adamw_logger off on both arms), loggers=True the as-shipped step (B).  A dict passed as
    `outputs` receives the step's predictions z and targets h."""
    from jepa_b200 import step as vj
    st["scheduler"].step()
    st["wd_scheduler"].step()
    h = vj.forward_target(st["target"], clips, masks_pred)
    z = st["encoder"](clips, masks_enc)
    z = st["predictor"](z, h, masks_enc, masks_pred)
    if outputs is not None:
        outputs.update(z=[t.detach() for t in z], h=h)
    loss = vj.jepa_loss(z, h)
    vj.reg_loss(z)
    scaler, opt = st["scaler"], st["optimizer"]
    scaler.scale(loss).backward()
    scaler.unscale_(opt)
    scaler.step(opt)
    scaler.update()
    if loggers:
        from src.utils.logging import adamw_logger, grad_logger
        grad_logger(st["encoder"].named_parameters())
        grad_logger(st["predictor"].named_parameters())
    opt.zero_grad()
    if loggers:
        adamw_logger(opt)
    vj.ema_update(st["encoder"], st["target"], next(st["momentum"]))
    return loss.detach()


def ddp_gradient_check(st, clips, masks_enc, masks_pred):
    """N > 1: the in-backward flat-buffer exchange (jepa_b200.distributed.FlatGradSync) must leave, on every rank, the mean
    of the per-rank gradients.  One backward WITH the exchange, one without it followed by a plain NCCL all-reduce(AVG) of
    the whole gradient vector; returns the rel-L2 distance (split-K wgrads are TMA reduce-adds, so the two backward passes
    differ by fp32 summation order, ~1e-6).  Makes the SCALE run itself prove gradient equality."""
    import torch.distributed as dist
    from jepa_b200 import step as vj

    def backward_once():
        h = vj.forward_target(st["target"], clips, masks_pred)
        z = st["encoder"](clips, masks_enc)
        z = st["predictor"](z, h, masks_enc, masks_pred)
        vj.jepa_loss(z, h).backward()
        out = []
        for net in (st["encoder"], st["predictor"]):
            out.append(torch.cat([p.grad.reshape(-1) for p in net.parameters() if p.grad is not None]).clone())
        st["optimizer"].zero_grad()
        return torch.cat(out)

    g_sync = backward_once()
    stash = []
    for net in (st["encoder"], st["predictor"]):
        for m in net.modules():
            if getattr(m, "_vj_grad_sync", None) is not None:
                stash.append((m, m._vj_grad_sync))
                m._vj_grad_sync = None
    try:
        g_local = backward_once()
    finally:
        for m, sy in stash:
            m._vj_grad_sync = sy
    g_mean = g_local.clone()
    dist.all_reduce(g_mean, op=dist.ReduceOp.AVG)
    torch.cuda.synchronize()
    rel = float((g_sync - g_mean).norm() / g_mean.norm())
    # the exchange must have DONE something: local and averaged gradients differ (different clips per rank)
    spread = float((g_local - g_mean).norm() / g_mean.norm())
    t = torch.tensor([rel, -spread], device=clips.device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return dict(rel_l2_sync_vs_allreduce_mean=float(t[0]), rel_l2_local_vs_mean_min=float(-t[1]), n_synced_modules=len(stash),
                n_grad_elements=int(g_mean.numel()))


def ncu_gemm_traffic(cfg_name):
    """DRAM bytes moved by the GEMM family in one step, from the committed ncu launch list of `bench.py --profile`
    (profiles/, vitl16 only); None when no capture exists for this config."""
    prof = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles")
    path = next((p for p in (os.path.join(prof, "r02_step_launches_summary.txt"),
                             os.path.join(prof, "r01_step_launches_final_summary.txt")) if os.path.exists(p)), "")
    if cfg_name != "vitl16" or not path:
        return None
    with open(path) as f:
        for line in f:
            if line.startswith("# gemm family:"):
                return int(float(line.split("DRAM traffic")[1].split("GB")[0]) * 1e9)
    return None


DUMP_SAMPLES = 1 << 20          # elements kept of each larger predicted / target array
DUMP_PARAM_SAMPLES = 4096       # elements kept of each larger parameter tensor


def dump_outputs(out_dir, st, loss, step_out):
    """`--dump-outputs DIR`: what the last timed step computed, as float32 DIR/<name>.npy - loss, the predictions z_<i>
    and targets h_<i> of every mask, and the encoder / predictor / target_encoder parameters the step left behind
    (AdamW and EMA applied; each tensor's sample concatenated in named_parameters order).  A larger array is written as
    its elements at positions drawn from a fixed seed, the same in every run of the same config, so the outputs of two
    builds can be compared element for element.  About 23 MB for ViT-L/16.  The step is not bit-reproducible (split-K
    weight gradients are reduce-adds in varying order): two runs of one build, vitl16 --steps 10 on a B200 at 1000 W,
    differed by rel-L2 ~1e-6 in loss, ~1e-5 in the weights, 3e-3 in z and 1e-2 in h."""
    import numpy as np
    from jepa_b200.step import unwrap

    def sample(t, n, seed):
        flat = t.detach().reshape(-1)
        if flat.numel() > n:
            idx = torch.randint(flat.numel(), (n,), generator=torch.Generator().manual_seed(seed))
            flat = flat[idx.to(flat.device)]
        return flat.float().cpu().numpy()

    arrays = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
    for i, (z, h) in enumerate(zip(step_out["z"], step_out["h"])):
        arrays[f"z_{i}"] = sample(z, DUMP_SAMPLES, seed=2 * i)
        arrays[f"h_{i}"] = sample(h, DUMP_SAMPLES, seed=2 * i + 1)
    for name, key in (("encoder", "encoder"), ("predictor", "predictor"), ("target_encoder", "target")):
        params = [p for _, p in unwrap(st[key]).named_parameters()]
        arrays[name] = np.concatenate([sample(p, DUMP_PARAM_SAMPLES, seed=j) for j, p in enumerate(params)])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch.distributed as dist
    from jepa_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 through torch.distributed.run")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        from jepa_b200.distributed import nccl_pg_options
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device, pg_options=nccl_pg_options())
    lib = _lib.load()

    model_name, D, L, heads, crop, frames, B = CONFIGS[args.config]
    if args.batch:
        B = args.batch
    N = (frames // 2) * (crop // 16) ** 2
    me, mp = seeded_masks(crop, frames, B, seed=0)   # first call of the seeded collator, reused every step
    Ke, Kp = [int(m.shape[1]) for m in me], [int(m.shape[1]) for m in mp]
    clips_host = torch.randn(B, 3, frames, crop, crop, generator=torch.Generator().manual_seed(rank)).pin_memory()
    me_host, mp_host = [m.pin_memory() for m in me], [m.pin_memory() for m in mp]
    st = build_training_state(args.config, device, world, rank)

    clips = clips_host.to(device)
    me_d, mp_d = [m.to(device) for m in me_host], [m.to(device) for m in mp_host]

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ddp_check = None
    if world > 1 and not args.profile:
        ddp_check = ddp_gradient_check(st, clips, me_d, mp_d)
        if not (ddp_check["rel_l2_sync_vs_allreduce_mean"] < 1e-4 and ddp_check["rel_l2_local_vs_mean_min"] > 1e-3):
            raise SystemExit(f"DDP gradient exchange check failed: {ddp_check}")

    # `--dynamic-masks`: a NEW collator call every step (Ke / Kp change: tensor maps re-encoded, allocator sees new shapes)
    dyn = None
    if args.dynamic_masks:
        from src.masks.multiblock3d import MaskCollator
        torch.manual_seed(0)
        coll = MaskCollator(cfgs_mask=VITL16_MASKS, crop_size=crop, num_frames=frames, patch_size=16, tubelet_size=2)
        dummy = [torch.zeros(1) for _ in range(B)]

        def dyn():
            _, a, b = coll(dummy)
            return [m.to(device, non_blocking=True) for m in a], [m.to(device, non_blocking=True) for m in b]

    def step_masks():
        return dyn() if dyn is not None else (me_d, mp_d)

    # ---- device-resident timing ("value") -------------------------------------------------------------
    for _ in range(args.warmup):
        train_step(st, clips, *step_masks(), loggers=args.loggers)
    sync_all()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = lib.vj_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last = {}
    e0.record()
    t_host0 = time.perf_counter()
    for i in range(args.steps):
        loss = train_step(st, clips, *step_masks(), loggers=args.loggers, outputs=last if i == args.steps - 1 else None)
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / args.steps   # host time to ENQUEUE a step (no sync inside)
    e1.record()
    sync_all()
    ms_total = e0.elapsed_time(e1)
    launches = lib.vj_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    last_loss = float(loss)
    if args.dump_outputs and rank == 0:   # before the passes below move the weights on
        dump_outputs(args.dump_outputs, st, loss, last)
    del last
    if world > 1:
        t = torch.tensor([ms_total], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t)
    ms_step = ms_total / args.steps
    value = B * world / (ms_step * 1e-3)
    if args.profile:   # run under ncu: only the bare steps, no auxiliary passes
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_step, "gpu_launches": int(launches)}), flush=True)
        return

    # ---- per-launch GEMM timing inside further steps (roofline of the dominant kernel) -------------
    from jepa_b200 import kernels as Kn
    gemm_events = []
    orig_gemm = Kn.gemm

    def timed_gemm(a, b, out, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r = orig_gemm(a, b, out, **kw)
        e.record()
        M, Nn = out.shape
        Kk = a.shape[0] if kw.get("a_mn") else a.shape[1]
        gemm_events.append((s, e, 2.0 * M * Nn * Kk))
        return r

    attn_events = []
    orig_af, orig_ab = Kn.attn_fwd, Kn.attn_bwd

    def timed_attn(fn, mult):
        def f(*a, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a, **kw)
            e.record()
            attn_events.append((s, e, mult))
            return r
        return f

    roof_steps = 2
    Kn.gemm = timed_gemm
    Kn.attn_fwd, Kn.attn_bwd = timed_attn(orig_af, 1), timed_attn(orig_ab, 2)
    try:
        for _ in range(roof_steps):
            train_step(st, clips, me_d, mp_d)
        torch.cuda.synchronize()
    finally:
        Kn.gemm = orig_gemm
        Kn.attn_fwd, Kn.attn_bwd = orig_af, orig_ab
    gemm_ms = sum(s.elapsed_time(e) for s, e, _ in gemm_events)
    gemm_flops_exec = sum(f for _, _, f in gemm_events)
    n_gemm = len(gemm_events)
    attn_fwd_ms = sum(s.elapsed_time(e) for s, e, m in attn_events if m == 1) / roof_steps
    attn_bwd_ms = sum(s.elapsed_time(e) for s, e, m in attn_events if m == 2) / roof_steps

    # ---- end-to-end: host inputs every step, loss read back ---------------------------------------------
    copy_stream = torch.cuda.Stream(device=device)
    bufs = [dict(clips=torch.empty_like(clips), me=[torch.empty_like(m) for m in me_d], mp=[torch.empty_like(m) for m in mp_d],
                 ready=torch.cuda.Event()) for _ in range(2)]
    h2d = clips_host.numel() * 4 + sum(m.numel() * 8 for m in me_host + mp_host)

    def prefetch(i):
        b = bufs[i % 2]
        with torch.cuda.stream(copy_stream):
            b["clips"].copy_(clips_host, non_blocking=True)
            for d, s in zip(b["me"] + b["mp"], me_host + mp_host):
                d.copy_(s, non_blocking=True)
            b["ready"].record(copy_stream)

    def e2e_loop(n):
        prefetch(0)
        out = 0.0
        for i in range(n):
            b = bufs[i % 2]
            torch.cuda.current_stream().wait_event(b["ready"])
            l = train_step(st, b["clips"], b["me"], b["mp"], loggers=args.loggers)
            if i + 1 < n:
                prefetch(i + 1)
            out = float(l)          # device -> host read of the step's result (4 bytes), syncs the step
        return out

    e2e_loop(2)
    sync_all()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    sync_all()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t)
    e2e_value = B * world * args.steps / e2e_s

    if rank == 0:
        peaks = measured_peaks()
        f_clip = flops_per_clip(D, L, N, Ke, Kp)
        fg_clip = gemm_flops_per_clip(D, L, N, Ke, Kp)
        fa_clip = f_clip - fg_clip
        gemm_ms_step = gemm_ms / roof_steps
        achieved = fg_clip * B / (gemm_ms_step * 1e-3) / 1e12
        peak = peaks["bf16_sustained"]
        step_tf = f_clip * B / (ms_step * 1e-3) / 1e12
        line = {
            "metric": "clips/sec ViT-L/16 16x224^2 synthetic V-JEPA pre-training step" if args.config == "vitl16"
                      else f"clips/sec {args.config} synthetic V-JEPA pre-training step",
            "value": round(value, 2), "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.config}: {model_name} 2x16x16 tubelets, {frames}x{crop}x{crop}, batch {B}/GPU, "
                                   f"multiblock3d masks Ke={Ke} Kp={Kp} (seed 0, first collator call), predictor 12x384, "
                                   "AdamW+GradScaler+EMA in step, logging helpers off",
                       "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2_policy": "inputs+weights+activations per step (>3 GB) exceed the 126 MB L2; no explicit flush",
                       "flops_per_clip": f_clip, "loss_last": last_loss},
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 2), "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "host_enqueue_ms_per_step": round(host_enqueue_ms, 2),
            "roofline": {
                "bound": "tensor", "scope": "whole train step (BASELINE metric: % tensor-pipe roofline of the step)",
                "achieved": round(step_tf, 1), "peak": peak, "unit": "TFLOP/s", "frac": round(step_tf / peak, 4),
                "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step)",
                "frac_of_burst": round(step_tf / peaks["bf16_burst"], 4), "frac_of_nominal_2250": round(step_tf / 2250.0, 4),
                "algorithmic_tflop_per_step": round(f_clip * B / 1e12, 3),
                "dominant_kernel": {
                    "kernel": "vj::gemm_kernel (all Linear / patch-embed GEMMs of a step)", "achieved": round(achieved, 1),
                    "frac": round(achieved / peak, 4), "launches_per_step": n_gemm // roof_steps,
                    "gemm_ms_per_step": round(gemm_ms_step, 3), "algorithmic_tflop_per_step": round(fg_clip * B / 1e12, 3),
                    "executed_tflop_per_step": round(gemm_flops_exec / roof_steps / 1e12, 3),
                    "timing": "CUDA events around every launch on the launching stream, 2 extra steps"},
                "attention": {
                    "kernel": "vj::attn_fwd/bwd kernels", "fwd_ms_per_step": round(attn_fwd_ms, 3),
                    "bwd_ms_per_step": round(attn_bwd_ms, 3), "algorithmic_tflop_per_step": round(fa_clip * B / 1e12, 3),
                    "achieved": round(fa_clip * B / ((attn_fwd_ms + attn_bwd_ms) * 1e-3) / 1e12, 1),
                    "frac": round(fa_clip * B / ((attn_fwd_ms + attn_bwd_ms) * 1e-3) / 1e12 / peak, 4)},
                "traffic": ncu_gemm_traffic(args.config),
                "traffic_unit": "DRAM bytes per step over the GEMM family's launches (dram__bytes_read.sum + "
                                "dram__bytes_write.sum, ncu launch list in profiles/)"},
        }
        if ddp_check is not None:
            line["ddp_check"] = ddp_check
        if args.dynamic_masks or args.loggers:
            line["config"]["variant"] = {"dynamic_masks": bool(args.dynamic_masks), "loggers": bool(args.loggers)}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.config, budget_s=25.0)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the same step on the host cores
# ------------------------------------------------------------------------------------------------------
def oracle_step_fn(cfg_name, B):
    """Returns a closure running ONE fp32 train step (target fwd, context+predictor fwd/bwd, loss, EMA) of the
    oracle on B clips.  AdamW is omitted on the CPU side (a few % of the CPU step), which favours the baseline."""
    from oracle import vjepa_oracle as O
    O.FUSED = True   # torch's fused CPU operators, i.e. the library calls the reference itself makes on CPU
    from jepa_b200.models import VisionTransformer, vit_predictor
    from functools import partial
    import torch.nn as nn
    model_name, D, L, heads, crop, frames, _ = CONFIGS[cfg_name]
    enc = VisionTransformer(img_size=crop, patch_size=16, num_frames=frames, tubelet_size=2, embed_dim=D, depth=L,
                            num_heads=heads, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                            uniform_power=True)
    pred = vit_predictor(img_size=crop, use_mask_tokens=True, patch_size=16, num_frames=frames, tubelet_size=2,
                         embed_dim=D, predictor_embed_dim=PRED_DIM, depth=PRED_DEPTH, num_heads=heads, uniform_power=True,
                         num_mask_tokens=2, zero_init_mask_tokens=True)
    S_enc = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    S_tgt = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    S_pred = {k: v.detach().clone() for k, v in pred.state_dict().items()}
    for S, frozen in ((S_enc, "pos_embed"), (S_pred, "predictor_pos_embed")):
        for k, v in S.items():
            if k != frozen:
                v.requires_grad_(True)
    # the GPU arm's masks (collator call at ITS batch size, seed 0), first B rows: identical kept-token counts per clip,
    # i.e. the same work per clip on both arms (a batch-1 collator call would keep more context tokens)
    me, mp = seeded_masks(crop, frames, CONFIGS[cfg_name][6], seed=0)
    me, mp = [m[:B].clone() for m in me], [m[:B].clone() for m in mp]
    clips = torch.randn(B, 3, frames, crop, crop, generator=torch.Generator().manual_seed(0))

    def step():
        for S in (S_enc, S_pred):
            for v in S.values():
                v.grad = None
        h = O.forward_target(S_tgt, clips, mp, L, heads)
        z = O.forward_context(S_enc, S_pred, clips, me, mp, L, heads, PRED_DEPTH, heads)
        loss = O.loss_fn(z, h)
        loss.backward()
        O.ema(S_tgt, S_enc, 0.998)
        return float(loss)

    return step


def usable_cores():
    """Host threads this process can really use: min(os.cpu_count, sched affinity, cgroup cpu quota), capped at
    VJ_CPU_THREADS if set (oversubscribing a quota-limited container is several times slower than matching it)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    if os.environ.get("VJ_CPU_THREADS"):
        n = min(n, int(os.environ["VJ_CPU_THREADS"]))
    return max(1, min(n, 64))   # torch intra-op scaling of this workload saturates well before 64 threads


def reference_cpu_run(cfg_name, B, steps, warmup, cores, timeout=1500):
    """The UNMODIFIED reference (baseline/_ref, tools/install_reference.sh) through its own app.vjepa.train.main on the
    host cores: fp32 (CPU autocast / GradScaler disable themselves), AdamW + EMA + its loggers in the step, synthetic clips,
    its own collator - SURVEY 8d's CPU baseline.  Runs in a subprocess (tools/ref_gpu.py --backend gloo) because the
    repo's drop-in src/ and app/ packages carry the reference's module names.  None if baseline/_ref is absent."""
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "app")):
        return None
    cmd = [sys.executable, os.path.join(ROOT, "tools", "ref_gpu.py"), "bench", "--config", cfg_name, "--backend", "gloo",
           "--batch", str(B), "--steps", str(steps), "--warmup", str(warmup), "--loggers", "on", "--threads", str(cores)]
    env = {k: v for k, v in os.environ.items() if k not in ("PYTHONPATH", "RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_PORT")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    env["MASTER_PORT"] = "29611"
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=tempfile.gettempdir(), env=env)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        out = json.loads(lines[-1]) if lines else None
    except Exception:
        return None
    if not out or "unavailable" in out or out.get("gpu_ms_per_step_median", -1) <= 0:
        return None
    return out


def cpu_baseline(cfg_name, budget_s=25.0):
    cores = usable_cores()
    ref = reference_cpu_run(cfg_name, B=2, steps=2, warmup=1, cores=cores)   # ~3 steps of 5-10 s at ViT-L
    if ref is not None:
        return {"value": ref["clips_per_s"], "unit": "clips/s", "cores": cores, "kind": "reference", "adamw": True,
                "sample": f"unmodified reference app.vjepa.train.main (baseline/_ref) on the host: 2 timed fp32 steps (+1 warm-up) "
                          f"at batch 2 of {cfg_name}, median {ref['gpu_ms_per_step_median'] / 1e3:.2f} s/step by its own "
                          f"wall-time column, AdamW/EMA/loggers in the step, {cores} torch threads"}
    torch.set_num_threads(cores)
    B = 1
    step = oracle_step_fn(cfg_name, B)
    t0 = time.perf_counter()
    step()                      # first step also pays allocator warm-up; keep it only if nothing else fits
    t_first = time.perf_counter() - t0
    times = []
    while sum(times) + t_first < budget_s and len(times) < 3:
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    t = min(times) if times else t_first
    return {"value": round(B / t, 4), "unit": "clips/s", "cores": cores, "kind": "port", "adamw": False,
            "sample": f"{1 + len(times)} fp32 train step(s) of the CPU oracle (oracle/vjepa_oracle.py; AdamW omitted) at batch {B} "
                      f"of {cfg_name}, best step {t:.2f}s, torch intra-op threads = {cores}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = usable_cores()
    model_name, D, L, heads, crop, frames, Bcfg = CONFIGS[args.config]
    N = (frames // 2) * (crop // 16) ** 2
    me, mp = seeded_masks(crop, frames, Bcfg, seed=0)
    Ke, Kp = [int(m.shape[1]) for m in me], [int(m.shape[1]) for m in mp]
    B = 2
    ref = reference_cpu_run(args.config, B=B, steps=args.steps, warmup=args.warmup, cores=cores)
    if ref is not None:
        kind, adamw = "reference", True
        value = ref["clips_per_s"]
        ms_step = ref["gpu_ms_per_step_median"]
        loss = ref["losses"][-1]
        sample = (f"each step = one fp32 train step of the UNMODIFIED reference (baseline/_ref, app.vjepa.train.main: target fwd, "
                  f"context+predictor fwd/bwd, AdamW, EMA, its loggers) on {B} clips of {args.config} ({model_name}, "
                  f"{frames}x{crop}x{crop}, its own MaskCollator at batch {B}); median of {args.steps} by its wall-time column; "
                  f"{cores} host threads")
    else:
        kind, adamw = "port", False
        torch.set_num_threads(cores)
        B = 1
        step = oracle_step_fn(args.config, B)
        for _ in range(args.warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            loss = step()
        dt = time.perf_counter() - t0
        value = B * args.steps / dt
        ms_step = dt / args.steps * 1e3
        sample = (f"baseline/_ref absent -> CPU oracle port: each step = one fp32 train step (AdamW omitted) on {B} clip of "
                  f"{args.config} ({model_name}, {frames}x{crop}x{crop}, masks Ke={Ke} Kp={Kp}); {cores} host threads")
    line = {
        "impl": "reference",
        "metric": "clips/sec ViT-L/16 16x224^2 synthetic V-JEPA pre-training step" if args.config == "vitl16"
                  else f"clips/sec {args.config} synthetic V-JEPA pre-training step",
        "value": round(value, 4), "unit": "clips/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.config}: {model_name} 2x16x16 tubelets, {frames}x{crop}x{crop}, CPU sample batch {B} "
                               f"(GPU arm: batch {Bcfg}/GPU)", "global_batch": B, "parallelism": "cpu", "loss_last": loss},
        "cpu_baseline": {"value": round(value, 4), "unit": "clips/s", "cores": cores, "kind": kind, "adamw": adamw,
                         "sample": sample},
        "e2e": {"value": round(value, 4), "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="vitl16", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch (debug only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dynamic-masks", action="store_true", help="new collator call every step (SURVEY 8d second run)")
    ap.add_argument("--loggers", action="store_true", help="as-shipped step: grad_logger x2 + adamw_logger inside the step")
    ap.add_argument("--profile", action="store_true", help="bare steps only (for ncu); never a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, seeded samples of large arrays)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        args.steps = args.steps if args.steps is not None else 3
        args.warmup = args.warmup if args.warmup is not None else 1
        run_reference(args)
    else:
        args.steps = args.steps if args.steps is not None else 20
        args.warmup = args.warmup if args.warmup is not None else 5
        if not args.profile:
            args.warmup = max(3, args.warmup)
        run_ours(args)


if __name__ == "__main__":
    main()
