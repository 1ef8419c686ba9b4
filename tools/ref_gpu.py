#!/usr/bin/env python
"""Run the UNMODIFIED reference (facebookresearch/jepa, installed into baseline/_ref by
tools/install_reference.sh) on cuda:0.  Measurement / test infrastructure only - the product never imports this.

  bench : the reference's own training entry app.vjepa.train.main(args) at a BASELINE config (bf16 autocast, eager
          PyTorch: cuBLASLt GEMMs, SDPA, cuDNN Conv3d, c10d DDP over a 1-rank NCCL group), synthetic clips, its own
          MaskCollator (seed 0, first call reused like bench.py), timed by its own gpu_timer -> the CSV column
          `gpu-time(ms)` (src/utils/logging.py:14-31, app/vjepa/train.py:499).  This is the GPU bar SURVEY 8d asks
          for: "the same reference code on the same B200".  --loggers off stubs grad_logger / adamw_logger
          (the ~1000 host syncs per step, SURVEY 8d (A)); --loggers on is the as-shipped step (B).

The repo root holds drop-in `src/` and `app/` packages with the reference's names, so this script must run in its own
process with the repo root OFF sys.path.
"""
import argparse
import json
import os
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.path.join(ROOT, "baseline", "_ref")
sys.path = [p for p in sys.path if os.path.abspath(p or os.getcwd()) != ROOT]
if not os.path.isdir(os.path.join(REF, "app")):
    print(json.dumps({"impl": "reference-gpu", "unavailable": "baseline/_ref missing: run tools/install_reference.sh"}))
    sys.exit(0)
sys.path.insert(0, REF)

import torch  # noqa: E402

VITL16_MASKS = [
    dict(aspect_ratio=[0.75, 1.5], num_blocks=8, spatial_scale=[0.15, 0.15], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
    dict(aspect_ratio=[0.75, 1.5], num_blocks=2, spatial_scale=[0.7, 0.7], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
]
CONFIGS = {   # name: (model_name, crop, frames, batch/GPU)  - BASELINE.json configs[1..4]
    "vitl16": ("vit_large", 224, 16, 32),
    "vith16": ("vit_huge", 224, 16, 24),
    "vith16_384": ("vit_huge", 384, 16, 10),
    "tiny": ("vit_tiny", 224, 8, 2),
}


def run_bench(a):
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29577")
    if a.backend == "nccl":
        torch.cuda.set_device(0)
    dist.init_process_group(a.backend, rank=0, world_size=1)   # init_distributed() then early-returns (distributed.py:20-21)
    if a.threads:
        torch.set_num_threads(a.threads)
    import app.vjepa.train as T
    model_name, crop, frames, B = CONFIGS[a.config]
    if a.batch:
        B = a.batch
    iters = a.warmup + a.steps
    clips = torch.randn(B, 3, frames, crop, crop, generator=torch.Generator().manual_seed(0))

    class Sampler:
        def set_epoch(self, e):
            pass

    class Loader:
        """What the reference's DataLoader yields: collator(list of (buffer=[clip], label, clip_indices))."""

        def __init__(self, collator):
            torch.manual_seed(0)
            self.fixed = collator([([clips[i]], 0, [0]) for i in range(B)])   # first collator call, reused (bench.py does the same)
            self.collator = collator

        def __len__(self):
            return iters

        def __iter__(self):
            for _ in range(iters):
                if a.dynamic_masks:
                    yield self.collator([([clips[i]], 0, [0]) for i in range(B)])
                else:
                    yield self.fixed

    def init_data(**kw):
        return Loader(kw["collator"]), Sampler()

    T.init_data = init_data
    T.make_transforms = lambda **kw: None
    if a.loggers == "off":
        class _Stats:
            first_layer = last_layer = 0.
            min = max = avg = 0.
            global_norm = 0.

        T.grad_logger = lambda named_params: _Stats()
        T.adamw_logger = lambda optimizer: None
    folder = tempfile.mkdtemp(prefix="ref_gpu_")
    args = {
        "meta": dict(load_checkpoint=False, read_checkpoint=None, seed=234, eval_freq=100, use_sdpa=True, dtype="bfloat16"),
        "mask": VITL16_MASKS,
        "model": dict(model_name=model_name, pred_depth=12, pred_embed_dim=384, uniform_power=True, use_mask_tokens=True,
                      zero_init_mask_tokens=True),
        "data": dict(dataset_type="VideoDataset", datasets=[], batch_size=B, num_clips=1, num_frames=frames, tubelet_size=2,
                     sampling_rate=4, crop_size=crop, patch_size=16, pin_mem=True, num_workers=0),
        "data_aug": dict(auto_augment=False, motion_shift=False, random_resize_aspect_ratio=[0.75, 1.35],
                         random_resize_scale=[0.3, 1.0], reprob=0.0),
        "loss": dict(loss_exp=1.0, reg_coeff=0.0),
        "optimization": dict(ipe=iters, ipe_scale=1.25, clip_grad=10.0, weight_decay=0.04, final_weight_decay=0.4,
                             epochs=1, warmup=40, start_lr=0.0002, lr=0.000625, final_lr=1e-6, ema=[0.998, 1.0]),
        "logging": dict(folder=folder, write_tag="jepa"),
    }
    real_save = torch.save
    torch.save = lambda *x, **k: None     # the 5 GB end-of-epoch checkpoint is not part of the step
    t0 = time.time()
    try:
        T.main(args)
    finally:
        torch.save = real_save
    wall = time.time() - t0
    gpu_ms, losses = [], []
    on_gpu = a.backend == "nccl"
    with open(os.path.join(folder, "jepa_r0.csv")) as f:
        header = f.readline().strip().split(",")
        # on the CPU the reference's gpu_timer returns -1 (logging.py:16): use its wall-time column (train.py:500)
        gi, li = header.index("gpu-time(ms)" if on_gpu else "wall-time(ms)"), header.index("loss")
        for line in f:
            c = line.strip().split(",")
            gpu_ms.append(float(c[gi]))
            losses.append(float(c[li]))
    timed = sorted(gpu_ms[a.warmup:])
    med = timed[len(timed) // 2]
    mean = sum(timed) / len(timed)
    out = {
        "impl": "reference-gpu" if on_gpu else "reference-cpu",
        "what": "unmodified facebookresearch/jepa app.vjepa.train.main, " + ("cuda:0, bf16 autocast, eager PyTorch" if on_gpu else
                f"CPU fp32 (torch.cuda.amp autocast / GradScaler disable themselves), {torch.get_num_threads()} threads"),
        "threads": torch.get_num_threads(),
        "config": a.config, "model": model_name, "batch": B, "frames": frames, "crop": crop, "loggers": a.loggers,
        "dynamic_masks": bool(a.dynamic_masks), "steps": a.steps, "warmup": a.warmup,
        "gpu_ms_per_step_median": med, "gpu_ms_per_step_mean": round(mean, 2), "gpu_ms_all": gpu_ms,
        "clips_per_s": round(B / (med * 1e-3), 4),
        "timer": "reference gpu_timer (CUDA events around train_step)" if on_gpu else "reference wall-time(ms) column",
        "losses": losses, "wall_s": round(wall, 1), "torch": torch.__version__,
        "max_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2) if torch.cuda.is_available() else None,
    }
    print(json.dumps(out), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="mode", required=True)
    b = sub.add_parser("bench")
    b.add_argument("--config", default="vitl16", choices=sorted(CONFIGS))
    b.add_argument("--steps", type=int, default=10)
    b.add_argument("--warmup", type=int, default=4)
    b.add_argument("--batch", type=int, default=0)
    b.add_argument("--loggers", default="off", choices=["off", "on"])
    b.add_argument("--dynamic-masks", action="store_true")
    b.add_argument("--out", default="")
    b.add_argument("--backend", default="nccl", help="nccl: cuda:0;  gloo: the reference's CPU path (fp32) on the host cores")
    b.add_argument("--threads", type=int, default=0)
    a = ap.parse_args()
    if not torch.cuda.is_available() and a.backend != "gloo":
        print(json.dumps({"impl": "reference-gpu", "unavailable": "no CUDA device"}))
        return
    run_bench(a)


if __name__ == "__main__":
    main()
