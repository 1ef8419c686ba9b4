"""The drop-in ENTRY POINT on a GPU (-m gpu): `app.scaffold.main('vjepa', cfg)` -> `app.vjepa.train.main` exactly as
`python -m app.main` would call it (reference app/main.py:28-60, app/scaffold.py:16-21), on the synthetic dataset:
CSV columns (train.py:199-209), reference-format checkpoint (train.py:307-324), resume through load_checkpoint
(app/vjepa/utils.py:28-83) with the flat AdamW state re-aliased, and the saved encoder / predictor matching the
state dicts of the UNMODIFIED reference modules key for key and shape for shape (what strict=True loading checks)."""
import csv
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MASKS = [
    dict(aspect_ratio=[0.75, 1.5], num_blocks=8, spatial_scale=[0.15, 0.15], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
    dict(aspect_ratio=[0.75, 1.5], num_blocks=2, spatial_scale=[0.7, 0.7], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
]


def _cfg(folder, epochs, load):
    return {
        "app": "vjepa",
        "meta": dict(load_checkpoint=load, read_checkpoint=None, seed=234, eval_freq=100, use_sdpa=True, dtype="bfloat16"),
        "mask": MASKS,
        "model": dict(model_name="vit_tiny", pred_depth=2, pred_embed_dim=384, uniform_power=True, use_mask_tokens=True,
                      zero_init_mask_tokens=True),
        "data": dict(dataset_type="synthetic", datasets=[], batch_size=2, num_clips=1, num_frames=8, tubelet_size=2,
                     sampling_rate=4, crop_size=224, patch_size=16, pin_mem=True, num_workers=0),
        "data_aug": dict(auto_augment=False, motion_shift=False, random_resize_aspect_ratio=[0.75, 1.35],
                         random_resize_scale=[0.3, 1.0], reprob=0.0),
        "loss": dict(loss_exp=1.0, reg_coeff=0.0),
        "optimization": dict(ipe=3, ipe_scale=1.25, clip_grad=10.0, weight_decay=0.04, final_weight_decay=0.4, epochs=epochs,
                             warmup=1, start_lr=0.0002, lr=0.000625, final_lr=1e-6, ema=[0.998, 1.0]),
        "logging": dict(folder=str(folder), write_tag="jepa"),
    }


def _rows(folder):
    with open(os.path.join(folder, "jepa_r0.csv")) as f:
        return list(csv.reader(f))


def test_app_main_train_save_resume(tmp_path):
    assert torch.cuda.is_available()
    from app.scaffold import main as app_main
    from jepa_b200 import _lib
    lib = _lib.load()
    n0 = lib.vj_launch_count()
    app_main("vjepa", _cfg(tmp_path, epochs=1, load=False))
    assert lib.vj_launch_count() - n0 > 300          # the steps ran on our kernels
    rows = _rows(tmp_path)
    assert rows[0] == ["epoch", "itr", "loss", "loss-jepa", "reg-loss", "enc-grad-norm", "pred-grad-norm", "gpu-time(ms)",
                       "wall-time(ms)"]
    assert [r[:2] for r in rows[1:]] == [["1", "0"], ["1", "1"], ["1", "2"]]
    losses = [float(r[2]) for r in rows[1:]]
    assert all(0.1 < l < 3.0 for l in losses), losses
    ckpt_path = os.path.join(tmp_path, "jepa-latest.pth.tar")
    ck = torch.load(ckpt_path, map_location="cpu")
    assert set(ck) == {"encoder", "predictor", "opt", "scaler", "target_encoder", "epoch", "loss", "batch_size", "world_size", "lr"}
    assert ck["epoch"] == 1 and "module.backbone.blocks.0.attn.qkv.weight" in ck["encoder"]
    assert len(ck["opt"]["param_groups"]) == 4
    st0 = next(iter(ck["opt"]["state"].values()))
    assert float(st0["step"]) == 3.0 and "exp_avg" in st0 and "exp_avg_sq" in st0
    assert ck["scaler"]["scale"] == 65536.0

    # ---- resume: second epoch continues from the checkpoint (schedulers / collator advanced, optimizer state restored)
    app_main("vjepa", _cfg(tmp_path, epochs=2, load=True))
    rows = _rows(tmp_path)
    body = [r for r in rows if r and r[0] != "epoch"]
    assert [r[:2] for r in body] == [["1", "0"], ["1", "1"], ["1", "2"], ["2", "0"], ["2", "1"], ["2", "2"]]
    ck2 = torch.load(ckpt_path, map_location="cpu")
    assert ck2["epoch"] == 2
    assert float(next(iter(ck2["opt"]["state"].values()))["step"]) == 6.0
    # EMA'd target moved, encoder trained on
    k = "module.backbone.blocks.1.mlp.fc1.weight"
    assert not torch.equal(ck["encoder"][k], ck2["encoder"][k]) and not torch.equal(ck["target_encoder"][k], ck2["target_encoder"][k])

    # ---- the checkpoint is the reference's format: its own modules take it with strict=True, i.e. after the DDP
    # 'module.' prefix every network has exactly the keys and shapes of the reference's state dict (stored from the
    # unmodified modules by tests/golden/make_golden_reference.py)
    ref = torch.load(os.path.join(ROOT, "tests", "golden", "golden_reference.pt"))["checkpoint_shapes"]
    for key, tag in (("encoder", "encoder"), ("predictor", "predictor"), ("target_encoder", "encoder")):
        assert all(k.startswith("module.") for k in ck[key]), key
        assert {k[len("module."):]: list(v.shape) for k, v in ck[key].items()} == ref[tag], key


def test_app_main_with_gpu_input_pipeline(tmp_path):
    """f3 end to end: dataset_type synthetic_uint8 feeds decoded-video-like uint8 frames through the reference-shaped
    transform (decisions on the host, RNG order of the reference) and the crop / flip / normalise kernel into the step."""
    assert torch.cuda.is_available()
    from app.scaffold import main as app_main
    cfg = _cfg(tmp_path, epochs=1, load=False)
    cfg["data"]["dataset_type"] = "synthetic_uint8"
    cfg["optimization"]["ipe"] = 2
    app_main("vjepa", cfg)
    body = [r for r in _rows(tmp_path) if r and r[0] != "epoch"]
    assert [r[:2] for r in body] == [["1", "0"], ["1", "1"]]
    assert all(0.1 < float(r[2]) < 3.0 for r in body), body
