"""Golden fixture of the UNMODIFIED reference (facebookresearch/jepa) run on a CUDA device, for
tests/test_gpu_reference.py and tests/test_gpu_train_entry.py:

    python tests/golden/make_golden_reference.py REFERENCE_DIR [--out tests/golden/golden_reference.pt]

REFERENCE_DIR is a checkout of the reference; its src/ package is imported.  For each step config (C1 and the 2-block
ViT-L/16 slice of tests/parity_util.py) one forward / backward of the reference modules on the seeded weights / clips /
masks the tests use, once under bf16 autocast (app/vjepa/train.py:453) and once in fp32 with TF32 off.  Stored: both
losses and, for every activation and parameter gradient, its shape and its bf16 / fp32 values at the positions
common.sample_index picks (the full tensors are ~150 MB).  Also stored: the reference's state-dict shapes of the tiny
encoder / predictor that test_gpu_train_entry.py saves, i.e. what its modules accept with strict=True.
"""
import argparse
import copy
import os
import sys
from functools import partial

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
# the repo root holds drop-in src/ and app/ packages with the reference's module names: keep it off sys.path
sys.path = [p for p in sys.path if os.path.abspath(p or os.getcwd()) != ROOT]

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402

ACT_SAMPLES = 1024     # per activation tensor (h / z_enc / z of each mask)
GRAD_SAMPLES = 48      # per parameter gradient


def reference_step(cfg, dev):
    """One reference step in bf16 autocast and in fp32: {tag: dict(loss_jepa, loss_reg, act, enc_grad, pred_grad)}."""
    from common import VITL16_MASKS, synth_clips, synth_state
    import src.models.vision_transformer as ref_vit
    import src.models.predictor as ref_pred
    from src.masks.multiblock3d import MaskCollator
    from src.masks.utils import apply_masks
    from src.models.utils.multimask import MultiMaskWrapper, PredictorMultiMaskWrapper
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    crop, frames, B = cfg["crop_size"], cfg["num_frames"], cfg["batch"]
    enc = ref_vit.VisionTransformer(img_size=crop, patch_size=16, num_frames=frames, tubelet_size=2, embed_dim=cfg["embed_dim"],
                                    depth=cfg["depth"], num_heads=cfg["heads"], mlp_ratio=4, qkv_bias=True,
                                    norm_layer=partial(nn.LayerNorm, eps=1e-6), uniform_power=True, use_sdpa=True)
    pred = ref_pred.vit_predictor(img_size=crop, use_mask_tokens=True, patch_size=16, num_frames=frames, tubelet_size=2,
                                  embed_dim=cfg["embed_dim"], predictor_embed_dim=cfg["pred_embed_dim"], depth=cfg["pred_depth"],
                                  num_heads=cfg["heads"], uniform_power=True, num_mask_tokens=2, zero_init_mask_tokens=True,
                                  use_sdpa=True)
    enc_shapes = {k: tuple(v.shape) for k, v in enc.state_dict().items()}
    pred_shapes = {k: tuple(v.shape) for k, v in pred.state_dict().items()}
    enc.load_state_dict(synth_state(enc_shapes, seed=11, keep=("pos_embed",)), strict=False)
    pred.load_state_dict(synth_state(pred_shapes, seed=12, keep=("pos_embed",)), strict=False)
    tgt = copy.deepcopy(enc)
    tgt.load_state_dict(synth_state(enc_shapes, seed=13, keep=("pos_embed",)), strict=False)
    enc, pred, tgt = MultiMaskWrapper(enc).to(dev), PredictorMultiMaskWrapper(pred).to(dev), MultiMaskWrapper(tgt).to(dev)
    for p in tgt.parameters():
        p.requires_grad = False
    clips = synth_clips(B, frames, crop, crop, seed=0).to(dev)
    torch.manual_seed(0)
    coll = MaskCollator(cfgs_mask=VITL16_MASKS, crop_size=crop, num_frames=frames, patch_size=16, tubelet_size=2)
    _, me, mp = coll([torch.zeros(1) for _ in range(cfg.get("mask_batch", B))])
    me, mp = [m[:B].to(dev) for m in me], [m[:B].to(dev) for m in mp]
    result = {}
    for tag, dtype, mixed in (("bf16", torch.bfloat16, True), ("fp32", torch.float32, False)):
        for net in (enc, pred):
            for p in net.parameters():
                p.grad = None
        with torch.autocast(dev.type, dtype=dtype, enabled=mixed):     # train.py:453
            with torch.no_grad():
                h = tgt(clips)
                h = F.layer_norm(h, (h.size(-1),))
                h = apply_masks(h, mp, concat=False)
            z_enc = enc(clips, me)
            z = pred(z_enc, h, me, mp)
            loss = sum(torch.mean(torch.abs(zi - hi)) for zi, hi in zip(z, h)) / len(mp)
            pstd = sum(torch.sqrt(zi.var(dim=1) + 0.0001) for zi in z) / len(z)
            loss_reg = torch.mean(F.relu(1. - pstd))
        (loss * (65536.0 if mixed else 1.0)).backward()              # GradScaler's initial scale, unscaled below
        inv = 1.0 / 65536.0 if mixed else 1.0
        act = {f"{key}[{i}]": t.detach().float().cpu() for key, ts in (("h", h), ("z_enc", z_enc), ("z", z))
               for i, t in enumerate(ts)}
        result[tag] = dict(
            loss_jepa=float(loss), loss_reg=float(loss_reg), act=act,
            enc_grad={n: (p.grad.detach().float() * inv).cpu() for n, p in enc.backbone.named_parameters() if p.grad is not None},
            pred_grad={n: (p.grad.detach().float() * inv).cpu() for n, p in pred.backbone.named_parameters() if p.grad is not None})
    return result


def sampled(bf16, fp32, n):
    """name -> tensor dicts of both runs -> their values at sample_index positions, concatenated in name order."""
    from common import sample_index
    assert set(bf16) == set(fp32)
    names, shapes, b, f = sorted(fp32), [], [], []
    for name in names:
        assert bf16[name].shape == fp32[name].shape, name
        idx = sample_index(fp32[name].numel(), n)
        shapes.append(list(fp32[name].shape))
        b.append(bf16[name].reshape(-1)[idx])
        f.append(fp32[name].reshape(-1)[idx])
    return dict(names=names, shapes=shapes, n=n, bf16=torch.cat(b).contiguous(), fp32=torch.cat(f).contiguous())


def checkpoint_shapes():
    """State-dict shapes of the reference modules test_gpu_train_entry.py's checkpoint must load into with strict=True."""
    import src.models.vision_transformer as vit
    import src.models.predictor as vp
    from src.models.utils.multimask import MultiMaskWrapper, PredictorMultiMaskWrapper
    enc = MultiMaskWrapper(vit.vit_tiny(img_size=224, patch_size=16, num_frames=8, tubelet_size=2, uniform_power=True,
                                        use_sdpa=True))
    pred = PredictorMultiMaskWrapper(vp.vit_predictor(img_size=224, use_mask_tokens=True, patch_size=16, num_frames=8,
                                                      tubelet_size=2, embed_dim=192, predictor_embed_dim=384, depth=2,
                                                      num_heads=3, uniform_power=True, num_mask_tokens=2,
                                                      zero_init_mask_tokens=True, use_sdpa=True))
    return {tag: {k: list(v.shape) for k, v in net.state_dict().items()} for tag, net in (("encoder", enc), ("predictor", pred))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("reference", help="checkout of facebookresearch/jepa")
    ap.add_argument("--out", default=os.path.join(HERE, "golden_reference.pt"))
    ap.add_argument("--device", default="cuda:0", help="cpu only for dry runs of this script")
    a = ap.parse_args()
    sys.path[:0] = [os.path.abspath(a.reference), HERE, os.path.dirname(HERE)]
    from parity_util import C1, VITL_2B
    dev = torch.device(a.device)
    steps = {}
    for name, cfg in (("c1_vit_tiny_12+12", C1), ("vitl16_2+2_blocks", VITL_2B)):
        r = reference_step(cfg, dev)
        rb, rf = r["bf16"], r["fp32"]
        steps[name] = dict(loss_jepa=dict(bf16=rb["loss_jepa"], fp32=rf["loss_jepa"]),
                           loss_reg=dict(bf16=rb["loss_reg"], fp32=rf["loss_reg"]),
                           act=sampled(rb["act"], rf["act"], ACT_SAMPLES),
                           enc_grad=sampled(rb["enc_grad"], rf["enc_grad"], GRAD_SAMPLES),
                           pred_grad=sampled(rb["pred_grad"], rf["pred_grad"], GRAD_SAMPLES))
        print(name, "loss bf16 / fp32:", rb["loss_jepa"], rf["loss_jepa"], flush=True)
    device = torch.cuda.get_device_name(dev) if dev.type == "cuda" else "cpu"
    torch.save(dict(steps=steps, checkpoint_shapes=checkpoint_shapes(), device=device, torch=str(torch.__version__)), a.out)
    print("wrote", a.out, os.path.getsize(a.out), "bytes")


if __name__ == "__main__":
    main()
