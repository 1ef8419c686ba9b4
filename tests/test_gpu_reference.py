"""GPU parity against the REFERENCE ITSELF (-m gpu): our CUDA path runs one step on the seeded weights / clips / masks of
tests/parity_util.py and is compared with what the unmodified facebookresearch/jepa modules computed for the same step on
a B200 - once under bf16 autocast (what app/vjepa/train.py:453 does) and once in fp32.  Those reference results live in
tests/golden/golden_reference.pt (written by tests/golden/make_golden_reference.py): both losses, and every activation
and parameter gradient at fixed sample positions (common.sample_index), where the errors below are measured.

SURVEY 8c tolerances:
  (i)   ours-bf16 vs reference-bf16-autocast: rel-L2 <= 2e-2 on target / context / predictor outputs, loss |d| <= 2e-3;
        gradients rel-L2 <= 3e-2 (two bf16 computations with different rounding points)
  (iii) both against the reference in fp32 on the GPU: our error must be <= 2x the reference's own bf16 error (+ 2e-3)
"""
import math
import os

import pytest
import torch

from common import C1, sample_index
from parity_util import VITL_2B, rel_l2, run_c1_step_cuda

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_reference.pt")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def gold():
    return torch.load(GOLDEN)


def _unpack(entry):
    """name -> (shape, sample positions, reference-bf16 values, reference-fp32 values) of one fixture group."""
    out, off = {}, 0
    for name, shape in zip(entry["names"], entry["shapes"]):
        idx = sample_index(math.prod(shape), entry["n"])
        k = len(idx)
        out[name] = (tuple(shape), idx, entry["bf16"][off:off + k], entry["fp32"][off:off + k])
        off += k
    assert off == entry["fp32"].numel()
    return out


def _errors(got, ref):
    """(ours vs ref-bf16, ours vs ref-fp32, ref-bf16 vs ref-fp32) rel-L2 per tensor over the stored positions."""
    assert set(got) == set(ref), set(got) ^ set(ref)
    errs = {}
    for n, (shape, idx, rb, rf) in ref.items():
        assert tuple(got[n].shape) == shape, (n, tuple(got[n].shape), shape)
        a = got[n].reshape(-1)[idx]
        errs[n] = (rel_l2(a, rb), rel_l2(a, rf), rel_l2(rb, rf))
    return errs


@pytest.mark.parametrize("name,cfg", [("c1_vit_tiny_12+12", C1), ("vitl16_2+2_blocks", VITL_2B)],
                         ids=["c1_vit_tiny_12+12", "vitl16_2+2_blocks"])
def test_step_vs_reference_on_same_gpu(dev, gold, name, cfg):
    ref = gold["steps"][name]
    got = run_c1_step_cuda(dev, cfg=cfg)
    assert abs(got["loss_jepa"] - ref["loss_jepa"]["bf16"]) <= 2e-3, (got["loss_jepa"], ref["loss_jepa"])
    assert abs(got["loss_jepa"] - ref["loss_jepa"]["fp32"]) <= 2e-3, (got["loss_jepa"], ref["loss_jepa"])
    report = {}
    acts = {f"{key}[{i}]": t for key in ("h", "z_enc", "z") for i, t in enumerate(got[key])}
    for n, (e_ours_b, e_ours_f, e_ref) in _errors(acts, _unpack(ref["act"])).items():
        report[n] = (e_ours_b, e_ours_f, e_ref)
        assert e_ours_b <= 2e-2, (n, e_ours_b)
        assert e_ours_f <= 2 * e_ref + 2e-3, (n, e_ours_f, e_ref)
    for key in ("enc_grad", "pred_grad"):
        for n, (e_ours_b, e_ours_f, e_ref) in _errors(got[key], _unpack(ref[key])).items():
            report[f"{key}.{n}"] = (e_ours_b, e_ours_f, e_ref)
            assert e_ours_f <= max(3e-2, 2 * e_ref + 2e-3), (n, e_ours_f, e_ref)
            assert e_ours_b <= max(3e-2, 3 * e_ref), (n, e_ours_b, e_ref)
    worst = sorted(report.items(), key=lambda kv: -kv[1][1])[:6]
    print(f"reference results from {gold['device']}, torch {gold['torch']}")
    print("ours-vs-ref-bf16 / ours-vs-ref-fp32 / ref-bf16-vs-ref-fp32 (rel-L2), worst by ours-vs-fp32:")
    for k, v in worst:
        print(f"  {k}: {v[0]:.4f} / {v[1]:.4f} / {v[2]:.4f}")
