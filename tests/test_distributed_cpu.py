"""world_size-2 gloo tests of the multi-process host logic (runs on CPU; NCCL is exercised under gpurun):
process-group bootstrap, the autograd-aware collectives, and the data-parallel gradient averaging contract
(every rank ends a step with identical averaged gradients => identical replicas, no data-path collective
other than the gradient all-reduce)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    from src.utils.distributed import AllGather, AllReduce, AllReduceSum, init_distributed
    ws, rk = init_distributed(port=port, rank_and_world_size=(rank, world))
    assert (ws, rk) == (world, rank) and dist.get_backend() == "gloo"
    assert init_distributed() == (world, rank)  # early return once a group exists (distributed.py:20-21)
    x = torch.tensor([float(rank + 1)], requires_grad=True)
    avg = AllReduce.apply(x * 1.0)
    tot = AllReduceSum.apply(x * 1.0)
    gat = AllGather.apply(torch.full((2, 3), float(rank)))
    (avg + tot).sum().backward()
    # DDP contract on a plain module: averaged grads identical on every rank
    torch.manual_seed(0)
    lin = torch.nn.Linear(4, 2)
    ddp = torch.nn.parallel.DistributedDataParallel(lin, static_graph=True)
    ddp(torch.full((3, 4), float(rank + 1))).sum().backward()
    q.put((rank, float(avg), float(tot), gat.tolist(), float(x.grad), lin.weight.grad.tolist()))
    dist.barrier()
    dist.destroy_process_group()


def _hide_gpus(monkeypatch):
    """The workers inherit this environment: without a visible GPU init_distributed() takes gloo, as on a CPU host."""
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")


def test_two_rank_gloo_collectives(monkeypatch):
    _hide_gpus(monkeypatch)
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, avg, tot, gat, xg, wg in res:
        assert avg == 1.5 and tot == 3.0 and xg == 2.0
        assert gat == [[0.0] * 3] * 2 + [[1.0] * 3] * 2
    assert res[0][5] == res[1][5] == [[4.5] * 4] * 2  # mean over ranks of 3 * (rank + 1)


class _FakeStore:
    """offset table of a 3-block toy network in a flat buffer (the layout jepa_b200.params.FlatParamStore produces)."""
    def __init__(self):
        self.offsets, off = {}, 0
        for name, n in [("embed.weight", 40), ("pos", 10)] + [(f"blocks.{i}.{k}", 25) for i in range(3)
                                                            for k in ("norm1.weight", "fc.weight")] + [("norm.weight", 7)]:
            self.offsets[name] = (off, n, (n,))
            off += n
        self.total = off


class _FlatBackward(torch.autograd.Function):
    """Writes a flat gradient buffer back to front the way engine.encoder_backward does and drives FlatGradSync."""
    @staticmethod
    def forward(ctx, x, store, sync, gflat, fill):
        ctx.args = (store, sync, gflat, fill)
        return x.sum()

    @staticmethod
    def backward(ctx, g):
        store, sync, gflat, fill = ctx.args
        sync.begin(gflat)
        o, n, _ = store.offsets["norm.weight"]
        gflat[o:o + n] = fill
        for i in (2, 1, 0):
            lo = store.offsets[f"blocks.{i}.norm1.weight"][0]
            gflat[lo:lo + 50] = fill * (i + 1)
            sync.ready_down_to(lo)
        gflat[:40] = fill * 10     # embed; "pos" stays zero (frozen)
        sync.finish()
        return g.expand(4), None, None, None, None


def _sync_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    from src.utils.distributed import DistributedDataParallel, FlatGradSync, init_distributed
    init_distributed(port=port, rank_and_world_size=(rank, world))
    store = _FakeStore()
    out = []
    for bucket_bytes in (4, 60 * 4, 1 << 30):     # a bucket per block / two blocks per bucket / one bucket at the end
        sync = FlatGradSync(bucket_bytes=bucket_bytes)
        gflat = torch.zeros(store.total)
        x = torch.ones(4, requires_grad=True)
        _FlatBackward.apply(x, store, sync, gflat, float(rank + 1)).backward()
        out.append((sync.n_calls, gflat.tolist()))
    # outside a backward pass: finish(wait=True)
    sync = FlatGradSync()
    g = torch.full((8,), float(rank))
    sync.begin(g)
    sync.finish(wait=True)
    # wrapper: rank-0 parameters everywhere, `module.` state-dict prefix, forward passthrough
    torch.manual_seed(rank)
    ddp = DistributedDataParallel(torch.nn.Linear(3, 2), static_graph=True)
    q.put((rank, out, g.tolist(), ddp.module.weight.tolist(), sorted(ddp.state_dict()),
           list(ddp(torch.ones(1, 3)).shape)))
    dist.barrier()
    dist.destroy_process_group()


def test_flat_grad_sync_two_ranks(monkeypatch):
    _hide_gpus(monkeypatch)
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sync_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    store = _FakeStore()
    want = torch.zeros(store.total)
    want[store.offsets["norm.weight"][0]:] = 1.5
    for i in range(3):
        lo = store.offsets[f"blocks.{i}.norm1.weight"][0]
        want[lo:lo + 50] = 1.5 * (i + 1)
    want[:40] = 15.0
    for (n0, g0), (n1, g1), n_expected in zip(res[0][1], res[1][1], (4, 2, 1)):
        assert n0 == n1 == n_expected                   # bucket schedule identical on every rank (collective order)
        assert g0 == g1 == want.tolist()                # averaged in place, frozen slot untouched
    assert res[0][2] == res[1][2] == [0.5] * 8
    assert res[0][3] == res[1][3]
    assert res[0][4] == ["module.bias", "module.weight"] and res[0][5] == [1, 2]


def test_init_distributed_without_slurm_returns_single_process(monkeypatch):
    from src.utils.distributed import init_distributed
    monkeypatch.delenv("SLURM_NTASKS", raising=False)
    assert init_distributed() == (1, 0)


def test_flat_layout_matches_backward_order():
    """FlatGradSync relies on the flat gradient buffer becoming final from its END towards its START while the
    hand-scheduled backward runs (engine.blocks_backward reports `offset(blocks.i.norm1.weight)` after block i):
    parameters must be registered as [input-side group][block 0]...[block L-1][output-side group], norm1.weight first
    inside a block.  Guards the registration order of the reference-compatible modules."""
    from functools import partial

    import torch.nn as nn

    from jepa_b200.models import VisionTransformer, vit_predictor
    enc = VisionTransformer(img_size=64, patch_size=16, num_frames=4, tubelet_size=2, embed_dim=64, depth=3, num_heads=2,
                            mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6), uniform_power=True)
    pred = vit_predictor(img_size=64, use_mask_tokens=True, patch_size=16, num_frames=4, tubelet_size=2, embed_dim=64,
                         predictor_embed_dim=64, depth=2, num_heads=2, uniform_power=True, num_mask_tokens=2,
                         zero_init_mask_tokens=True)
    for mod, prefix, head, tail in (
            (enc, "blocks.", ("patch_embed.", "pos_embed"), ("norm.",)),
            (pred, "predictor_blocks.", ("predictor_embed.", "mask_tokens.", "predictor_pos_embed"),
             ("predictor_norm.", "predictor_proj."))):
        names = [n for n, _ in mod.named_parameters()]
        kinds = []
        for n in names:
            if n.startswith(prefix):
                kinds.append(1 + int(n[len(prefix):].split(".")[0]))
            elif n.startswith(head):
                kinds.append(0)
            else:
                assert n.startswith(tail), n
                kinds.append(10 ** 6)
        assert kinds == sorted(kinds), names            # head group, blocks ascending, tail group
        depth = max(k for k in kinds if k < 10 ** 6)
        for i in range(depth):
            first = names[kinds.index(1 + i)]
            assert first == f"{prefix}{i}.norm1.weight", first
