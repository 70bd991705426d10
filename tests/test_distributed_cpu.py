"""World-size-2 gloo tests of the multi-GPU host logic (batch sharding, logits gather, DDP gradient averaging)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from heuristique_style_transfer_code_b200 import distributed as D


def test_shard_bounds_cover_the_batch():
    for n in (0, 1, 7, 8, 256, 513):
        for world in (1, 2, 3, 8):
            spans = [D.shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    torch.manual_seed(0)
    torch.set_num_threads(1)
    from torchvision import models
    from oracle.torch_port import PortModel
    r, w, _, device = D.init_from_env(backend="gloo")
    assert (r, w) == (rank, world) and device.type == "cpu"
    model = PortModel(models.resnet50(weights=None), 5, 3, 8, return_embeddings=True)
    model.eval()                                   # eval-mode BN: sharded == unsharded (SURVEY section 5)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(5, 3, 32, 32, generator=g)     # 5 rows over 2 ranks: uneven shards
    y = torch.tensor([0, 1, 2, 0, 1])
    with torch.no_grad():
        emb_full, logits_full = model(x)
        emb, logits = model(D.shard_batch(x, rank, world))
    gathered = D.gather_rows(logits, 5, world)
    gathered_emb = D.gather_rows(emb, 5, world)
    ok_gather = torch.allclose(gathered, logits_full, atol=1e-5) and torch.allclose(gathered_emb, emb_full, atol=1e-5)

    # DDP: averaged shard gradients == full-batch gradient when every shard has the same size (4 rows / 2 ranks)
    ddp = D.wrap_ddp(model, device)
    xs, ys = x[:4], y[:4]
    lo, hi = D.shard_bounds(4, rank, world)
    _, out_shard = ddp(xs[lo:hi])
    torch.nn.functional.cross_entropy(out_shard, ys[lo:hi]).backward()
    g_ddp = model.classifier.weight.grad.clone()
    model.zero_grad()
    _, out_full = model(xs)
    torch.nn.functional.cross_entropy(out_full, ys).backward()
    ok_ddp = torch.allclose(g_ddp, model.classifier.weight.grad, rtol=1e-4, atol=1e-6)
    t = D.max_over_ranks(float(rank + 1), device)
    D.barrier(device)
    if rank == 0:
        out.put((bool(ok_gather), bool(ok_ddp), t))
    dist.destroy_process_group()


def test_two_rank_gloo_sharded_inference_and_ddp(monkeypatch):
    # the workers are CPU ranks whatever the machine has: with a GPU visible, init_from_env would give rank r cuda:r
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=240)
        assert p.exitcode == 0
    ok_gather, ok_ddp, t = q.get(timeout=5)
    assert ok_gather and ok_ddp and t == 2.0


def _ddp_options_worker(rank, world, port, out):
    import os
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from heuristique_style_transfer_code_b200 import distributed as D
    torch.manual_seed(0)
    results = {}
    for name, kw in (("plain", {}), ("static", dict(static_graph=True, bucket_cap_mb=1)),
                     ("side_stream_flag", dict(for_graph_capture=True))):
        torch.manual_seed(0)
        net = torch.nn.Sequential(torch.nn.Linear(8, 16), torch.nn.ReLU(), torch.nn.Linear(16, 4))
        ddp = D.wrap_ddp(net, torch.device("cpu"), **kw)
        x = torch.arange(32, dtype=torch.float32).reshape(4, 8) / 10 + rank
        ddp(x).square().mean().backward()
        results[name] = torch.cat([p.grad.flatten() for p in net.parameters()])
    try:
        D.wrap_ddp(torch.nn.Linear(2, 2), torch.device("cpu"), grad_compression="fp8")
        bad = False
    except ValueError:
        bad = True
    if rank == 0:
        out.put((results["plain"].tolist(), results["static"].tolist(), results["side_stream_flag"].tolist(), bad))
    dist.destroy_process_group()


def test_wrap_ddp_options_give_the_same_averaged_gradients():
    """distributed.wrap_ddp on 2 gloo ranks: bucket size, static_graph and the graph-capture construction flag (a no-op
    on CPU) do not change the averaged gradients; unknown compression names are refused."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29741
    procs = [ctx.Process(target=_ddp_options_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    plain, static, flag, bad = out.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert plain == static == flag and bad
