"""GPU: the user-facing training loop — persia_b200.api.TrainCtx (the mirror of persia/ctx.py:655-1055) driving a
DLRM-style PyTorch dense tower on top of the persia_core surface and libpersia_b200, end to end:

    PersiaBatch -> get_embedding_from_data -> ctx.forward (model(non_id, embeddings)) -> loss -> ctx.backward

checked two ways: the loss falls on a learnable synthetic click task, and after k steps the embedding rows equal the
oracle's when it is fed the same id batches and the very gradients autograd produced (the hot path is exact; the dense
tower is PyTorch's business)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

pytestmark = pytest.mark.gpu


@pytest.fixture()
def env(oracle):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from persia_b200 import persia_core as PC

    PC.reset()
    os.environ.pop("RANK", None)
    os.environ.pop("WORLD_SIZE", None)
    yield torch, PC
    PC.reset()


def _batch(rng, api, names, card, B, n_dense, w_true):
    ids = [rng.integers(0, card[i], size=B, dtype=np.uint64) for i in range(len(names))]
    dense = rng.standard_normal((B, n_dense)).astype(np.float32)
    score = dense @ w_true + sum(((ids[i] % 7).astype(np.float32) - 3.0) * 0.3 for i in range(len(names)))
    label = (score > 0).astype(np.float32).reshape(B, 1)
    pb = api.PersiaBatch([api.IDTypeFeatureWithSingleID(names[i], ids[i]) for i in range(len(names))],
                         non_id_type_features=[api.NonIDTypeFeature(dense, name="dense")],
                         labels=[api.Label(label, name="click")], requires_grad=True)
    return pb, ids, label


@pytest.mark.parametrize("dim,optim", [(16, "adagrad"), (32, "sgd")])
def test_trainctx_dlrm_loss_falls_and_rows_match_oracle(env, oracle, dim, optim):
    torch, PC = env
    from persia_b200 import api
    from persia_b200 import workload as W

    rng = np.random.default_rng(3)
    names = [f"slot{i}" for i in range(6)]
    card, B, n_dense, steps = [5, 40, 300, 3000, 50000, 11], 512, 8, 30
    PC.set_embedding_config({"slots_config": {n: {"dim": dim} for n in names}})
    torch.manual_seed(0)
    model = W.make_dlrm_tower(len(names), dim, n_dense=n_dense, bottom=(32,), top=(64, 32)).cuda()
    if optim == "adagrad":
        emb_opt, o_opt = api.Adagrad(lr=0.05), oracle.Optim(oracle.ADAGRAD, lr=0.05, init_acc=0.01, eps=1e-10)
    else:
        emb_opt, o_opt = api.SGD(lr=0.1, weight_decay=1e-4), oracle.Optim(oracle.SGD, lr=0.1, wd=1e-4)
    dense_opt = torch.optim.SGD(model.parameters(), lr=0.3)
    loss_fn = torch.nn.BCEWithLogitsLoss()
    _, slots = PC.parse_embedding_config({"slots_config": {n: {"dim": dim} for n in names}})
    w = oracle.Worker([oracle.SlotCfg(dim, prefix=s.index_prefix) for s in slots], n_ps=1)
    w.configure(wb=10.0)
    w.set_optimizer(o_opt)
    w_true = rng.standard_normal(n_dense).astype(np.float32)
    oracle.set_rsqrt_exact(True)
    losses, seen = [], [set() for _ in names]
    try:
        with api.TrainCtx(model=model, embedding_optimizer=emb_opt, dense_optimizer=dense_opt, device_id=0,
                          mixed_precision=False, embedding_config=api.EmbeddingConfig()) as ctx:
            for step in range(steps):
                pb, ids, label = _batch(rng, api, names, card, B, n_dense, w_true)
                tb = ctx.get_embedding_from_data(pb, 0)
                out, labels = ctx.forward(tb)
                # the embeddings handed to the tower are the oracle's, bit for bit
                flat = np.concatenate(ids)
                want, octx = w.forward(flat, np.arange(len(names) * B + 1, dtype=np.uint32), B, training=True)
                embs = ctx.current_batch.id_type_feature_embedding_torch_tensors
                for i in range(len(names)):
                    assert embs[i].detach().cpu().numpy().tobytes() == want[i].tobytes()
                    seen[i].update(w.ctx_signs(octx, i).tolist())
                loss = loss_fn(out, labels[0].squeeze(1))
                losses.append(float(loss))
                ctx.backward(loss)
                grads = [c[-1].grad.detach().cpu().numpy() for c in ctx.current_batch.id_type_feature_embedding_cache_torch_tensors]
                assert all(g.dtype == np.float16 for g in grads)
                w.backward(octx, grads)
            ctx.backward_engine.flush()
            torch.cuda.synchronize()
            for i, s in enumerate(seen):
                signs = np.array(sorted(s), np.uint64)
                got = ctx.common_context.get_entries(signs, dim)
                for k, sign in enumerate(signs):
                    assert got[k].tobytes() == w.get_entry(int(sign)).tobytes(), (i, k)
        assert np.mean(losses[-5:]) < np.mean(losses[:5]), losses  # it learns; the parity asserts above are the test
    finally:
        oracle.set_rsqrt_exact(False)


# ---- two processes, two GPUs: DDP dense tower + the sharded embedding worker behind TrainCtx ------------------------------
def _trainctx_rank(rank, world, port, result_dir):
    import torch

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    import oracle
    from persia_b200 import api
    from persia_b200 import persia_core as PC
    from persia_b200 import workload as W

    PC.reset()
    names = [f"slot{i}" for i in range(5)]
    card, B, n_dense, steps, dim = [5, 40, 300, 3000, 50000], 256, 8, 6, 32
    PC.set_embedding_config({"slots_config": {n: {"dim": dim} for n in names}})
    torch.manual_seed(0)
    model = W.make_dlrm_tower(len(names), dim, n_dense=n_dense, bottom=(32,), top=(64, 32)).cuda()
    dense_opt = torch.optim.SGD(model.parameters(), lr=0.1)
    loss_fn = torch.nn.BCEWithLogitsLoss()
    rng = np.random.default_rng(11)
    w_true = rng.standard_normal(n_dense).astype(np.float32)
    rec = {"ids": [], "embs": [], "grads": []}
    with api.TrainCtx(model=model, embedding_optimizer=api.Adagrad(lr=0.05), dense_optimizer=dense_opt, device_id=rank,
                      mixed_precision=False, embedding_config=api.EmbeddingConfig()) as ctx:
        assert ctx.world_size == world and type(ctx.model).__name__ == "DistributedDataParallel"
        for step in range(steps):
            batches = [_batch(rng, api, names, card, B, n_dense, w_true) for _ in range(world)]  # all drawn, own kept
            pb, ids, label = batches[rank]
            out, labels = ctx.forward(ctx.get_embedding_from_data(pb, 0))
            rec["ids"].append(np.concatenate(ids))
            rec["embs"].append(np.stack([e.detach().cpu().numpy() for e in ctx.current_batch.id_type_feature_embedding_torch_tensors]))
            loss = loss_fn(out, labels[0].squeeze(1))
            ctx.backward(loss)
            rec["grads"].append(np.stack([c[-1].grad.detach().cpu().numpy()
                                          for c in ctx.current_batch.id_type_feature_embedding_cache_torch_tensors]))
        ctx.backward_engine.flush()
        torch.cuda.synchronize()
        import torch.distributed as dist

        dist.barrier()
        # DDP kept the dense towers identical
        flat = torch.cat([p.detach().flatten() for p in model.parameters()])
        both = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(both, flat)
        assert torch.equal(both[0], both[1])
        _, slots = PC.parse_embedding_config({"slots_config": {n: {"dim": dim} for n in names}})
        np.savez(os.path.join(result_dir, f"prefix{rank}.npz"), prefix=np.array([s.index_prefix for s in slots], np.uint64))
        # every sign any rank used, asked of this rank's shard
        seen = set()
        for step in range(steps):
            t = torch.from_numpy(rec["ids"][step].view(np.int64)).cuda()
            got = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(got, t)
            for g_ in got:
                a = g_.cpu().numpy().view(np.uint64)
                for i in range(len(names)):
                    seen.update(oracle.add_prefix(a[i * B:(i + 1) * B], 8, slots[i].index_prefix).tolist())
        signs = np.array(sorted(seen), np.uint64)
        ent = ctx.common_context.get_entries(signs, dim, missing_ok=True)
        keep = [k for k, e in enumerate(ent) if e is not None]
        np.savez(os.path.join(result_dir, f"rank{rank}.npz"), ids=np.stack(rec["ids"]), embs=np.stack(rec["embs"]),
                 grads=np.stack(rec["grads"]), signs=signs[keep], ent=np.stack([ent[k] for k in keep]))
        dist.barrier()
    PC.reset()


@pytest.mark.gpu
def test_two_process_trainctx_ddp_matches_oracle(env, oracle, tmp_path):
    """persia.ctx.TrainCtx on two ranks: DDP dense tower, embeddings served by the sharded worker (each rank's batch =
    one lookup request per owner, gradient requests applied in rank order — what two nn-workers against two
    parameter servers do, embedding_worker_service/mod.rs:876-1000).  Each rank records ids, embeddings and the f16
    embedding gradients autograd produced; the oracle with 2 parameter servers replays them."""
    torch, PC = env
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket

    import torch.multiprocessing as mp

    world = 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_trainctx_rank, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    res = [np.load(os.path.join(str(tmp_path), f"rank{r}.npz")) for r in range(world)]
    prefix = np.load(os.path.join(str(tmp_path), "prefix0.npz"))["prefix"]
    S, B, dim = 5, 256, 32
    w = oracle.Worker([oracle.SlotCfg(dim, prefix=int(p)) for p in prefix], n_ps=world)
    w.configure(wb=10.0)
    w.set_optimizer(oracle.Optim(oracle.ADAGRAD, lr=0.05, init_acc=0.01, eps=1e-10))
    oracle.set_rsqrt_exact(True)
    try:
        row_off = np.arange(S * B + 1, dtype=np.uint32)
        for step in range(res[0]["ids"].shape[0]):
            octx = [w.forward(res[r]["ids"][step], row_off, B, training=True) for r in range(world)]
            for r in range(world):
                for i in range(S):
                    assert res[r]["embs"][step][i].tobytes() == octx[r][0][i].tobytes(), (step, r, i)
            for r in range(world):
                w.backward(octx[r][1], [res[r]["grads"][step][i] for i in range(S)])
        n = 0
        for r in range(world):
            for k, sign in enumerate(res[r]["signs"]):
                assert res[r]["ent"][k].tobytes() == w.get_entry(int(sign)).tobytes(), (r, k)
                n += 1
        assert n > 0
    finally:
        oracle.set_rsqrt_exact(False)
