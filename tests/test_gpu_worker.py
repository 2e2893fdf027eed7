"""GPU: the sharded path (pb_forward_sharded / pb_backward_sharded through ShardedEmbeddingWorker) against the oracle's
embedding worker with R parameter servers.

R virtual ranks share cuda:0 (own table, context, stream and receive area each; the kernels and the flag protocol are
the ones a multi-GPU box runs, "peer" stores just land in the same GPU; one host thread enqueues them phase by phase), so the R > 1 parity runs on every box,
including the driver's 1-GPU lease.  With >= 2 GPUs the same comparison also runs with one process per GPU over
symmetric memory (torch.multiprocessing spawn).

Semantics checked: a rank's batch is one request per owner; an owner applies the R gradient requests of a step in
rank order (the reference with R NN workers applies them in arrival order).  The oracle therefore runs R forward
requests, then R backward requests in rank order.  Everything bit for bit (Adagrad against the oracle's exact-rsqrt
mode), incl. the per-slot NaN / skipped-slot rule on the requesting rank (mod.rs:731-746)."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from util import f16_ulp_diff, full_row_off, make_batch, to_dev_i32, to_dev_ids  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _optim(N, oracle, kind):
    if kind == oracle.SGD:
        return dict(kind=N.OPT_SGD, lr=0.05, wd=0.001), oracle.Optim(oracle.SGD, lr=0.05, wd=0.001)
    if kind == oracle.ADAGRAD:
        return (dict(kind=N.OPT_ADAGRAD, lr=0.02, initialization=0.01, eps=1e-10),
                oracle.Optim(oracle.ADAGRAD, lr=0.02, init_acc=0.01, eps=1e-10))
    if kind == oracle.ADAM:
        return (dict(kind=N.OPT_ADAM, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8),
                oracle.Optim(oracle.ADAM, lr=0.01, b1=0.9, b2=0.999, eps=1e-8))
    return (dict(kind=N.OPT_ADAGRAD_VW, lr=0.02, initialization=0.01, eps=1e-10),
            oracle.Optim(oracle.ADAGRAD_VW, lr=0.02, init_acc=0.01, eps=1e-10))


def _group(torch, oracle, R, S, dim, kind, B, sqrt=None, rows_f32=False, max_ids=1):
    from persia_b200 import native as N
    from persia_b200.worker import ShardedEmbeddingWorker

    pf = [oracle.index_prefix(i) for i in range(S)]
    gpu_opt, cpu_opt = _optim(N, oracle, kind)
    ws = ShardedEmbeddingWorker.local_group(R, S, dim, pf, 1 << 16, cap=S * B * max_ids, optimizer=gpu_opt, max_batch=B,
                                            sqrt_scaling=sqrt, rows_f32=rows_f32, max_ids_per_sample=max_ids)
    w = oracle.Worker([oracle.SlotCfg(dim, sqrt_scaling=bool(sqrt[i]) if sqrt else False, prefix=pf[i]) for i in range(S)], n_ps=R)
    w.configure()
    w.set_optimizer(cpu_opt)
    for x in ws:  # table storage is allocated on first use, with a device-wide sync: not while a peer spins on a flag
        x.shard.get_entries(torch.zeros(1, dtype=torch.int64, device=DEV))
    torch.cuda.synchronize()
    return ws, w, pf


def _check_rows(torch, oracle, ws, w, signs, R):
    signs = np.array(sorted(signs), np.uint64)
    owner = oracle.shard_of(signs, R)
    for r in range(R):
        mine = signs[owner == r]
        if not mine.size:
            continue
        ent, found = ws[r].shard.get_entries(to_dev_ids(mine, DEV))
        ent = ent.cpu().numpy()
        assert found.all()
        for k, sign in enumerate(mine):
            ref = w.get_entry(int(sign))
            assert ref is not None and ent[k].tobytes() == ref.tobytes(), (r, k, sign)
        assert len(ws[r].shard) == w.ps_len(r)
    for x in ws:
        assert x.status() == (False, False)
        assert x.shard.counters()["wait_errors"] == 0


@pytest.mark.parametrize("R,dim,kind,f32", [(2, 64, 0, False), (2, 128, 1, False), (4, 128, 1, False), (8, 128, 1, False),
                                            (3, 16, 2, True), (2, 12, 0, False), (1, 64, 1, False),
                                            (2, 32, 3, False), (4, 16, 3, True)])  # Adam: beta powers per feature group and request
def test_virtual_ranks_match_oracle(torch_cuda, oracle, R, dim, kind, f32):
    from persia_b200.worker import ShardedEmbeddingWorker as W

    torch = torch_cuda
    oracle.set_rsqrt_exact(True)
    try:
        rng = np.random.default_rng(100 * R + dim)
        S, B, card = 5, 600, [3, 50, 2000, 100000, 11]
        ws, w, pf = _group(torch, oracle, R, S, dim, kind, B)
        outs = [torch.empty((S, B, dim), dtype=torch.float16, device=DEV) for _ in range(R)]
        seen = set()
        for step in range(4):
            ids = [make_batch(rng, S, B, card)[0] for _ in range(R)]
            d_ids = [to_dev_ids(ids[r], DEV) for r in range(R)]
            torch.cuda.synchronize()
            W.group_forward(ws, d_ids, B, training=True, outs=outs)
            torch.cuda.synchronize()
            octx = []
            for r in range(R):
                want, c = w.forward(ids[r], full_row_off(S, B), B, training=True)
                octx.append(c)
                got = outs[r].cpu().numpy()
                for i in range(S):
                    np.testing.assert_array_equal(got[i].view(np.uint16), want[i].view(np.uint16))
                    seen.update(w.ctx_signs(c, i).tolist())
            g = (rng.standard_normal((R, S, B, dim)) * 1e-2).astype(np.float32 if f32 else np.float16)
            skip = [None] * R
            if step == 1:
                g[0, 2, B // 2, dim - 1] = np.nan          # rank 0 drops slot 2 of ITS request; the other ranks' stand
            dg = [[torch.from_numpy(g[r, i]).to(DEV) for i in range(S)] for r in range(R)]
            if step == 2 and R > 1:
                dg[R - 1][0] = None                          # add_skipped_gradient on the last rank
                skip[R - 1] = [1] + [0] * (S - 1)
            torch.cuda.synchronize()
            sts = W.group_backward(ws, dg, want_status=True)
            torch.cuda.synchronize()
            for r in range(R):
                ost = w.backward(octx[r], [g[r, i] for i in range(S)], skip=skip[r])
                assert sts[r].cpu().numpy().tolist() == ost, (step, r)
        _check_rows(torch, oracle, ws, w, seen, R)
    finally:
        oracle.set_rsqrt_exact(False)


def test_virtual_ranks_ragged_sqrt_scale(torch_cuda, oracle):
    """Ragged LIL (several ids per sample, empty samples), sqrt scaling and a loss scale: f32 rows travel, pooling and
    the gradient's sample factors are applied on the requester."""
    from persia_b200.worker import ShardedEmbeddingWorker as W

    torch = torch_cuda
    rng = np.random.default_rng(7)
    R, S, B, dim, card = 3, 4, 300, 32, [5, 300, 40000, 17]
    sqrt = [True, False, True, False]
    ws, w, pf = _group(torch, oracle, R, S, dim, oracle.SGD, B, sqrt=sqrt, rows_f32=True, max_ids=5)
    seen = set()
    for step in range(3):
        batches = [make_batch(rng, S, B, card, max_ids=5, allow_empty=True) for _ in range(R)]
        outs = []
        torch.cuda.synchronize()
        dev_in = [(to_dev_ids(b[0], DEV), to_dev_i32(b[1], DEV)) for b in batches]
        pre = [torch.empty((S, B, dim), dtype=torch.float16, device=DEV) for _ in range(R)]
        torch.cuda.synchronize()
        outs = W.group_forward(ws, [d[0] for d in dev_in], B, training=True, row_offs=[d[1] for d in dev_in],
                               slot_occ_offs=[b[2] for b in batches], outs=pre)
        torch.cuda.synchronize()
        octx = []
        for r in range(R):
            want, c = w.forward(batches[r][0], batches[r][1], B, training=True)
            octx.append(c)
            got = outs[r].cpu().numpy()
            for i in range(S):
                # the f32 sum order of a sample's ids differs (sample order here, shard order there): one f16 step of the
                # largest summand (trained rows reach +-8 in this test and cancel inside a sample)
                np.testing.assert_allclose(got[i].astype(np.float32), want[i].astype(np.float32), rtol=2e-3, atol=8e-3)
                seen.update(w.ctx_signs(c, i).tolist())
        g = (rng.integers(-64, 65, size=(R, S, B, dim)) / 4.0).astype(np.float16)  # x 1/128 stays exact in f32
        scale = [128.0, 1.0, 128.0, 1.0]
        dg = [[torch.from_numpy(g[r, i]).to(DEV) for i in range(S)] for r in range(R)]
        torch.cuda.synchronize()
        W.group_backward(ws, dg, scales=scale)
        torch.cuda.synchronize()
        for r in range(R):
            w.backward(octx[r], [g[r, i] for i in range(S)], scale=scale)
    _check_rows(torch, oracle, ws, w, seen, R)


def test_virtual_ranks_graph_replay(torch_cuda, oracle):
    """The sharded step of every rank — kernels, peer stores, flag waits — captured in CUDA graphs (one per rank and
    phase, since one host thread drives the virtual ranks phase by phase; a process per GPU captures the whole step in
    one graph, bench.py --gpus N) and replayed.  Phase counters live on the device, so replays stay in step."""
    from persia_b200 import native as N

    torch = torch_cuda
    oracle.set_rsqrt_exact(True)
    try:
        rng = np.random.default_rng(11)
        R, S, B, dim, card = 4, 6, 512, 128, [3, 17, 900, 50000, 50000, 11]
        ws, w, pf = _group(torch, oracle, R, S, dim, oracle.ADAGRAD, B)
        ids_dev = [torch.zeros(S * B, dtype=torch.int64, device=DEV) for _ in range(R)]
        g_dev = [torch.zeros((S, B, dim), dtype=torch.float16, device=DEV) for _ in range(R)]
        outs = [torch.empty((S, B, dim), dtype=torch.float16, device=DEV) for _ in range(R)]
        plan = [("f", N.PHASE_SEND), ("f", N.PHASE_SERVE), ("f", N.PHASE_FINISH), ("b", N.PHASE_SEND), ("b", N.PHASE_SERVE)]

        def enqueue(r, kind, ph):
            if kind == "f":
                ws[r].forward(ids_dev[r], B, training=True, out=outs[r], phases=ph)
            else:
                ws[r].backward(g_dev[r], phases=ph)

        def oracle_step(ids, g):
            octx = [w.forward(ids[r], full_row_off(S, B), B, training=True) for r in range(R)]
            for r in range(R):
                w.backward(octx[r][1], [g[r, i] for i in range(S)])
            return [o[0] for o in octx]

        zero_ids = [np.zeros(S * B, np.uint64) for _ in range(R)]
        zero_g = np.zeros((R, S, B, dim), np.float16)
        torch.cuda.synchronize()
        for kind, ph in plan:  # eager warm-up step (id 0 in every slot, zero gradients)
            for r in range(R):
                enqueue(r, kind, ph)
        torch.cuda.synchronize()
        oracle_step(zero_ids, zero_g)
        graphs = {}
        for r in range(R):
            for kind, ph in plan:
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=ws[r].stream, capture_error_mode="thread_local"):
                    enqueue(r, kind, ph)
                graphs[(r, kind, ph)] = gph
        seen = {int(oracle.add_prefix(np.zeros(1, np.uint64), 8, p)[0]) for p in pf}
        for it in range(3):
            ids = [make_batch(rng, S, B, card)[0] for _ in range(R)]
            g = (rng.standard_normal((R, S, B, dim)) * 1e-2).astype(np.float16)
            for r in range(R):
                ids_dev[r].copy_(to_dev_ids(ids[r], DEV))
                g_dev[r].copy_(torch.from_numpy(g[r]).to(DEV))
            torch.cuda.synchronize()
            for kind, ph in plan:
                for r in range(R):
                    with torch.cuda.stream(ws[r].stream):
                        graphs[(r, kind, ph)].replay()
            torch.cuda.synchronize()
            want = oracle_step(ids, g)
            for r in range(R):
                got = outs[r].cpu().numpy()
                for i in range(S):
                    np.testing.assert_array_equal(got[i].view(np.uint16), want[r][i].view(np.uint16))
                    seen.update(oracle.add_prefix(ids[r][i * B:(i + 1) * B], 8, pf[i]).tolist())
        _check_rows(torch, oracle, ws, w, seen, R)
    finally:
        oracle.set_rsqrt_exact(False)


def test_overflow_is_flagged(torch_cuda, oracle):
    """A pair that needs more than cap slots raises the status flag (the excess signs read as zeros)."""
    torch = torch_cuda
    from persia_b200 import native as N
    from persia_b200.worker import ShardedEmbeddingWorker

    S, B, dim, R = 2, 256, 16, 2
    pf = [oracle.index_prefix(i) for i in range(S)]
    ws = ShardedEmbeddingWorker.local_group(R, S, dim, pf, 1 << 12, cap=16, optimizer=dict(kind=N.OPT_SGD, lr=0.1), max_batch=B)
    for x in ws:
        x.shard.get_entries(torch.zeros(1, dtype=torch.int64, device=DEV))
    ids = [to_dev_ids(np.arange(S * B, dtype=np.uint64) + 1000 * r, DEV) for r in range(R)]
    outs = [torch.empty((S, B, dim), dtype=torch.float16, device=DEV) for _ in range(R)]
    torch.cuda.synchronize()
    ShardedEmbeddingWorker.group_forward(ws, ids, B, training=False, outs=outs)
    torch.cuda.synchronize()
    assert all(x.status()[0] for x in ws) and not any(x.status()[1] for x in ws)


# ---- one process per GPU over symmetric memory (needs >= 2 GPUs) --------------------------------------------------------
def _rank_main(rank, world, port, result_dir):
    import torch
    import torch.distributed as dist

    import oracle
    from persia_b200 import native as N
    from persia_b200.worker import ShardedEmbeddingWorker

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    S, B, dim, card = 5, 600, 128, [3, 50, 2000, 100000, 11]
    pf = [oracle.index_prefix(i) for i in range(S)]
    wk = ShardedEmbeddingWorker.distributed(S, dim, pf, 1 << 16, cap=S * B, device=dev, max_batch=B,
                                            optimizer=dict(kind=N.OPT_ADAGRAD, lr=0.02, initialization=0.01, eps=1e-10))
    rng = np.random.default_rng(42)
    outs, seen = [], set()
    for step in range(3):
        ids = [make_batch(rng, S, B, card)[0] for _ in range(world)]  # every rank draws all, keeps its own
        g = (rng.standard_normal((world, S, B, dim)) * 1e-2).astype(np.float16)
        out = wk.forward(torch.from_numpy(ids[rank].view(np.int64)).to(dev), B, training=True)
        wk.backward(torch.from_numpy(g[rank]).to(dev))
        torch.cuda.synchronize()
        dist.barrier()
        outs.append(out.cpu().numpy())
        for r in range(world):
            for i in range(S):
                seen.update(oracle.add_prefix(ids[r][i * B:(i + 1) * B], 8, pf[i]).tolist())
    signs = np.array(sorted(seen), np.uint64)
    mine = signs[oracle.shard_of(signs, world) == rank]
    ent, found = wk.shard.get_entries(torch.from_numpy(mine.view(np.int64)).to(dev))
    assert found.all() and wk.status() == (False, False)
    np.savez(os.path.join(result_dir, f"rank{rank}.npz"), outs=np.stack(outs), signs=mine, ent=ent.cpu().numpy())
    dist.barrier()
    dist.destroy_process_group()


def test_two_processes_symmetric_memory(torch_cuda, oracle, tmp_path):
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs; the virtual-rank tests above cover R > 1 on one GPU")
    import torch.multiprocessing as mp

    world = 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank_main, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    oracle.set_rsqrt_exact(True)
    try:
        S, B, dim, card = 5, 600, 128, [3, 50, 2000, 100000, 11]
        pf = [oracle.index_prefix(i) for i in range(S)]
        w = oracle.Worker([oracle.SlotCfg(dim, prefix=p) for p in pf], n_ps=world)
        w.configure()
        w.set_optimizer(oracle.Optim(oracle.ADAGRAD, lr=0.02, init_acc=0.01, eps=1e-10))
        rng = np.random.default_rng(42)
        res = [np.load(os.path.join(str(tmp_path), f"rank{r}.npz")) for r in range(world)]
        for step in range(3):
            ids = [make_batch(rng, S, B, card)[0] for _ in range(world)]
            g = (rng.standard_normal((world, S, B, dim)) * 1e-2).astype(np.float16)
            octx = [w.forward(ids[r], full_row_off(S, B), B, training=True) for r in range(world)]
            for r in range(world):
                for i in range(S):
                    np.testing.assert_array_equal(res[r]["outs"][step][i].view(np.uint16), octx[r][0][i].view(np.uint16))
            for r in range(world):
                w.backward(octx[r][1], [g[r, i] for i in range(S)])
        for r in range(world):
            for k, sign in enumerate(res[r]["signs"]):
                assert res[r]["ent"][k].tobytes() == w.get_entry(int(sign)).tobytes()
    finally:
        oracle.set_rsqrt_exact(False)
