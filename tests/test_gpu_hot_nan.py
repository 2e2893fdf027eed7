"""The NaN rule (mod.rs:731-746) on slots whose signs go through the hot path of the backward.

The hot items' gradient sums are computed without the NaN verdict (beside the scan) and stepped only afterwards, so a
slot with a NaN, or without a gradient, must still leave its rows untouched, and every other slot must match the CPU
oracle bit for bit.  Slots of cardinality 3 / 5 / 40 at batch 4096 hold giant (> 1024 occurrences), huge (> 256) and
hot items; the last slot holds mostly cold ones.  Also the NaN scan's verdict on its own: the f16 and f32 NaN tests,
the element tail after the last whole 16-byte vector, a gradient that does not start on a 16-byte boundary, and slots
that do not influence each other.
"""
import numpy as np
import pytest

from util import full_row_off, make_batch, to_dev_ids

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
CARD = [3, 5, 40, 100000]
OPTIM_KW = {
    0: dict(lr=0.05, wd=0.001),
    1: dict(lr=0.01, mom=1.0, init_acc=0.01, eps=1e-10),
    2: dict(lr=0.02, mom=0.9, init_acc=0.1, eps=1e-8),
    3: dict(lr=0.01, b1=0.9, b2=0.999, eps=1e-8),
}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return torch


@pytest.fixture(scope="module")
def pb(torch_cuda):
    from persia_b200 import shard

    return shard


@pytest.fixture
def exact_rsqrt(oracle):
    oracle.set_rsqrt_exact(True)
    yield
    oracle.set_rsqrt_exact(False)


def _pair(pb, oracle, dim, kind, n_slots=4):
    """A GPU shard + context and an oracle worker (R=1) with one feature group per slot."""
    pf = [oracle.index_prefix(i) for i in range(n_slots)]
    kw = OPTIM_KW[kind]
    s = pb.EmbeddingShard(dim, 1 << 17, 0)
    s.set_optimizer(kind, **{{"mom": "g_square_momentum", "init_acc": "initialization", "b1": "beta1",
                              "b2": "beta2"}.get(k, k): v for k, v in kw.items()})
    s.configure()
    ctx = pb.BatchContext(1 << 18, 1 << 18, pf)
    w = oracle.Worker([oracle.SlotCfg(dim, prefix=pf[i]) for i in range(n_slots)], n_ps=1)
    w.configure()
    w.set_optimizer(oracle.Optim(kind, **kw))
    return s, ctx, w


def _rows(s, signs):
    ent, found = s.get_entries(to_dev_ids(signs, DEV))
    assert found.cpu().numpy().all()
    return ent.cpu().numpy()


def _equal_oracle(s, w, signs):
    ent = _rows(s, signs)
    for k, sign in enumerate(signs):
        ref = w.get_entry(int(sign))
        assert ref is not None and ent[k].tobytes() == ref.tobytes(), (k, int(sign), ent[k], ref)


def _step(torch, s, ctx, w, rng, B, dim, f32=False, scale=None, nan=None, skip=None):
    """One forward + backward on both sides.  nan = (slot, sample, element): a NaN planted there; skip = a slot sent
    without a gradient.  Checks the status, that a dropped slot's rows did not move, and every touched row."""
    S = len(CARD)
    ids, _, slot_off = make_batch(rng, S, B, CARD)
    got = ctx.forward(s, to_dev_ids(ids, DEV), slot_off, B, training=True).cpu().numpy()
    want, octx = w.forward(ids, full_row_off(S, B), B, training=True)
    for i in range(S):
        np.testing.assert_array_equal(got[i].view(np.uint16), want[i].view(np.uint16))
    stats = ctx.batch_stats()
    signs = [np.array(sorted(set(w.ctx_signs(octx, i).tolist())), np.uint64) for i in range(S)]
    g = (rng.standard_normal((S, B, dim)) * 1e-2).astype(np.float32 if f32 else np.float16)
    if nan is not None:
        g[nan] = np.nan
    grads = [torch.from_numpy(g[i]).to(DEV) for i in range(S)]
    skip_v = None
    if skip is not None:
        grads[skip] = None
        skip_v = [int(i == skip) for i in range(S)]
    dropped = [sl for sl in (nan[0] if nan else None, skip) if sl is not None]
    before = {sl: _rows(s, signs[sl]) for sl in dropped}
    st = ctx.backward(s, grads, scales=scale, want_status=True).cpu().numpy().tolist()
    ost = w.backward(octx, [g[i] for i in range(S)], scale=scale, skip=skip_v)
    assert st == ost
    for sl in dropped:
        assert st[sl] == (1 if sl == skip else 2)
        np.testing.assert_array_equal(_rows(s, signs[sl]).view(np.uint32), before[sl].view(np.uint32))
    for i in range(S):
        _equal_oracle(s, w, signs[i])
    return stats


@pytest.mark.parametrize("f32,scale", [(False, None), (False, [1024.0, 3.0, 1.0, 128.0]), (True, None),
                                       (True, [1024.0, 3.0, 1.0, 128.0])])
def test_nan_in_slot_with_hot_items(torch_cuda, pb, oracle, exact_rsqrt, f32, scale):
    """A NaN in the slot of the giant items, then in the slot of the plain hot items: those slots keep their rows, the
    others match the oracle, and the clean batch after each matches too (the hot bitmaps were all zeroed again)."""
    torch = torch_cuda
    rng = np.random.default_rng(5 + int(f32))
    B, dim = 4096, 64
    s, ctx, w = _pair(pb, oracle, dim, oracle.ADAGRAD)
    stats = _step(torch, s, ctx, w, rng, B, dim, f32, scale)
    assert stats["hot"] >= 3 + 5 + 40 - 2  # (a sign of a tiny slot may be missing from a batch)
    _step(torch, s, ctx, w, rng, B, dim, f32, scale, nan=(0, B - 1, dim - 1))
    _step(torch, s, ctx, w, rng, B, dim, f32, scale)
    _step(torch, s, ctx, w, rng, B, dim, f32, scale, nan=(2, 0, 0))
    _step(torch, s, ctx, w, rng, B, dim, f32, scale)
    assert s.counters()["wait_errors"] == 0


def test_skipped_slot_with_hot_items(torch_cuda, pb, oracle):
    """A slot sent without a gradient (its pointer is never read) that holds giant and huge items."""
    torch = torch_cuda
    rng = np.random.default_rng(11)
    B, dim = 4096, 32
    s, ctx, w = _pair(pb, oracle, dim, oracle.SGD)
    _step(torch, s, ctx, w, rng, B, dim)
    _step(torch, s, ctx, w, rng, B, dim, skip=0)
    _step(torch, s, ctx, w, rng, B, dim, skip=1)
    _step(torch, s, ctx, w, rng, B, dim)


@pytest.mark.parametrize("kind,dim", [(0, 13), (1, 128), (2, 30), (3, 130)])
def test_hot_nan_and_skip_every_optimizer(torch_cuda, pb, oracle, exact_rsqrt, kind, dim):
    """SGD, Adagrad, Adagrad-vectorwise and Adam, with dims that end in a partial group of elements per lane.  For Adam
    every slot is its own feature group: a slot dropped for a NaN must not advance its group's beta powers, which the
    clean steps after it would show."""
    torch = torch_cuda
    rng = np.random.default_rng(100 + dim)
    B = 4096
    s, ctx, w = _pair(pb, oracle, dim, kind)
    _step(torch, s, ctx, w, rng, B, dim)
    _step(torch, s, ctx, w, rng, B, dim, nan=(1, B // 2, dim // 2))
    _step(torch, s, ctx, w, rng, B, dim, skip=0)
    _step(torch, s, ctx, w, rng, B, dim, nan=(0, 7, 0), skip=2)
    _step(torch, s, ctx, w, rng, B, dim)
    _step(torch, s, ctx, w, rng, B, dim)


def test_graph_replay_nan_verdict_from_data(torch_cuda, pb, oracle, exact_rsqrt):
    """A step captured on clean gradients and replayed with a NaN planted before the second replay: the verdict is
    computed from the data on every replay, not frozen at capture."""
    torch = torch_cuda
    rng = np.random.default_rng(23)
    S, B, dim = len(CARD), 4096, 64
    s, ctx, w = _pair(pb, oracle, dim, oracle.ADAM)
    ids_np, _, slot_off = make_batch(rng, S, B, CARD)
    ids_dev = to_dev_ids(ids_np, DEV)
    g_dev = torch.zeros((S, B, dim), dtype=torch.float16, device=DEV)
    out = torch.empty((S, B, dim), dtype=torch.float16, device=DEV)
    grads = [g_dev[i] for i in range(S)]
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        ctx.forward(s, ids_dev, slot_off, B, training=True, out=out)  # eager step (allocations happen here)
        ctx.backward(s, grads)
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            ctx.forward(s, ids_dev, slot_off, B, training=True, out=out)
            ctx.backward(s, grads)
    _, octx = w.forward(ids_np, full_row_off(S, B), B, training=True)
    w.backward(octx, [np.zeros((B, dim), np.float16)] * S)
    for it in range(4):
        ids_np, _, _ = make_batch(rng, S, B, CARD)
        g = (rng.standard_normal((S, B, dim)) * 1e-2).astype(np.float16)
        if it == 1:
            g[0, B - 1, 3] = np.nan
        if it == 2:
            g[2, 0, dim - 1] = np.nan
        ids_dev.copy_(to_dev_ids(ids_np, DEV))
        g_dev.copy_(torch.from_numpy(g).to(DEV))
        graph.replay()
        torch.cuda.synchronize()
        _, octx = w.forward(ids_np, full_row_off(S, B), B, training=True)
        signs = [np.array(sorted(set(w.ctx_signs(octx, i).tolist())), np.uint64) for i in range(S)]
        ost = w.backward(octx, [g[i] for i in range(S)])
        assert ost == [2 if (it, i) in ((1, 0), (2, 2)) else 0 for i in range(S)]
        for i in range(S):
            _equal_oracle(s, w, signs[i])


def _scan_status(torch, pb, oracle, B, dim, bits, f32, offset=0):
    """Status of one backward whose slot gradients hold the given raw bit patterns.  offset: elements between the
    start of an allocation and the start of the gradient (it then does not start on a 16-byte boundary)."""
    S = len(bits)
    s, ctx, _ = _pair(pb, oracle, dim, oracle.SGD, n_slots=S)
    rng = np.random.default_rng(0)
    ids = rng.integers(0, 50, size=S * B, dtype=np.uint64)
    ctx.forward(s, to_dev_ids(ids, DEV), [i * B for i in range(S + 1)], B, training=True)
    it, ft = (torch.int32, torch.float32) if f32 else (torch.int16, torch.float16)
    grads = []
    for b in bits:  # (copied as integers: the bit patterns arrive unchanged)
        buf = torch.zeros(offset + B * dim, dtype=it, device=DEV)
        buf[offset:] = torch.from_numpy(np.ascontiguousarray(b).view(np.int32 if f32 else np.int16)).to(DEV)
        grads.append(buf.view(ft)[offset:].view(B, dim))
    return ctx.backward(s, grads, want_status=True).cpu().numpy().tolist()


@pytest.mark.parametrize("B,dim", [(7, 3), (64, 8), (4096, 64)])
def test_nan_scan_verdict_f16(torch_cuda, pb, oracle, B, dim):
    """f16: NaN iff (h & 0x7fff) > 0x7c00 — +-inf (0x7c00 / 0xfc00) is not NaN, 0x7c01 and -NaN are.  At the first and
    the last element (in the tail after the whole vectors when B * dim % 8 != 0), each slot on its own."""
    torch = torch_cuda
    n = B * dim
    rng = np.random.default_rng(n)
    base = (rng.standard_normal(n) * 1e-2).astype(np.float16).view(np.uint16)

    def with_(pairs):
        b = base.copy()
        for k, v in pairs:
            b[k] = v
        return b

    bits = [with_([(0, 0x7c01)]), with_([(0, 0x7c00), (n - 1, 0xfc00), (n // 2, 0x7c00)]), with_([(n - 1, 0xfe00)]),
            base, with_([(n // 3, 0x7fff)])]
    assert _scan_status(torch, pb, oracle, B, dim, bits, False) == [2, 0, 2, 0, 2]
    # not starting on a 16-byte boundary (8-byte aligned, as a row-major f16 slice with dim % 4 == 0 can be)
    if dim % 4 == 0:
        bits = [with_([(0, 0x7c01)]), with_([(3, 0x7c00), (4, 0xfc00)]), with_([(n - 1, 0x7d00)]), with_([(4, 0x7e00)])]
        assert _scan_status(torch, pb, oracle, B, dim, bits, False, offset=4) == [2, 0, 2, 2]


@pytest.mark.parametrize("B,dim", [(7, 3), (512, 16)])
def test_nan_scan_verdict_f32(torch_cuda, pb, oracle, B, dim):
    """f32: isnan — +-inf (0x7f800000 / 0xff800000) is not NaN, 0x7f800001 and -NaN are."""
    torch = torch_cuda
    n = B * dim
    rng = np.random.default_rng(n)
    base = (rng.standard_normal(n) * 1e-2).astype(np.float32).view(np.uint32)

    def with_(pairs):
        b = base.copy()
        for k, v in pairs:
            b[k] = v
        return b

    bits = [with_([(n - 1, 0x7f800001)]), with_([(0, 0x7f800000), (n - 1, 0xff800000)]), base,
            with_([(0, 0xffc00000)])]
    assert _scan_status(torch, pb, oracle, B, dim, bits, True) == [2, 0, 0, 2]
