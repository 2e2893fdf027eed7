"""CPU: the `persia_core` surface (SURVEY.md §8b).  Checks the module layout `persia/prelude.py` expects and replays
what the reference's OWN Python package, run unchanged on top of this surface, read from it and called on it (its
data / optim classes, and its test/embedding/test_data.py), recorded in tests/golden/persia_core_calls.json."""
import os
import sys
import types

import numpy as np
import pytest


@pytest.fixture()
def pc():
    from persia_b200 import persia_core

    persia_core.reset()
    yield persia_core.install()
    persia_core.reset()


def test_module_layout_matches_prelude(pc):
    import persia_core
    from persia_core import PersiaCommonContext, is_cuda_feature_available  # noqa: F401
    from persia_core.backward import Backward  # noqa: F401
    from persia_core.data import PersiaBatch, check_pyarray_dtype_valid  # noqa: F401
    from persia_core.forward import Forward, PersiaTrainingBatch, Tensor  # noqa: F401
    from persia_core.nats import initialize_dataflow  # noqa: F401
    from persia_core.optim import OptimizerBase  # noqa: F401
    from persia_core.utils import (PersiaBatchDataChannel, PersiaBatchDataReceiver, PersiaBatchDataSender,  # noqa: F401
                                   PersiaMessageQueueClient, PersiaMessageQueueServer)

    for sub in ("data", "forward", "backward", "optim", "utils", "nats"):
        assert isinstance(getattr(persia_core, sub), types.ModuleType)
    ctx = PersiaCommonContext(10, 0, 1, None)
    for name in ("init_nats_publisher", "init_master_discovery_service", "get_embedding_worker_addr_list",
                 "init_rpc_client_with_addr", "wait_servers_ready", "get_embedding_size", "clear_embeddings", "dump", "load",
                 "wait_for_serving", "wait_for_emb_loading", "wait_for_emb_dumping", "shutdown_servers",
                 "send_id_type_features_to_embedding_worker", "send_non_id_type_features_to_nn_worker",
                 "configure_embedding_parameter_servers", "get_embedding_from_data", "get_embedding_from_bytes",
                 "read_from_file", "dump_to_file", "set_embedding"):
        assert callable(getattr(ctx, name)), name
    assert isinstance(ctx.master_addr, str)
    two = PersiaCommonContext(10, 1, 2, None)  # R GPUs: accepted; the sharded worker is built by the first batch
    assert two.get_embedding_worker_addr_list() == ["local"]
    PersiaCommonContext(10, 0, 1, None)


def test_prefix_rule_and_batch_semantics(pc):
    from persia_b200.persia_core import parse_embedding_config

    bits, slots = parse_embedding_config({
        "feature_index_prefix_bit": 12,
        "slots_config": {"a": {"dim": 8}, "b": {"dim": 8}, "c": {"dim": 16, "sqrt_scaling": True}},
        "feature_groups": {"g": ["b", "c"]},
    })
    by = {s.name: s for s in slots}
    assert bits == 12
    assert by["b"].index_prefix == by["c"].index_prefix == 1 << 52  # explicit groups first
    assert by["a"].index_prefix == 2 << 52                          # then one group per remaining slot
    b = pc.data.PersiaBatch()
    b.add_id_type_feature_with_single_id(np.arange(4, dtype=np.uint64), "a")
    with pytest.raises(RuntimeError):  # data.rs:236-240
        b.converted_id_type_features2embedding_tensor(True)
    b = pc.data.PersiaBatch()
    b.add_id_type_feature([np.array([1, 2], np.uint64), np.array([], np.uint64)], "a")
    b.add_label(np.zeros((2, 1), np.float32), np.dtype(np.float32), "y")
    b.converted_id_type_features2embedding_tensor(True)
    assert isinstance(b.to_bytes(), bytes)
    with pytest.raises(RuntimeError):
        b.batch_id()
    with pytest.raises(RuntimeError):  # FeatureBatch::new panics above u16::MAX samples
        pc.data.PersiaBatch().add_id_type_feature_with_single_id(np.zeros(65536, np.uint64), "a")
    ch = pc.utils.PersiaBatchDataChannel(4)
    fwd = pc.forward.Forward(8, False, 1)
    fwd.set_input_channel(ch.get_receiver())
    with pytest.raises(RuntimeError):
        fwd.set_input_channel(ch.get_receiver())
    fwd.launch(2)
    with pytest.raises(TimeoutError):  # forward.rs:875
        fwd.get_batch(5)


def _decode(v, objs):
    if isinstance(v, dict):
        (kind, x), = v.items()
        if kind == "handle":
            return objs[x]
        if kind == "bytes":
            return bytes.fromhex(x)
        if kind == "ndarray":
            return np.array(x["data"], dtype=np.dtype(x["dtype"])).reshape(x["shape"])
        if kind == "dtype":
            return np.dtype(x)
        if kind == "nptype":
            return np.dtype(x).type
        if kind == "npscalar":
            return np.dtype(x["dtype"]).type(x["value"])
        if kind in ("list", "tuple"):
            return (list if kind == "list" else tuple)(_decode(e, objs) for e in x)
        raise ValueError(kind)
    return v


def _replay(scenario):
    """Replays, against this persia_core, every name the reference's `persia` package read from persia_core and every
    call it made, in order, checking each call's outcome: the type it returned or the exception it raised
    (tests/golden/persia_core_calls.json, recorded by tests/golden/make_persia_core_calls.py)."""
    import json

    fx = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "persia_core_calls.json")))
    events = fx["scenarios"][scenario]
    objs = {}

    def resolve(target):
        head, *rest = target.split(".")
        obj = objs[int(head[1:])] if head.startswith("$") else sys.modules[head]
        for part in rest:
            obj = getattr(obj, part)
        return obj

    n_calls = 0
    for k, ev in enumerate(events):
        where = f"event {k}: {ev['target']}"
        if ev["op"] == "getattr":
            v = resolve(ev["target"])
            assert "type" not in ev or type(v).__name__ == ev["type"], where
            continue
        fn = resolve(ev["target"])
        args = [_decode(a, objs) for a in ev["args"]]
        kwargs = {key: _decode(a, objs) for key, a in ev["kwargs"].items()}
        want = ev["result"]
        n_calls += 1
        if "raises" in want:
            with pytest.raises(Exception) as e:
                fn(*args, **kwargs)
            assert type(e.value).__name__ == want["raises"], where
            continue
        r = fn(*args, **kwargs)
        if "handle" in want:
            objs[want["handle"]] = r
        else:
            assert type(r).__name__ == want["type"], where
    return n_calls


def test_reference_python_package_runs_on_the_surface(pc):
    """What the reference's own `persia` package (persia/prelude.py, persia/embedding/{data,optim}.py) asks of
    persia_core when its data, optimizer and config classes are driven: the batch assembly with ids, dense features,
    labels and meta, the requires_grad-without-labels refusal, serialisation, and the three optimizer inits."""
    assert _replay("package_surface") == 18




def test_farmhash_numpy_matches_golden(pc):
    import json

    from persia_b200.persia_core import SlotConfig, _hashstack, farmhash64_np

    fx = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "farmhash64_kat.json")))
    ids = np.array([int(k) for k in fx["hash64"]], np.uint64)
    np.testing.assert_array_equal(farmhash64_np(ids), np.array([int(v, 16) for v in fx["hash64"].values()], np.uint64))
    slot = SlotConfig("t", 32, hash_stack_rounds=2, hash_stack_embedding_size=10)
    got = _hashstack(ids, slot)  # the reference's own test vector (mod.rs:1570-1613)
    assert [g.tolist() for g in got] == [list(v) for v in fx["hashstack_rounds2_size10"].values()]


def test_reference_own_test_file_passes_unmodified(pc):
    """What the reference's test/embedding/test_data.py (5 tests, all passing on this persia_core when recorded) asks
    of persia_core: check_pyarray_dtype_valid over every supported dtype, the requires_grad-without-labels refusal and
    serialisation."""
    assert _replay("reference_test_data") == 15
