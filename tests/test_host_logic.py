"""CPU: host-side logic of the drop-in classes (no compute calls)."""
import json

import numpy as np
import pytest
import torch

import two_tower_model_v2_b200 as pkg
from two_tower_model_v2_b200.vector_db import read_flat_ip_file, write_flat_ip_file


def test_buyer_tower_constructor_and_state_dict():
    m = pkg.BuyerTower()                      # defaults: 384, attention, 128 (buyer_tower.py:14-16)
    assert m.embedding_dim == 384 and m.aggregation_method == "attention"
    sd = m.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {
        "attention.0.weight": (128, 384), "attention.0.bias": (128,),
        "attention.2.weight": (1, 128), "attention.2.bias": (1,)}
    assert sum(v.numel() for v in sd.values()) == 49409
    assert len(pkg.BuyerTower(384, "weighted_avg").state_dict()) == 0
    with pytest.raises(ValueError, match="Unknown aggregation method: nope"):
        pkg.BuyerTower(384, "nope")
    m.aggregation_method = "nope"             # forward re-checks (buyer_tower.py:122)
    with pytest.raises(ValueError, match="Unknown aggregation method"):
        m(torch.zeros(1, 1, 384), torch.zeros(1, 1))


def test_buyer_tower_loads_reference_style_checkpoint():
    sd = {"attention.0.weight": torch.randn(128, 384), "attention.0.bias": torch.randn(128),
          "attention.2.weight": torch.randn(1, 128), "attention.2.bias": torch.randn(1)}
    m = pkg.BuyerTower()
    m.load_state_dict(sd, strict=True)
    assert torch.equal(m.attention[0].weight, sd["attention.0.weight"])


def test_buyer_tower_has_no_cpu_fallback():
    m = pkg.BuyerTower(8, "weighted_avg")
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(2, 3, 8), torch.ones(2, 3))
    with pytest.raises(ValueError):
        m(torch.zeros(2, 3, 8), torch.ones(2, 4))


def test_vector_database_errors_match_reference(tmp_path):
    db = pkg.VectorDatabase(embedding_dim=16)
    assert db.index is None and db.product_ids is None and db.id_to_index is None and db.index_to_id is None
    with pytest.raises(ValueError, match="Embedding dimension mismatch: expected 16, got 8"):
        db.build_index(np.zeros((4, 8), np.float32), ["a", "b", "c", "d"])
    with pytest.raises(ValueError, match="Index not built"):
        db.retrieve(np.zeros(16, np.float32))
    with pytest.raises(ValueError, match="Index not built"):
        db.retrieve_batch(np.zeros((2, 16), np.float32))
    with pytest.raises(ValueError, match="Index not built"):
        db.save_index(str(tmp_path / "nope.faiss"))
    assert not (tmp_path / "nope.faiss").exists()
    assert db.get_embedding("x") is None
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            db.build_index(np.zeros((4, 16), np.float32), ["a", "b", "c", "d"])


def test_flat_file_round_trip(tmp_path):
    rows = np.random.default_rng(0).standard_normal((37, 12)).astype(np.float32)
    p = tmp_path / "product_index.faiss"
    write_flat_ip_file(str(p), rows)
    raw = p.read_bytes()
    assert raw[:4] == b"IxFI" and len(raw) == 45 + rows.nbytes
    assert np.array_equal(read_flat_ip_file(str(p)), rows)
    p.write_bytes(b"IxF2" + raw[4:])
    with pytest.raises(ValueError, match="not an IndexFlatIP"):
        read_flat_ip_file(str(p))
    p.write_bytes(raw[:-4])
    with pytest.raises(ValueError, match="truncated"):
        read_flat_ip_file(str(p))
    p.write_bytes(raw + b"\0\0\0\0")
    with pytest.raises(ValueError, match="unexpected bytes"):
        read_flat_ip_file(str(p))


def test_flat_file_is_byte_exact_faiss_indexflatip_layout(tmp_path):
    """Fence for the on-disk format (reference: faiss.write_index / read_index at vector_db.py:117,77).  The fixture is
    assembled here field by field in the order upstream faiss serialises an IndexFlatIP - faiss/impl/index_write.cpp:
    write_index(): WRITE1(fourcc("IxFI")); write_index_header(): WRITE1(d) [int], WRITE1(ntotal) [idx_t = int64],
    WRITE1(dummy = 1 << 20) twice [idx_t], WRITE1(is_trained) [bool], WRITE1(metric_type) [int, METRIC_INNER_PRODUCT = 0];
    then WRITEXBVECTOR(codes) (faiss/impl/io_macros.h): size_t count of 4-byte units, raw bytes - independently of
    the struct string the writer uses.  faiss itself is not installable in this image: the layout is restated, not
    verified against a real file (INTEGRATION.md says so), which is why the reader rejects anything else."""
    import struct
    rows = (np.arange(3 * 5, dtype=np.float32).reshape(3, 5) - 7.0) / 3.0
    fixture = b"".join([
        b"IxFI",                                 # fourcc: 'I' | 'x' << 8 | 'F' << 16 | 'I' << 24, little endian
        struct.pack("<i", 5),                    # int d
        struct.pack("<q", 3),                    # idx_t ntotal
        struct.pack("<q", 1 << 20),              # idx_t dummy
        struct.pack("<q", 1 << 20),              # idx_t dummy
        struct.pack("<?", True),                 # bool is_trained
        struct.pack("<i", 0),                    # MetricType metric_type = METRIC_INNER_PRODUCT
        struct.pack("<Q", 3 * 5),                # size_t codes.size() / 4
        rows.astype("<f4").tobytes(),            # codes: ntotal * d floats, row-major
    ])
    assert len(fixture) == 45 + 60
    p = tmp_path / "fixture.faiss"
    write_flat_ip_file(str(p), rows)
    assert p.read_bytes() == fixture, "writer must produce the faiss IndexFlatIP byte stream"
    p.write_bytes(fixture)
    assert np.array_equal(read_flat_ip_file(str(p)), rows)
    # everything else is refused loudly: other index types, other metrics, size mismatches
    for tag in (b"IxF2", b"IwFl", b"IxMp", b"ABCD"):
        p.write_bytes(tag + fixture[4:])
        with pytest.raises(ValueError, match="not an IndexFlatIP"):
            read_flat_ip_file(str(p))
    bad_metric = fixture[:33] + struct.pack("<i", 1) + fixture[37:]
    p.write_bytes(bad_metric)
    with pytest.raises(ValueError, match="inconsistent"):
        read_flat_ip_file(str(p))
    bad_count = fixture[:37] + struct.pack("<Q", 14) + fixture[45:]
    p.write_bytes(bad_count)
    with pytest.raises(ValueError, match="inconsistent"):
        read_flat_ip_file(str(p))
    db = pkg.VectorDatabase(embedding_dim=384)
    p.write_bytes(fixture)
    with pytest.raises(ValueError, match="Embedding dimension mismatch"):
        db.load_index(str(p))


def test_event_weights():
    cfg = {"event_weights": {"view": 1, "add_to_cart": 5, "purchase": 10}}
    got = [pkg.get_event_weight(e, cfg) for e in ("View", "AddToCart", "add_to_cart", "Purchase", "BUY", "wishlist")]
    assert got == [1, 5, 5, 10, 10, 1]
    assert pkg.get_event_weight("purchase", {}) == 1


def test_shard_bounds_cover_catalog():
    for n, g in [(10, 4), (10_000_000, 8), (7, 8), (0, 2), (100, 1)]:
        spans = [pkg.shard_bounds(n, g, r) for r in range(g)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert all(0 <= hi - lo <= -(-n // g) for lo, hi in spans)
    with pytest.raises(ValueError):
        pkg.shard_bounds(10, 2, 2)


def _plan(N, D, nq, K):
    import ctypes
    from two_tower_model_v2_b200 import _native
    out = (ctypes.c_int32 * 16)()
    _native.check(_native.load().tt_flat_plan_describe(N, D, nq, K, out), "tt_flat_plan_describe")
    names = ("supported unit_queries k_blocks stages query_units tiles use_threshold route_exact target cap "
             "stride slots rank main_slices seg_cap smem").split()
    return dict(zip(names, out))


def test_search_planner_invariants():
    """The host-side planner (no GPU needed): smem budget, tiling and candidate-budget routing."""
    for N, D, nq, K in [(10_000_000, 384, 128, 100), (1_000_000, 384, 4096, 100), (100_000_000, 384, 1, 100),
                        (10_000_000, 768, 64, 100), (20_000, 384, 2000, 10), (9_000, 64, 16, 1000),
                        (70_000, 256, 40, 500), (2_049, 32, 9, 100), (1, 8, 1, 1), (12_500_000, 384, 1024, 1000),
                        (10_000_000, 384, 129, 100), (10_000_000, 768, 300, 100)]:
        p = _plan(N, D, nq, K)
        assert p["supported"] == 1 and p["smem"] <= 227 * 1024 and p["stages"] >= 2
        # CTA pairs (256 queries per unit) exactly when nq > 128 (rows wider than 640 stream part of the query
        # block); single CTAs keep 128 resident queries while >= 3 full stages fit (D <= 512), else 64
        # (wide rows take pairs from nq > 64: one pass over the catalog instead of two M = 64 units)
        want = 256 if (nq > 128 or (D > 512 and nq > 64)) else (64 if D > 512 else 128)
        assert p["unit_queries"] == want
        assert p["k_blocks"] == -(-D // 64) and p["tiles"] == -(-N // 256)
        assert p["query_units"] == -(-nq // want)
        assert p["stages"] <= 8
        assert 1 <= p["main_slices"] <= max(1, p["tiles"])
        assert not (p["use_threshold"] and p["route_exact"])
        if p["use_threshold"]:
            assert p["target"] >= 2 * K and (p["cap"] >= 4 * p["target"] or p["cap"] == 16384)
            assert 1 <= p["rank"] <= p["slots"] * 8 and p["slots"] <= 4096
            assert p["seg_cap"] >= min(512, -(-p["tiles"] // p["main_slices"]) * 256)
        elif not p["route_exact"]:
            assert p["cap"] >= N and p["seg_cap"] * p["main_slices"] >= N   # every row is a candidate and must fit
    assert _plan(10_000_000, 384, 128, 100)["use_threshold"] == 1
    assert _plan(9_000, 64, 16, 1000)["use_threshold"] == 0
    # units fill the machine: one unit per SM (single) / SM pair (pair) on a 148-SM part
    assert _plan(10_000_000, 384, 128, 100)["main_slices"] == 148
    assert _plan(10_000_000, 384, 256, 100)["main_slices"] == 74



def test_retrieval_pipeline_history_encoding():
    """encode_histories mirrors encoder.py:263-273: timestamp sort only when every interaction has one, last
    `max_interaction_history` kept, event weights by name, unknown ids -> row -1 / counted, padding (-1, 0)."""
    from two_tower_model_v2_b200.retrieval import RetrievalPipeline

    class _Db:
        id_to_index = {"a": 0, "b": 1, "c": 2}
    pipe = RetrievalPipeline.__new__(RetrievalPipeline)
    pipe.db, pipe.max_history = _Db(), 3
    pipe.config = {"event_weights": {"view": 1, "add_to_cart": 5, "purchase": 10}}
    batch = [
        [{"product_id": "c", "event_type": "purchase", "timestamp": "2024-01-03"},
         {"product_id": "a", "event_type": "view", "timestamp": "2024-01-01"},
         {"product_id": "b", "event_type": "AddToCart", "timestamp": "2024-01-02"},
         {"product_id": "zz", "event_type": "buy", "timestamp": "2024-01-04"}],
        [{"product_id": "b", "event_type": "wishlist"}, {"product_id": "a", "event_type": "view", "timestamp": "2020"}],
        [],
    ]
    idx, w, unknown = pipe.encode_histories(batch)
    assert idx.tolist() == [[1, 2, -1], [1, 0, -1], [-1, -1, -1]]       # sorted, truncated to the last 3; unsorted; empty
    assert w.tolist() == [[5.0, 10.0, 10.0], [1.0, 1.0, 0.0], [0.0, 0.0, 0.0]]
    assert unknown == 1 and idx.dtype.name == "int64" and w.dtype.name == "float32"


def test_micro_batcher_groups_requests_and_truncates_k():
    import threading
    from two_tower_model_v2_b200 import MicroBatcher
    calls = []

    def batch_fn(payloads, k):
        calls.append((list(payloads), k))
        return [[(f"{p}-{j}", 1.0 - 0.01 * j) for j in range(k)] for p in payloads]

    with MicroBatcher(batch_fn, max_batch=4, max_wait_ms=200.0) as mb:
        futs = [mb.submit(f"q{i}", k=3 + (i % 2)) for i in range(4)]         # fills one batch at once
        res = [f.result(timeout=5) for f in futs]
        assert [len(r) for r in res] == [3, 4, 3, 4] and res[1][0][0] == "q1-0"
        assert len(calls) == 1 and calls[0] == (["q0", "q1", "q2", "q3"], 4)  # one call, largest k
        out = []
        ts = [threading.Thread(target=lambda i=i: out.append(mb(f"t{i}", 2))) for i in range(6)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert len(out) == 6 and all(len(r) == 2 for r in out)
        assert mb.requests == 10 and 2 <= mb.batches <= 7 and max(len(c[0]) for c in calls) <= 4


def test_micro_batcher_propagates_errors_and_closes():
    import pytest
    from two_tower_model_v2_b200 import MicroBatcher

    def bad(payloads, k):
        raise ValueError("index not built")
    mb = MicroBatcher(bad, max_batch=8, max_wait_ms=1.0)
    f1, f2 = mb.submit("a"), mb.submit("b")
    for f in (f1, f2):
        with pytest.raises(ValueError):
            f.result(timeout=5)
    mb.close()
    with pytest.raises(RuntimeError):
        mb.submit("c")


def test_search_planner_properties_random_shapes():
    """Property test of the host planner over random (N, D, nq, K): shared-memory budget, ring depth, capacities and
    workspace sizes stay consistent for shapes no example-based test covers."""
    from hypothesis import given, settings, strategies as st
    from two_tower_model_v2_b200 import _native
    lib = _native.load()

    @settings(max_examples=300, deadline=None)
    @given(N=st.one_of(st.integers(1, 5000), st.integers(5000, 200_000_000)), D=st.integers(1, 1024),
           nq=st.integers(1, 8192), K=st.integers(1, 2048))
    def check(N, D, nq, K):
        K = min(K, N)
        p = _plan(N, D, nq, K)
        assert p["k_blocks"] == -(-D // 64) and p["tiles"] == -(-N // 256)
        if not p["supported"]:
            assert D > 512                                   # only very wide rows may be rejected
            return
        assert p["smem"] <= 227 * 1024 and p["stages"] >= 2 and p["stages"] <= 8
        assert p["unit_queries"] in (64, 128, 256)
        assert (p["unit_queries"] == 256) == (nq > 128 or (D > 512 and nq > 64))
        assert p["query_units"] * p["unit_queries"] >= nq
        assert 1 <= p["main_slices"] <= max(p["tiles"], 1) and p["main_slices"] <= 1024
        ws = lib.tt_flat_search_workspace_bytes(N, D, nq, K)
        assert ws > 0
        if p["route_exact"]:
            assert not p["use_threshold"] and N > 16384
            return
        assert p["seg_cap"] >= 1 and p["cap"] <= 16384
        if p["use_threshold"]:
            assert p["slots"] >= 1 and p["stride"] >= 1 and p["rank"] >= 1 and p["target"] >= K
            assert p["slots"] <= 4096 and (p["slots"] - 1) * p["stride"] < p["tiles"]
            assert p["cap"] >= min(4 * p["target"], 16384) or p["cap"] == 16384
        else:
            assert N <= 16384 and p["seg_cap"] * p["main_slices"] >= N     # every row can be a candidate
        # candidate segments fit the workspace the ABI asks for
        assert ws >= nq * p["main_slices"] * p["seg_cap"] * 8
    check()


def test_shard_plan_decision_is_rank_independent():
    """tt_flat_shard_plan_ok depends on (N_total, D, nq, K) and on N_local >= K only: every rank decides alike."""
    from two_tower_model_v2_b200 import _native
    lib = _native.load()
    for n_total, d, nq, k in [(10_000_000, 384, 4096, 100), (10_000_000, 768, 1, 10), (3_000_000, 64, 200, 100),
                              (1_000_000, 384, 300, 100), (50_000, 32, 8, 10)]:
        decisions = {lib.tt_flat_shard_plan_ok(nl, n_total, d, nq, k) for nl in (k, 1000 + k, n_total // 8, n_total // 2)}
        assert len(decisions) == 1, (n_total, d, nq, k, decisions)
        assert lib.tt_flat_shard_plan_ok(max(k - 1, 1), n_total, d, nq, k) == (0 if k > 1 else decisions.pop())
    assert lib.tt_flat_shard_plan_ok(1_250_000, 10_000_000, 384, 4096, 100) == 1      # the benchmarked configuration
    assert lib.tt_flat_shard_workspace_bytes(1_250_000, 10_000_000, 384, 4096, 100) > 0
    assert lib.tt_flat_shard_plan_ok(125_000, 1_000_000, 384, 300, 100) == 0          # 1M rows: chunk-mode sample


def test_native_shard_file_roundtrip_and_validation(tmp_path):
    import pytest
    from two_tower_model_v2_b200 import read_native_shard, write_native_shard
    rng = np.random.default_rng(5)
    rows, d, dp = 37, 100, 128
    xn = rng.standard_normal((rows, d)).astype(np.float32)
    xh = rng.integers(0, 65536, (rows, dp), dtype=np.uint16)
    stats = np.array([1.0007, 0.0021, 0.0, 0.0], np.float32)
    p = tmp_path / "shard3.ttb2"
    write_native_shard(str(p), xn, xh, stats, id_offset=1234, n_total=5000)
    assert p.stat().st_size == 64 + rows * d * 4 + rows * dp * 2
    gx, gh, gs, off, ntot = read_native_shard(str(p))
    assert np.array_equal(gx, xn) and np.array_equal(gh, xh) and np.array_equal(gs, stats) and (off, ntot) == (1234, 5000)
    raw = p.read_bytes()
    (tmp_path / "cut").write_bytes(raw[:-10])
    with pytest.raises(ValueError, match="truncated"):
        read_native_shard(str(tmp_path / "cut"))
    (tmp_path / "bad").write_bytes(b"X" + raw[1:])
    with pytest.raises(ValueError, match="not a tt_b200 shard"):
        read_native_shard(str(tmp_path / "bad"))
    with pytest.raises(ValueError, match="pitch"):
        write_native_shard(str(tmp_path / "x"), xn, xh[:, :100], stats)


def test_micro_batcher_hands_out_array_rows_without_python_lists():
    """MicroBatcher + ArrayRows: every caller gets its own row views truncated to its k (a batch_fn returning arrays
    must resolve EVERY future of the batch)."""
    import threading
    calls = []

    def batch_fn(payloads, k):
        calls.append(len(payloads))
        ids = np.stack([np.arange(k) + 100 * p for p in payloads])
        return pkg.ArrayRows(ids, ids.astype(np.float32) / 7)
    out = {}
    with pkg.MicroBatcher(batch_fn, max_batch=8, max_wait_ms=20.0) as mb:
        def client(c):
            out[c] = mb(c, 3 + c % 4)
        ths = [threading.Thread(target=client, args=(c,)) for c in range(20)]
        [t.start() for t in ths]
        [t.join(timeout=30) for t in ths]
        assert not any(t.is_alive() for t in ths), "a caller never got its result"
    for c in range(20):
        ids, scores = out[c]
        assert len(out[c]) == 3 + c % 4 and ids[0] == 100 * c and np.allclose(scores, ids / 7)
    assert sum(calls) == 20 and max(calls) <= 8


def test_infonce_loss_surface_and_no_cpu_fallback():
    """Same constructor / forward signature as the reference InfoNCELoss (losses.py:8-36); CPU tensors raise (there is no
    CPU path), malformed shapes raise ValueError before anything is launched."""
    import torch
    from two_tower_model_v2_b200 import InfoNCELoss
    crit = InfoNCELoss()
    assert crit.temperature == 0.07 and InfoNCELoss(temperature=0.2).temperature == 0.2
    b, p, n = torch.randn(4, 8), torch.randn(4, 8), torch.randn(4, 2, 8)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        crit(b, p, n)
    with pytest.raises(ValueError):
        crit(b, torch.randn(5, 8), n)
    with pytest.raises(ValueError):
        crit(b, p, torch.randn(4, 8))
    with pytest.raises(ValueError):
        crit(b, p, torch.randn(3, 2, 8))
