"""Pin the oracle: the plain-C restatement vs (a) the reference's 17 golden recalls, (b) the committed
outputs of the reference itself, (c) the compiled reference on random non-integer inputs (stored outputs),
(d) a double-precision model with the reference's own tolerance."""
import numpy as np
import pytest

from conftest import bits, recall_at_k


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_oracle_reproduces_golden_recalls_and_reference_outputs(oracle, dataset, ref_outputs, golden_recalls, metric):
    idx = oracle.index(dataset.data, dataset.graph, dataset.entry_point, metric)
    for e in golden_recalls[metric]:
        ids, dists = idx.search(dataset.queries[100:], 10, e["window"], e["capacity"])
        # tests/integration/vamana/index_search.cpp:138,189-190
        assert abs(recall_at_k(ids, dataset.gt[metric][100:]) - e["recall"]) < 0.0005
        tag = f"{metric}_f32_f32_w{e['window']}_c{e['capacity']}"
        assert np.array_equal(ids, ref_outputs[tag + "_ids"].astype(np.uint64)), tag
        assert np.array_equal(bits(dists), bits(ref_outputs[tag + "_dists"])), tag
    hops, evals = idx.counts(dataset.queries[:64], 32, 48)
    assert np.array_equal(hops, ref_outputs[f"{metric}_counts_w32_c48_hops"])
    assert np.array_equal(evals, ref_outputs[f"{metric}_counts_w32_c48_evals"])


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("pair", ["f32_f16", "f16_f16", "f16_f32", "f32_i8", "i8_i8", "f32_u8", "u8_u8"])
def test_oracle_element_type_pairs(oracle, dataset, ref_outputs, metric, pair):
    q, x = dataset.variant(pair)
    ids, dists = oracle.index(x, dataset.graph, dataset.entry_point, metric).search(q[:256], 10, 24, 40)
    tag = f"{metric}_{pair}_w24_c40"
    assert np.array_equal(ids, ref_outputs[tag + "_ids"].astype(np.uint64)), tag
    assert np.array_equal(bits(dists), bits(ref_outputs[tag + "_dists"])), tag


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("code", [np.int8, np.uint8])
def test_oracle_scalar_quantisation(oracle, dataset, ref_outputs, metric, code):
    raw = dataset.data * np.float32(0.37) + np.float32(1.5)
    idx, codes, scale, bias = oracle.sq_index(raw, dataset.graph, dataset.entry_point, metric, code)
    name = np.dtype(code).name
    assert np.array_equal(codes, ref_outputs[f"sq_{name}_codes"])
    assert np.array_equal(np.array([scale, bias], dtype=np.float32), ref_outputs[f"sq_{name}_scale_bias"])
    qf = dataset.queries * np.float32(0.37) + np.float32(1.5)
    for qn, q in (("f32", qf), ("f16", qf.astype(np.float16))):
        ids, dists = idx.search(q[:256], 10, 24, 40)
        tag = f"{metric}_sq_{name}_{qn}_w24_c40"
        assert np.array_equal(ids, ref_outputs[tag + "_ids"].astype(np.uint64)), tag
        assert np.array_equal(bits(dists), bits(ref_outputs[tag + "_dists"])), tag


def test_oracle_distances_vs_double_precision(oracle):
    """tests/svs/core/distances/distance_euclidean.cpp:42-78: D = 160 and ragged 223, every pair, against a
    double reference with Catch::Approx's default epsilon (100 * FLT_EPSILON relative)."""
    rng = np.random.default_rng(5)
    eps = 100 * np.finfo(np.float32).eps
    for dim in (160, 223):
        for qd, xd in ((np.float32, np.float32), (np.float32, np.float16), (np.float16, np.float16),
                       (np.float32, np.int8), (np.int8, np.int8), (np.uint8, np.uint8)):
            def draw(dt, shape):
                if np.issubdtype(dt, np.integer):
                    info = np.iinfo(dt)
                    return rng.integers(info.min, info.max + 1, shape).astype(dt)
                return rng.standard_normal(shape).astype(dt)
            q, x = draw(qd, dim), draw(xd, (64, dim))
            qq, xx = q.astype(np.float64), x.astype(np.float64)
            want = {"l2": ((xx - qq) ** 2).sum(1), "ip": xx @ qq,
                    "cosine": (xx @ qq) / (np.sqrt((xx * xx).sum(1)) * np.sqrt((qq * qq).sum()))}
            for metric, w in want.items():
                got = oracle.distance_rows(metric, q, x).astype(np.float64)
                scale = np.maximum(np.abs(w), 1.0) if metric != "l2" else np.abs(w)
                assert np.all(np.abs(got - w) <= eps * np.maximum(scale, 1e-30) * 4), (dim, qd, xd, metric)


def test_oracle_matches_compiled_reference_live(oracle, ref_checks):
    """Bit-exact distances and searches against the compiled reference on random non-integer inputs (inputs and
    the reference's outputs stored in tests/golden/ref_checks.npz by tests/golden/make_golden.py)."""
    for dim in (17, 96, 100, 768):
        q, x = ref_checks[f"live_q_{dim}"], ref_checks[f"live_x_{dim}"]
        for metric in ("l2", "ip", "cosine"):
            for p, (qq, xx) in enumerate(((q, x), (q, x.astype(np.float16)), (q.astype(np.float16), x.astype(np.float16)))):
                want = ref_checks[f"live_dist_{dim}_{metric}_{p}"]
                assert np.array_equal(bits(oracle.distance_rows(metric, qq, xx)), bits(want)), (dim, metric, p)
    x, qs, graph = ref_checks["live_x"], ref_checks["live_queries"], ref_checks["live_graph"]
    for metric in ("l2", "ip", "cosine"):
        b = ref_checks[f"live_{metric}_ids"].astype(np.uint64), ref_checks[f"live_{metric}_dists"]
        a = oracle.index(x, graph, 5, metric).search(qs, 5, 9, 14)
        assert np.array_equal(a[0], b[0]) and np.array_equal(bits(a[1]), bits(b[1]))
        a = oracle.index(x, graph, 5, metric).search(qs, 5, 9, 14, visited_set=True)
        assert np.array_equal(a[0], b[0]) and np.array_equal(bits(a[1]), bits(b[1]))


def test_oracle_edge_cases(oracle):
    """Isolated entry point (fewer than k reachable), zero-degree nodes, capacity < k bump, window 1."""
    rng = np.random.default_rng(3)
    x = rng.standard_normal((50, 16)).astype(np.float32)
    q = rng.standard_normal((7, 16)).astype(np.float32)
    graph = np.zeros((50, 5), dtype=np.uint32)
    graph[0, :3] = (2, 1, 2)      # 0 -> {1, 2}; 1 and 2 have no out-edges
    idx = oracle.index(x, graph, 0, "l2")
    ids, dists = idx.search(q, 5, 4, 4)          # capacity 4 < k 5  -> both become 5
    assert np.all(ids[:, 3:] == np.uint64(0xFFFFFFFFFFFFFFFF)) and np.all(np.isposinf(dists[:, 3:]))
    assert np.all(np.sort(ids[:, :3], axis=1) == np.array([0, 1, 2]))
    assert np.all(np.diff(dists[:, :3], axis=1) >= 0)
    with pytest.raises(RuntimeError):
        idx.search(q, 5, 8, 4)                   # window > capacity (SearchBufferConfig::check_invariants)


def test_oracle_lvq8_codec_roundtrip(oracle):
    """LVQ-8 own spec: decode error is bounded by half a quantisation step (+ float16 rounding of the
    per-vector constants); constant vectors and the float16 clamp edge are handled."""
    rng = np.random.default_rng(8)
    x = (rng.standard_normal((200, 100)) * 0.4 + 2.0).astype(np.float32)
    mean = x.mean(axis=0, dtype=np.float64).astype(np.float32)
    x[5] = mean + np.float32(0.75)                # constant after centring: delta == 0
    rows = oracle.lvq8_compress(x, mean)
    assert rows.shape == (200, 128)               # 100 codes + 4 constant bytes, padded to 32
    delta = rows[:, 100:102].copy().view(np.float16).astype(np.float32)
    lower = rows[:, 102:104].copy().view(np.float16).astype(np.float32)
    dec = delta * rows[:, :100].astype(np.float32) + lower + mean
    step = np.maximum(delta, 1e-3)
    assert np.all(np.abs(dec - x) <= 0.5 * step + 1e-5)
    assert np.all(rows[5, :100] == 0) and float(delta[5, 0]) == 0.0
    assert np.all(rows[:, 104:] == 0)
