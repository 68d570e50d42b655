"""GPU parity: the CUDA path (through the C ABI) vs the reference's own outputs and the oracle.

Bar (BASELINE.json north_star): neighbour ids bit-exact at a fixed search window; the design
goal -- and what is asserted here -- is bit-exact distances too (tolerance 0 ulp).
"""
import numpy as np
import pytest

from conftest import bits, knn_graph, recall_at_k

pytestmark = pytest.mark.gpu

METRICS = {"l2": 0, "ip": 1, "cosine": 2}


def make_index(data, graph, ep, metric, **kw):
    from scalablevectorsearch_b200 import DistanceType, Vamana
    return Vamana.from_arrays(data, graph, ep, DistanceType(METRICS[metric]), **kw)


def search(index, queries, k, window, capacity=None):
    from scalablevectorsearch_b200 import SearchBufferConfig
    index.search_parameters.buffer_config = SearchBufferConfig(window, capacity)
    return index.search(queries, k)


def assert_same(got, want_ids, want_dists, tag):
    ids, dists = got
    assert np.array_equal(ids.astype(np.uint64), want_ids.astype(np.uint64)), f"{tag}: neighbour ids differ"
    assert np.array_equal(bits(dists), bits(want_dists)), f"{tag}: distances differ (bit-exact bar)"


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_golden_configs_match_reference(dataset, ref_outputs, golden_recalls, metric):
    """All 17 (window, capacity) goldens: ids and distances equal the reference's, recall equals the TOML's."""
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, metric)
    for e in golden_recalls[metric]:
        got = search(index, dataset.queries[100:], 10, e["window"], e["capacity"])
        tag = f"{metric}_f32_f32_w{e['window']}_c{e['capacity']}"
        assert_same(got, ref_outputs[tag + "_ids"], ref_outputs[tag + "_dists"], tag)
        # tests/integration/vamana/index_search.cpp:138,189-190: |recall - expected| < 0.0005
        assert abs(recall_at_k(got[0], dataset.gt[metric][100:]) - e["recall"]) < 0.0005


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("pair", ["f32_f16", "f16_f16", "f16_f32", "f32_i8", "i8_i8", "f32_u8", "u8_u8"])
def test_element_type_pairs_match_reference(dataset, ref_outputs, metric, pair):
    q, x = dataset.variant(pair)
    index = make_index(x, dataset.graph, dataset.entry_point, metric)
    got = search(index, q[:256], 10, 24, 40)
    tag = f"{metric}_{pair}_w24_c40"
    assert_same(got, ref_outputs[tag + "_ids"], ref_outputs[tag + "_dists"], tag)


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("code", ["int8", "uint8"])
def test_scalar_quantised_matches_reference(dataset, ref_outputs, metric, code):
    codes = ref_outputs[f"sq_{code}_codes"]
    scale, bias = ref_outputs[f"sq_{code}_scale_bias"]
    index = make_index(codes, dataset.graph, dataset.entry_point, metric, sq=(scale, bias))
    qf = dataset.queries * np.float32(0.37) + np.float32(1.5)
    for qn, q in (("f32", qf), ("f16", qf.astype(np.float16))):
        got = search(index, q[:256], 10, 24, 40)
        tag = f"{metric}_sq_{code}_{qn}_w24_c40"
        assert_same(got, ref_outputs[tag + "_ids"], ref_outputs[tag + "_dists"], tag)


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_counters_match_reference_tracker(dataset, ref_outputs, metric):
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, metric)
    index.set_counting(True)
    search(index, dataset.queries[:64], 10, 32, 48)
    hops, evals = index.counters(64)
    assert np.array_equal(hops, ref_outputs[f"{metric}_counts_w32_c48_hops"])
    assert np.array_equal(evals, ref_outputs[f"{metric}_counts_w32_c48_evals"])
    fetched = index.fetched(64)
    assert np.all(fetched <= evals) and np.all(fetched >= hops)


@pytest.mark.parametrize("slots", [0, 64, 1024, 16384])
def test_visited_filter_never_changes_results(dataset, ref_outputs, slots):
    """search_buffer.h:420 "Visited set use does not affect accuracy": any filter size, same bits."""
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    index.set_option("visited_filter_slots", slots)
    index.set_counting(True)
    got = search(index, dataset.queries[100:], 10, 22, 23)
    assert_same(got, ref_outputs["l2_f32_f32_w22_c23_ids"], ref_outputs["l2_f32_f32_w22_c23_dists"], f"filter {slots}")
    hops, evals = index.counters(900)
    fetched = index.fetched(900)
    if slots == 0:
        # without the filter every neighbour is read, except the in-row repeats removed at upload
        assert np.all(fetched <= evals) and fetched.sum() > 0.98 * evals.sum()
    else:
        assert fetched.sum() < evals.sum()


@pytest.mark.parametrize("dim,max_degree", [(17, 8), (96, 64), (100, 32), (223, 24), (300, 12), (768, 16)])
@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_ragged_dims_vs_oracle(oracle, dim, max_degree, metric):
    """Non-integer data, ragged dimensions (masked tail), several graph degrees, every float pair."""
    rng = np.random.default_rng(dim * 7 + max_degree)
    n = 1500
    x = rng.standard_normal((n, dim)).astype(np.float32)
    q = rng.standard_normal((200, dim)).astype(np.float32)
    graph = knn_graph(x, max_degree, rng)
    for xt, qt in ((x, q), (x.astype(np.float16), q), (x.astype(np.float16), q.astype(np.float16))):
        index = make_index(xt, graph, 3, metric)
        want = oracle.index(xt, graph, 3, metric)
        for window, cap in ((1, 1), (8, 8), (16, 40), (64, 64)):
            k = min(10, cap)
            got = search(index, qt, k, window, cap)
            wi, wd = want.search(qt, k, window, cap)
            assert_same(got, wi, wd, f"{metric} d{dim} R{max_degree} {xt.dtype}/{qt.dtype} w{window} c{cap}")


def test_window_smaller_than_k_is_bumped(dataset, oracle):
    """index/vamana/index.h:590-592: capacity < k resets window = capacity = k."""
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    want = oracle.index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    got = search(index, dataset.queries[:100], 10, 1, 1)
    wi, wd = want.search(dataset.queries[:100], 10, 1, 1)
    assert_same(got, wi, wd, "bump")
    assert_same(got, *want.search(dataset.queries[:100], 10, 10, 10), "bump==w10")


def test_large_window_and_batch_properties(dataset):
    """Size-independent properties at a large window: sortedness, no duplicate ids, the single-query
    result equals the batched row (bindings/python/tests/test_vamana.py:111-137), idempotence."""
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    q = np.tile(dataset.queries, (4, 1))
    ids, dists = search(index, q, 50, 200, 256)
    assert np.all(np.diff(dists, axis=1) >= 0)
    assert all(len(set(r.tolist())) == len(r) for r in ids)
    assert np.array_equal(ids[:1000], ids[1000:2000]) and np.array_equal(ids[:1000], ids[3000:])
    one = search(index, q[7:8], 50, 200, 256)
    assert np.array_equal(one[0][0], ids[7]) and np.array_equal(bits(one[1][0]), bits(dists[7]))
    again = search(index, q, 50, 200, 256)
    assert np.array_equal(again[0], ids) and np.array_equal(bits(again[1]), bits(dists))


def test_error_behaviour(dataset):
    from scalablevectorsearch_b200 import SearchBufferConfig, Svsb200Error
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    with pytest.raises(ValueError):
        SearchBufferConfig(20, 10)
    with pytest.raises(ValueError):
        index.search(dataset.queries[:, :64], 10)
    with pytest.raises(Svsb200Error):   # unsupported query dtype throws (index_search.cpp)
        index.search(dataset.queries.astype(np.int8), 10)
    ids, dists = index.search(dataset.queries[:0], 10)   # empty batch
    assert ids.shape == (0, 10)


def test_cpp_adapter_cli_matches_python_path(dataset, ref_outputs, tmp_path):
    """BASELINE config #1 through the C++ boundary: the reference's `search_index` CLI with a
    GpuVamanaIndex behind `svs::Vamana` (scalablevectorsearch_b200/cpp) writes the same ids as the
    reference's CPU path (committed outputs) for the prebuilt test graph."""
    import os
    import subprocess
    from conftest import ROOT
    from scalablevectorsearch_b200 import io
    exe = os.path.join(ROOT, "scalablevectorsearch_b200", "cpp", "_build", "search_index_gpu")
    if not os.path.exists(exe):
        pytest.skip("search_index_gpu not built (needs the reference headers at build time)")
    io.write_svs(str(tmp_path / "data.svs"), dataset.data)
    io.write_svs(str(tmp_path / "graph.svs"), dataset.graph)
    io.write_vecs(str(tmp_path / "queries.fvecs"), dataset.queries[100:])
    (tmp_path / "config.toml").write_text(
        "__version__ = 'v0.0.2'\n[object]\n__schema__ = 'vamana_index_parameters'\n__version__ = 'v0.0.3'\n"
        f"entry_point = {dataset.entry_point}\nname = 'vamana index parameters'\n"
        "[object.build_parameters]\n__schema__ = 'vamana_build_parameters'\n__version__ = 'v0.0.1'\nalpha = 1.2\n"
        "graph_max_degree = 128\nmax_candidate_pool_size = 1000\nname = 'vamana build parameters'\nprune_to = 128\n"
        "use_full_search_history = true\nwindow_size = 200\n"
        "[object.search_parameters]\n__schema__ = 'vamana_search_parameters'\n__version__ = 'v0.0.1'\n"
        "prefetch_lookahead = 0\nprefetch_step = 0\nsearch_buffer_capacity = 0\nsearch_buffer_visited_set = false\n"
        "search_window_size = 0\n")
    out = subprocess.run([exe, "float", "float", str(tmp_path / "queries.fvecs"), "15", "10", "2",
                          str(tmp_path / "config.toml"), str(tmp_path / "graph.svs"), str(tmp_path / "data.svs"),
                          str(tmp_path / "res"), "L2"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "GpuVamanaIndex" in out.stdout
    ids = io.read_vecs(str(tmp_path / "res_idx.ivecs"))
    assert np.array_equal(ids.astype(np.uint32), ref_outputs["l2_f32_f32_w15_c15_ids"])


@pytest.mark.parametrize("metric", ["l2", "ip"])
@pytest.mark.parametrize("dim", [96, 100])
def test_lvq8_fused_decompress_distance_vs_oracle(oracle, metric, dim):
    """LVQ-8 (own specification -- the reference's LVQ is closed source, parity with Intel's binary is
    UNPINNED): GPU encoder bytes == oracle encoder bytes, fused decompress+distance search == oracle,
    and the compressed search keeps recall close to the uncompressed one."""
    from scalablevectorsearch_b200 import lvq8_compress
    rng = np.random.default_rng(dim)
    n = 3000
    centres = rng.standard_normal((20, dim)).astype(np.float32)
    x = (centres[rng.integers(0, 20, n)] + 0.3 * rng.standard_normal((n, dim))).astype(np.float32)
    q = (centres[rng.integers(0, 20, 300)] + 0.3 * rng.standard_normal((300, dim))).astype(np.float32)
    graph = knn_graph(x, 32, rng)
    rows, mean = lvq8_compress(x)
    want_rows = oracle.lvq8_compress(x, mean)
    assert np.array_equal(rows, want_rows), "LVQ-8 encoder bytes differ from the oracle"
    index = make_index(rows, graph, 7, metric, lvq8=(dim, mean))
    want = oracle.lvq8_index(rows, dim, mean, graph, 7, metric)
    for qq in (q, q.astype(np.float16)):
        for window, cap in ((8, 8), (32, 48)):
            got = search(index, qq, 8, window, cap)
            wi, wd = want.search(qq, 8, window, cap)
            assert_same(got, wi, wd, f"lvq8 {metric} d{dim} {qq.dtype} w{window}")
    # recall of the compressed index vs the exact index on the same graph (scalar_search.cpp uses eps 0.008)
    exact = search(make_index(x, graph, 7, metric), q, 8, 32, 48)[0]
    comp = search(index, q, 8, 32, 48)[0]
    overlap = np.mean([len(set(a.tolist()) & set(b.tolist())) for a, b in zip(exact, comp)]) / 8
    assert overlap > 0.93, overlap


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_exhaustive_scan_is_exact_topk(oracle, metric):
    """svsb200_exhaustive_device: top-k over all base vectors with the search path's own distance code,
    ties broken by id -- checked against oracle distances sorted by (distance, id)."""
    import torch
    rng = np.random.default_rng(1)
    n, dim, nq, k = 3000, 100, 40, 12
    x = np.round(rng.standard_normal((n, dim)) * 3).astype(np.float32)      # coarse grid: plenty of exact ties
    q = np.round(rng.standard_normal((nq, dim)) * 3).astype(np.float32)
    graph = np.zeros((n, 2), dtype=np.uint32)
    index = make_index(x, graph, 0, metric)
    dq = torch.from_numpy(q).cuda()
    ids = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dists = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    index.exhaustive_device(dq.data_ptr(), np.float32, nq, k, ids.data_ptr(), dists.data_ptr(),
                            stream=torch.cuda.current_stream().cuda_stream or 1)
    torch.cuda.synchronize()
    ids, dists = ids.cpu().numpy(), dists.cpu().numpy()
    for i in range(nq):
        d = oracle.distance_rows(metric, q[i], x)
        key = -d if metric != "l2" else d
        order = np.lexsort((np.arange(n), key))[:k]
        assert np.array_equal(ids[i], order), (metric, i)
        assert np.array_equal(bits(dists[i]), bits(d[order]))


def test_assemble_from_files_like_the_reference_binding(dataset, ref_outputs, tmp_path):
    """`svs.Vamana(config_path, GraphLoader(...), VectorDataLoader(...), distance)` (bindings/python/src/vamana.cpp:340-348)
    over on-disk files in the reference's formats, then `search_window_size` + `search`."""
    from scalablevectorsearch_b200 import DataType, DistanceType, GraphLoader, Vamana, VectorDataLoader, io
    io.write_svs(str(tmp_path / "data.svs"), dataset.data)
    io.write_svs(str(tmp_path / "graph.svs"), dataset.graph)
    (tmp_path / "config.toml").write_text(
        f"[object]\nentry_point = {dataset.entry_point}\n[object.search_parameters]\nsearch_window_size = 7\n"
        "search_buffer_capacity = 9\n")
    index = Vamana(str(tmp_path / "config.toml"), GraphLoader(str(tmp_path / "graph.svs")),
                   VectorDataLoader(str(tmp_path / "data.svs"), DataType.float32, dims=128), distance=DistanceType.Cosine)
    assert (index.size, index.dimensions, index.graph_max_degree) == (10000, 128, 128)
    # index.apply(config): the saved search parameters are the defaults (index/vamana/index.h:1047-1048)
    cfg = index.search_parameters.buffer_config
    assert (cfg.search_window_size, cfg.search_buffer_capacity) == (7, 9)
    from scalablevectorsearch_b200 import Svsb200Error
    with pytest.raises(Svsb200Error):      # VectorDataLoader(dims=...) is checked against the file
        Vamana(str(tmp_path / "config.toml"), GraphLoader(str(tmp_path / "graph.svs")),
               VectorDataLoader(str(tmp_path / "data.svs"), DataType.float32, dims=96))
    with pytest.raises(TypeError):         # declared query type (default float32) is enforced
        index.search(dataset.queries[:4].astype(np.float16), 10)
    # the same data as .fvecs goes through the strided vecs reader
    io.write_vecs(str(tmp_path / "data.fvecs"), dataset.data)
    index2 = Vamana(str(tmp_path / "config.toml"), GraphLoader(str(tmp_path / "graph.svs")),
                    VectorDataLoader(str(tmp_path / "data.fvecs"), DataType.float32), distance=DistanceType.Cosine)
    index2.search_window_size = 100
    i2, d2 = index2.search(dataset.queries[100:], 10)
    assert_same((i2, d2), ref_outputs["cosine_f32_f32_w100_c100_ids"], ref_outputs["cosine_f32_f32_w100_c100_dists"],
                "assemble from fvecs")
    index.search_window_size = 100
    assert index.search_parameters.buffer_config.search_buffer_capacity == 100
    ids, dists = index.search(dataset.queries[100:], 10)
    assert ids.dtype == np.uint64 and dists.dtype == np.float32
    assert_same((ids, dists), ref_outputs["cosine_f32_f32_w100_c100_ids"], ref_outputs["cosine_f32_f32_w100_c100_dists"],
                "assemble-from-files cosine w100")


def test_assemble_rejects_a_device_listed_twice(dataset, tmp_path):
    """Assembling from files checks the device list like creating from arrays does: one replica per device."""
    from scalablevectorsearch_b200 import DataType, GraphLoader, Svsb200Error, Vamana, VectorDataLoader, io
    io.write_svs(str(tmp_path / "data.svs"), dataset.data)
    io.write_svs(str(tmp_path / "graph.svs"), dataset.graph)
    (tmp_path / "config.toml").write_text(f"[object]\nentry_point = {dataset.entry_point}\n")
    with pytest.raises(Svsb200Error, match="svsb200_index_assemble: device listed twice"):
        Vamana(str(tmp_path / "config.toml"), GraphLoader(str(tmp_path / "graph.svs")),
               VectorDataLoader(str(tmp_path / "data.svs"), DataType.float32), device=[0, 0])


# ------------------------------------------------------------------------------------------------
# round 2: the holes VERDICT r1 listed + the lean kernel against the generic one
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_fewer_than_k_reachable_matches_oracle(oracle, metric):
    """Isolated entry point / zero-degree nodes / fewer than k reachable (tests/integration/vamana/index_search.cpp
    never has this; the reference copies stale buffer slots, extensions.h:588-590): the kernel and the oracle pad
    with id = all-ones and +inf (L2) / -inf (IP, cosine), and agree bit for bit on the valid prefix."""
    rng = np.random.default_rng(3)
    x = rng.standard_normal((50, 16)).astype(np.float32)
    q = rng.standard_normal((7, 16)).astype(np.float32)
    graph = np.zeros((50, 5), dtype=np.uint32)
    graph[0, :3] = (2, 1, 2)      # 0 -> {1, 2}; 1 and 2 have no out-edges
    graph[7, :2] = (1, 7)         # a self-loop elsewhere
    for ep, nvalid in ((0, 3), (1, 1), (7, 1)):
        index = make_index(x, graph, ep, metric)
        want = oracle.index(x, graph, ep, metric)
        for generic in (0, 1):
            index.set_option("generic_kernel", generic)
            got = search(index, q, 5, 4, 4)        # capacity 4 < k 5 -> both become 5 (index.h:590-592)
            wi, wd = want.search(q, 5, 4, 4)
            assert_same(got, wi, wd, f"{metric} ep{ep} generic{generic}")
            assert np.all(got[0][:, nvalid:] == np.uint64(0xFFFFFFFFFFFFFFFF))
            pad = got[1][:, nvalid:]
            assert np.all(np.isposinf(pad) if metric == "l2" else np.isneginf(pad))


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_lean_and_generic_kernels_agree(dataset, oracle, metric):
    """Every configuration the lean kernel takes gives the generic kernel's bits (and both the oracle's): window
    past one 128-entry block, split buffer, tiny window, wide graph rows (128 neighbours = 4 register words)."""
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, metric)
    want = oracle.index(dataset.data, dataset.graph, dataset.entry_point, metric)
    q = dataset.queries[:192]
    for window, cap, k in ((1, 1, 1), (10, 10, 10), (33, 97, 20), (128, 128, 10), (130, 300, 50), (300, 300, 100)):
        wi, wd = want.search(q, k, window, cap)
        for generic in (0, 1):
            index.set_option("generic_kernel", generic)
            got = search(index, q, k, window, cap)
            assert index.get_option("last_kernel") == 1 - generic
            assert_same(got, wi, wd, f"{metric} w{window} c{cap} generic{generic}")


def test_configurations_outside_the_lean_kernel_fall_back(oracle):
    """max_degree > 128 and filter-off runs take the generic kernel; same bits as the oracle either way."""
    rng = np.random.default_rng(11)
    n, dim = 1200, 32
    x = rng.standard_normal((n, dim)).astype(np.float32)
    q = rng.standard_normal((64, dim)).astype(np.float32)
    graph = knn_graph(x, 140, rng)
    index = make_index(x, graph, 1, "l2")
    wi, wd = oracle.index(x, graph, 1, "l2").search(q, 10, 40, 64)
    assert_same(search(index, q, 10, 40, 64), wi, wd, "R140")
    assert index.get_option("last_kernel") == 0
    graph64 = knn_graph(x, 64, rng)
    index = make_index(x, graph64, 1, "l2")
    wi, wd = oracle.index(x, graph64, 1, "l2").search(q, 10, 40, 64)
    assert_same(search(index, q, 10, 40, 64), wi, wd, "R64 lean")
    assert index.get_option("last_kernel") == 1
    index.set_option("visited_filter_slots", 0)
    assert_same(search(index, q, 10, 40, 64), wi, wd, "R64 filter off")
    assert index.get_option("last_kernel") == 0
    from scalablevectorsearch_b200 import Svsb200Error
    with pytest.raises(Svsb200Error):
        index.set_option("visited_filter_slots", 4)     # would break the 16-byte alignment of the arrays behind it


@pytest.mark.parametrize("id_bytes", [4, 8])
def test_search_device_matches_host_path(dataset, ref_outputs, id_bytes):
    """svsb200_search_device (device-resident buffers, caller's stream; the path bench.py times as `value`)."""
    import torch
    from scalablevectorsearch_b200 import SearchBufferConfig
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    index.search_parameters.buffer_config = SearchBufferConfig(22, 23)
    q = torch.from_numpy(dataset.queries[100:]).cuda()
    ids = torch.empty((900, 10), dtype=torch.int32 if id_bytes == 4 else torch.int64, device="cuda")
    dists = torch.empty((900, 10), dtype=torch.float32, device="cuda")
    index.search_device(q.data_ptr(), np.float32, 900, 10, ids.data_ptr(), dists.data_ptr(),
                        stream=torch.cuda.current_stream().cuda_stream or 1, id_bytes=id_bytes)
    torch.cuda.synchronize()
    assert_same((ids.cpu().numpy(), dists.cpu().numpy()), ref_outputs["l2_f32_f32_w22_c23_ids"],
                ref_outputs["l2_f32_f32_w22_c23_dists"], f"search_device id_bytes={id_bytes}")


@pytest.mark.parametrize("greater", [False, True])
@pytest.mark.parametrize("shards", [2, 3, 8])
def test_merge_topk_device_is_the_total_order(shards, greater):
    """svsb200_merge_topk_device == sort of all shards' candidates by TotalOrder (distance, then id;
    lib/neighbor.h:143-155), with exact ties across and INSIDE shards (a shard's list is in insertion order,
    not id order), -1 padding and short lists."""
    import torch
    from scalablevectorsearch_b200.multi_gpu import cuda_merge, merge_topk_reference_order
    rng = np.random.default_rng(shards * 2 + greater)
    nq, k = 257, 10
    ids = np.full((shards, nq, k), -1, dtype=np.int64)
    dists = np.zeros((shards, nq, k), dtype=np.float32)
    sign = -1.0 if greater else 1.0
    for s in range(shards):
        for q in range(nq):
            m = int(rng.integers(0, k + 1))                          # short lists, sometimes empty
            d = np.sort(rng.integers(0, 4, size=m).astype(np.float32))    # 4 distinct values: ties everywhere
            if q % 7 == 0:
                d = d * 0.0 - (0.0 if q % 14 else 0.0)               # all-equal rows
            if q % 11 == 0 and m:
                d[0] = -0.0                                            # -0 == +0 under operator<
            pool = rng.permutation(1000)[:m] + 1000 * s               # shard-disjoint ids, NOT sorted inside ties
            ids[s, q, :m] = pool
            dists[s, q, :m] = sign * d
            dists[s, q, m:] = -np.inf if greater else np.inf
    want_i, want_d = merge_topk_reference_order(ids, dists, k, greater)
    got_i, got_d = cuda_merge(torch.from_numpy(ids).cuda(), torch.from_numpy(dists).cuda(), k, greater)
    torch.cuda.synchronize()
    assert np.array_equal(got_i.cpu().numpy(), want_i)
    assert np.array_equal(got_d.cpu().numpy() + 0.0, want_d + 0.0)   # +0.0: -0 and +0 compare equal


def test_concurrent_host_threads_get_their_own_streams(dataset, ref_outputs):
    """"threadpool -> CUDA streams": several host threads search one index at once (the reference allows this with
    external scratch, index/vamana/index.h:455-470); every call checks out its own stream + scratch."""
    import threading
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    from scalablevectorsearch_b200 import SearchBufferConfig
    index.search_parameters.buffer_config = SearchBufferConfig(22, 23)
    q = np.tile(dataset.queries[100:], (8, 1))
    results, errors = {}, []

    def work(i):
        try:
            for _ in range(4):
                results[i] = index.search(q, 10)
        except Exception as e:   # noqa: BLE001
            errors.append(e)
    threads = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    for i in range(4):
        for b in range(8):
            assert_same((results[i][0][900 * b:900 * (b + 1)], results[i][1][900 * b:900 * (b + 1)]),
                        ref_outputs["l2_f32_f32_w22_c23_ids"], ref_outputs["l2_f32_f32_w22_c23_dists"], f"thread {i}")
    assert index.get_option("streams") >= 2


def test_cancellation_predicate(dataset, ref_outputs):
    """`cancel` (index/vamana/index.h:568, polled at greedy_search.h:155 / extensions.h:579): a predicate that is
    already true returns before any work; one that never fires leaves the results untouched; one that fires while
    the batch runs makes the call return early (rows of unfinished queries are unspecified)."""
    import time
    from scalablevectorsearch_b200 import SearchBufferConfig
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    index.search_parameters.buffer_config = SearchBufferConfig(22, 23)
    got = index.search(dataset.queries[100:], 10, cancel=lambda: False)
    assert_same(got, ref_outputs["l2_f32_f32_w22_c23_ids"], ref_outputs["l2_f32_f32_w22_c23_dists"], "cancel never")
    ids, _ = index.search(dataset.queries[100:], 10, cancel=lambda: True)
    assert ids.shape == (900, 10)
    # a long batch (large window, many queries): cancel after the first poll, compare with the uncancelled time
    index.search_parameters.buffer_config = SearchBufferConfig(400, 400)
    q = np.tile(dataset.queries, (300, 1))
    index.search(q, 10)   # (first call of this size: scratch allocation)
    index.search(q, 10)
    full_ms = index.last_kernel_ms()
    calls = []

    def fire():
        calls.append(1)
        return len(calls) > 2
    index.search(q, 10, cancel=fire)
    cancelled_ms = index.last_kernel_ms()
    assert len(calls) > 2
    # the kernel stops at the next hop / query boundary and runs a fraction of the uncancelled time (`full_ms`: the
    # last piece of the batch, which spans the whole run -- without a predicate a host batch is cut into pieces whose
    # copies overlap the kernels).  Wall time is no measure here: the pageable copies of 300k queries dominate it.
    assert cancelled_ms < 0.5 * full_ms, (cancelled_ms, full_ms)


def test_sharded_index_in_one_process_matches_reference_per_shard_plus_merge(dataset, oracle):
    """svsb200_search_sharded (mode B, single process): two shards on the same device here (the multi-GPU form
    differs only in where the shards live) == oracle per shard + TotalOrder merge."""
    from scalablevectorsearch_b200 import SearchBufferConfig, ShardedVamana
    from scalablevectorsearch_b200.multi_gpu import merge_topk_reference_order
    rng = np.random.default_rng(5)
    x = dataset.data
    n = x.shape[0]
    cuts = [0, 3300, 7100, n]
    shards, parts = [], []
    q = dataset.queries[:128]
    for a, b in zip(cuts[:-1], cuts[1:]):
        g = knn_graph(x[a:b], 24, rng)
        sh = make_index(x[a:b], g, 5, "l2")
        shards.append(sh)
        wi, wd = oracle.index(x[a:b], g, 5, "l2").search(q, 10, 32, 48)
        parts.append((wi.astype(np.int64) + a, wd))
    sv = ShardedVamana(shards, cuts[:-1])
    sv.search_parameters.buffer_config = SearchBufferConfig(32, 48)
    ids, dists = sv.search(q, 10)
    want_i, want_d = merge_topk_reference_order(np.stack([p[0] for p in parts]), np.stack([p[1] for p in parts]), 10, False)
    assert np.array_equal(ids.astype(np.int64), want_i) and np.array_equal(bits(dists), bits(want_d))


def test_filtered_and_range_search(dataset, oracle):
    """The runtime ABI's filtered / range searches (vamana_index.h:75-92) with the filter evaluated on the device:
    checked against the oracle's plain search results post-processed on the host (members in result order; results
    inside the radius)."""
    from scalablevectorsearch_b200 import SearchBufferConfig
    index = make_index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    index.search_parameters.buffer_config = SearchBufferConfig(64)
    want = oracle.index(dataset.data, dataset.graph, dataset.entry_point, "l2")
    q = dataset.queries[:100]
    rng = np.random.default_rng(0)
    allowed = rng.random(dataset.data.shape[0]) < 0.3
    ids, dists, found = index.search_filtered(q, 10, allowed)
    assert np.all(found == 10)
    assert np.all(allowed[ids.astype(np.int64)])
    assert np.all(np.diff(dists, axis=1) >= 0)
    # the first 10 members of the oracle's result list of the same length (64 first; the whole batch is re-run with a
    # 256-entry list when any query found fewer than 10 members in it)
    w64 = want.search(q, 64, 64, 64)
    w256 = want.search(q, 256, 256, 256)
    grown = any(int(allowed[w64[0][i].astype(np.int64)].sum()) < 10 for i in range(len(q)))
    wi, wd = w256 if grown else w64
    for i in range(len(q)):
        keep = [j for j in range(wi.shape[1]) if allowed[int(wi[i, j])]][:10]
        assert np.array_equal(ids[i], wi[i, keep]) and np.array_equal(bits(dists[i]), bits(wd[i, keep])), i
    wi, wd = w256
    # nothing allowed -> empty rows, padded
    ids0, d0, f0 = index.search_filtered(q[:5], 3, np.zeros(dataset.data.shape[0], dtype=bool))
    assert np.all(f0 == 0) and np.all(ids0 == np.uint64(0xFFFFFFFFFFFFFFFF)) and np.all(np.isposinf(d0))
    # range search: everything closer than the 20th-nearest distance of query 0
    radius = float(wd[0, 20])
    res = index.range_search(q[:8], radius)
    for i, (ri, rd) in enumerate(res):
        assert np.all(rd < radius) and np.all(np.diff(rd) >= 0)
        assert len(ri) >= int(np.sum(wd[i, :50] < radius)) - 1


def test_runtime_abi_demo_program(tmp_path):
    """A C++ program written against the reference's runtime header only (svs::runtime::v0::VamanaIndex: build / add /
    search / IDFilter / range_search / get_distance), linked with libsvsb200_runtime.so instead of libsvs_runtime."""
    import os
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "scalablevectorsearch_b200", "cpp", "_build", "runtime_demo")
    if not os.path.exists(exe):
        pytest.skip("runtime_demo not built (needs the reference's runtime headers at build time)")
    rng = np.random.default_rng(4)
    n, dim, nq, k = 5000, 32, 16, 5
    x = rng.standard_normal((n, dim)).astype(np.float32)
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    x.tofile(tmp_path / "x.f32")
    q.tofile(tmp_path / "q.f32")
    out = subprocess.run([exe, str(tmp_path / "x.f32"), str(n), str(dim), str(tmp_path / "q.f32"), str(nq)],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    rows = {"plain": [], "even": [], "range": [], "get_distance": []}
    for line in out.stdout.splitlines():
        tag, label, dist = line.split()
        rows[tag].append((int(label), float(dist)))
    d = ((q[:, None, :] - x[None, :, :]) ** 2).sum(-1)
    gt = np.argsort(d, axis=1)[:, :k]
    plain = np.array([r[0] for r in rows["plain"]]).reshape(nq, k)
    recall = np.mean([len(set(plain[i]) & set(gt[i])) for i in range(nq)]) / k
    assert recall > 0.9, recall
    even = np.array([r[0] for r in rows["even"]]).reshape(nq, k)
    assert np.all(even % 2 == 0)
    gt_even = np.argsort(np.where(np.arange(n)[None, :] % 2 == 0, d, np.inf), axis=1)[:, :k]
    assert np.mean([len(set(even[i]) & set(gt_even[i])) for i in range(nq)]) / k > 0.85
    radius = rows["even"][k - 1][1]  # the demo passes the filtered search's k-th distance of query 0
    assert rows["range"] and all(dist < radius for _, dist in rows["range"])
    label, dist = rows["get_distance"][0]
    assert label == rows["even"][0][0] and dist == pytest.approx(rows["even"][0][1], rel=1e-6)   # l, d hold the filtered search


@pytest.mark.parametrize("metric", ["l2", "cosine"])
def test_several_entry_points(dataset, oracle, metric):
    """EntryPointInitializer pushes every entry point (greedy_search.h:62-94; index.h:304-312 holds a vector)."""
    eps = [9426, 17, 4242, 9999, 5]
    index = make_index(dataset.data, dataset.graph, eps[0], metric)
    index.set_entry_points(eps)
    want = oracle.index(dataset.data, dataset.graph, eps[0], metric)
    want.set_entry_points(eps)
    q = dataset.queries[:128]
    for window, cap in ((3, 3), (20, 33), (64, 64)):
        wi, wd = want.search(q, 3 if cap < 10 else 10, window, cap)
        for generic in (0, 1):
            index.set_option("generic_kernel", generic)
            got = search(index, q, 3 if cap < 10 else 10, window, cap)
            assert_same(got, wi, wd, f"{metric} eps w{window} generic{generic}")
