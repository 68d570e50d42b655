"""GPU Vamana graph construction (svsb200_build_vamana) against the reference's own builder.

The reference's build result depends on thread timing, so its own tests compare recall, not graphs
(tests/integration/vamana/index_build.cpp:96,139-140: |recall - expected| < 0.005 between runs of the same builder).
Here: same data, same parameters, the graph from the GPU builder vs the graph from the reference's CPU builder
(its entry point, average degree and recall@10 under the bit-exact search, stored in tests/golden/ref_checks.npz);
recall@10 must agree within 0.01 and the graphs must have a similar density.  Structural checks: degrees within bounds, no self loops, no repeated neighbours, ids in range."""
import numpy as np
import pytest

from conftest import recall_at_k

pytestmark = pytest.mark.gpu


def _structural(graph, n, R):
    deg = graph[:, 0]
    assert deg.max() <= R and deg.min() >= 1
    for i in range(0, n, max(1, n // 500)):
        nb = graph[i, 1:1 + deg[i]]
        assert len(set(nb.tolist())) == len(nb) and i not in nb and nb.max() < n


def _recall(data, graph, ep, queries, gt, metric, window):
    from scalablevectorsearch_b200 import DistanceType, SearchBufferConfig, Vamana
    index = Vamana.from_arrays(data, graph, ep, {"l2": DistanceType.L2, "ip": DistanceType.MIP, "cosine": DistanceType.Cosine}[metric])
    index.search_parameters.buffer_config = SearchBufferConfig(window)
    ids, _ = index.search(queries, 10)
    return recall_at_k(ids, gt)


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
def test_build_on_reference_dataset_matches_reference_builder_recall(dataset, ref_checks, metric):
    """data/test_dataset (10k x 128), the reference's own build test shape (index_build.cpp: R=64... here R=32,
    window 64 to keep the CPU side quick)."""
    from scalablevectorsearch_b200 import DistanceType, VamanaBuildParameters, build_graph
    dist = {"l2": DistanceType.L2, "ip": DistanceType.MIP, "cosine": DistanceType.Cosine}[metric]
    alpha = 1.2 if metric == "l2" else 0.95
    params = VamanaBuildParameters(alpha=alpha, graph_max_degree=32, window_size=64)
    g_gpu, ep_gpu = build_graph(dataset.data, dist, params)
    _structural(g_gpu, dataset.data.shape[0], 32)
    ep_ref = int(ref_checks[f"build_{metric}_entry_point"])
    assert ep_gpu == ep_ref, "medoid entry point differs from the reference's"
    q, gt = dataset.queries, dataset.gt[metric]
    for window, r_ref in zip((10, 30), ref_checks[f"build_{metric}_recall_w10_w30"]):
        r_gpu = _recall(dataset.data, g_gpu, ep_gpu, q, gt, metric, window)
        assert r_gpu >= r_ref - 0.01, (metric, window, r_gpu, r_ref)
    d_gpu, d_ref = g_gpu[:, 0].mean(), float(ref_checks[f"build_{metric}_avg_degree"])
    assert 0.8 * d_ref <= d_gpu <= 1.25 * d_ref, (d_gpu, d_ref)


def test_build_synthetic_f16_and_index_build_api(ref_checks):
    """Clustered unit vectors (the bench's law), float16 storage, through Vamana.build; recall vs brute force."""
    from scalablevectorsearch_b200 import DistanceType, SearchBufferConfig, Vamana, VamanaBuildParameters
    from scalablevectorsearch_b200.synthetic import clustered_unit_vectors
    base, queries = clustered_unit_vectors(30_000, 500, 96)
    base16 = base.astype(np.float16)
    index = Vamana.build(VamanaBuildParameters(graph_max_degree=64, window_size=128), base16, DistanceType.L2)
    index.search_parameters.buffer_config = SearchBufferConfig(64)
    ids, _ = index.search(queries, 10)
    x = base16.astype(np.float32)
    d = (queries ** 2).sum(1)[:, None] + (x ** 2).sum(1)[None, :] - 2.0 * queries @ x.T
    gt = np.argsort(d, axis=1, kind="stable")[:, :10]
    # the reference's CPU builder (R 64, window 128, alpha 1.2) on the same data, searched at window 64
    r_gpu, r_ref = recall_at_k(ids, gt), float(ref_checks["build_synthetic_f16_recall_w64"])
    assert r_gpu >= r_ref - 0.01 and r_gpu > 0.9, (r_gpu, r_ref)
