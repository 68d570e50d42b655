"""Generate the committed golden fixtures under tests/golden/ (run in the authoring container).

Inputs : /root/reference/data/test_dataset (the reference's own 10k x 128 fixtures, prebuilt
         Vamana graph, ground truth) and oracle/_ref/libsvsref.so (the reference compiled
         from /root/reference by `make -C oracle ref`).
Outputs: test_dataset.npz   compact copy of the fixtures the parity tests need on the GPU box
         ref_outputs.npz    ids / distances / work counters the *reference itself* produces
         golden_recalls.json the 17 (window, capacity) -> recall@10 goldens of
                            data/test_dataset/reference/vamana_reference.toml (vamana_test_search)
         ref_checks.npz     the reference on random non-integer inputs and its CPU graph builder's results
                            (write_ref_checks)

    python tests/golden/make_golden.py
"""
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.bindings import RefLib  # noqa: E402
from scalablevectorsearch_b200 import io  # noqa: E402

SRC = "/root/reference/data/test_dataset"
OUT = os.path.dirname(os.path.abspath(__file__))


def parse_goldens(path):
    """Pull (distance, window, capacity, recall) of every vamana_test_search entry."""
    text = open(path).read()
    out = {}
    for block in text.split("[[vamana_test_search]]")[1:]:
        block = block.split("[[vamana_test_build]]")[0]
        dist = re.search(r"distance = '(\w+)'", block).group(1)
        entries = []
        for sub in block.split("[[vamana_test_search.config_and_recall]]")[1:]:
            recall = float(re.search(r"^\s*recall = ([0-9.eE+-]+)", sub, re.M).group(1))
            cap = int(re.search(r"search_buffer_capacity = (\d+)", sub).group(1))
            win = int(re.search(r"search_window_size = (\d+)", sub).group(1))
            k = int(re.search(r"num_neighbors = (\d+)", sub).group(1))
            nq = int(re.search(r"num_queries = (\d+)", sub).group(1))
            entries.append({"window": win, "capacity": cap, "recall": recall, "k": k, "num_queries": nq})
        out[{"L2": "l2", "MIP": "ip", "Cosine": "cosine"}[dist]] = entries
    return out


def main():
    ref = RefLib()
    assert ref.avx512(), "goldens must come from the AVX-512 expression tree"
    X = io.read_svs(f"{SRC}/data_f32.svs", np.float32)
    G = io.read_graph(f"{SRC}/graph_128.svs")
    Q = io.read_vecs(f"{SRC}/queries_f32.fvecs")
    assert np.array_equal(X, np.round(X)) and np.abs(X).max() <= 127
    assert np.array_equal(Q, np.round(Q)) and np.abs(Q).max() <= 127
    ep = int(re.search(r"entry_point = (\d+)", open(f"{SRC}/vamana_config.toml").read()).group(1))
    gts = {m: io.read_vecs(f"{SRC}/groundtruth_{f}.ivecs")[:, :10].astype(np.uint32)
           for m, f in (("l2", "euclidean"), ("ip", "mip"), ("cosine", "cosine"))}
    np.savez_compressed(f"{OUT}/test_dataset.npz", data=X.astype(np.int8), graph=G, queries=Q.astype(np.int8),
                        entry_point=np.uint32(ep), gt_l2=gts["l2"], gt_ip=gts["ip"], gt_cosine=gts["cosine"])

    goldens = parse_goldens(f"{SRC}/reference/vamana_reference.toml")
    json.dump(goldens, open(f"{OUT}/golden_recalls.json", "w"), indent=1)

    outs = {}
    threads = os.cpu_count() or 1
    # (a) the 17 golden configurations, f32 data / f32 queries, last 900 queries
    for metric, entries in goldens.items():
        idx = ref.index(X, G, ep, metric, threads=threads)
        for e in entries:
            ids, dists = idx.search(Q[100:], 10, e["window"], e["capacity"])
            tag = f"{metric}_f32_f32_w{e['window']}_c{e['capacity']}"
            outs[tag + "_ids"] = ids.astype(np.uint32)
            outs[tag + "_dists"] = dists
        hops, evals = idx.counts(Q[:64], 32, 48)
        outs[f"{metric}_counts_w32_c48_hops"] = hops.astype(np.uint32)
        outs[f"{metric}_counts_w32_c48_evals"] = evals.astype(np.uint32)
    # (b) every supported (query, data) element-type pair at one split-buffer configuration
    variants = {
        "f32_f16": (Q, X.astype(np.float16)), "f16_f16": (Q.astype(np.float16), X.astype(np.float16)),
        "f16_f32": (Q.astype(np.float16), X), "f32_i8": (Q, X.astype(np.int8)),
        "i8_i8": (Q.astype(np.int8), X.astype(np.int8)),
        "f32_u8": (Q, (X + 127).astype(np.uint8)),
        "u8_u8": ((Q + 127).astype(np.uint8), (X + 127).astype(np.uint8)),
    }
    for metric in goldens:
        for name, (q, x) in variants.items():
            idx = ref.index(x, G, ep, metric, threads=threads)
            ids, dists = idx.search(q[:256], 10, 24, 40)
            outs[f"{metric}_{name}_w24_c40_ids"] = ids.astype(np.uint32)
            outs[f"{metric}_{name}_w24_c40_dists"] = dists
        # (c) scalar quantisation: the reference compresses, we keep codes + scale/bias
        for code in (np.int8, np.uint8):
            idx, codes, scale, bias = ref.sq_index(X * np.float32(0.37) + np.float32(1.5), G, ep, metric, code,
                                                   threads=threads)
            cname = np.dtype(code).name
            if metric == "l2":
                outs[f"sq_{cname}_codes"] = codes
                outs[f"sq_{cname}_scale_bias"] = np.array([scale, bias], dtype=np.float32)
            for qn, q in (("f32", Q * np.float32(0.37) + np.float32(1.5)),
                          ("f16", (Q * np.float32(0.37) + np.float32(1.5)).astype(np.float16))):
                ids, dists = idx.search(q[:256], 10, 24, 40)
                outs[f"{metric}_sq_{cname}_{qn}_w24_c40_ids"] = ids.astype(np.uint32)
                outs[f"{metric}_sq_{cname}_{qn}_w24_c40_dists"] = dists
    np.savez_compressed(f"{OUT}/ref_outputs.npz", **outs)
    for f in ("test_dataset.npz", "ref_outputs.npz", "golden_recalls.json"):
        print(f, os.path.getsize(f"{OUT}/{f}") // 1024, "KiB")
    write_ref_checks(ref)


def write_ref_checks(ref):
    """ref_checks.npz: what the reference computes for tests/test_oracle_golden.py (distances and searches on
    random non-integer inputs, stored with them) and tests/test_gpu_build.py (its CPU builder's entry point, average
    degree and the recall@10 of its graphs, searched by the oracle, which is bit-identical to the GPU search)."""
    from oracle.bindings import OracleLib
    from scalablevectorsearch_b200.synthetic import clustered_unit_vectors
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import Dataset, knn_graph, recall_at_k

    out = {}
    rng = np.random.default_rng(11)
    for dim in (17, 96, 100, 768):
        q = rng.standard_normal(dim).astype(np.float32)
        x = rng.standard_normal((40, dim)).astype(np.float32)
        out[f"live_q_{dim}"], out[f"live_x_{dim}"] = q, x
        for metric in ("l2", "ip", "cosine"):
            for p, (qq, xx) in enumerate(((q, x), (q, x.astype(np.float16)), (q.astype(np.float16), x.astype(np.float16)))):
                out[f"live_dist_{dim}_{metric}_{p}"] = ref.distance_rows(metric, qq, xx)
    n, dim = 1200, 48
    x = rng.standard_normal((n, dim)).astype(np.float32)
    qs = rng.standard_normal((100, dim)).astype(np.float32)
    graph = knn_graph(x, 12, rng)
    out["live_x"], out["live_queries"], out["live_graph"] = x, qs, graph
    for metric in ("l2", "ip", "cosine"):
        ids, dists = ref.index(x, graph, 5, metric).search(qs, 5, 9, 14)
        out[f"live_{metric}_ids"], out[f"live_{metric}_dists"] = ids.astype(np.uint32), dists

    oracle, ds = OracleLib(), Dataset()
    for metric in ("l2", "ip", "cosine"):
        g, ep = ref.build(ds.data, metric, 32, 64, alpha=1.2 if metric == "l2" else 0.95, threads=4)
        idx = oracle.index(ds.data, g, ep, metric)
        out[f"build_{metric}_entry_point"] = np.uint32(ep)
        out[f"build_{metric}_avg_degree"] = np.float64(g[:, 0].mean())
        out[f"build_{metric}_recall_w10_w30"] = np.array(
            [recall_at_k(idx.search(ds.queries, 10, w, w)[0], ds.gt[metric]) for w in (10, 30)])
    base, queries = clustered_unit_vectors(30_000, 500, 96)
    base16 = base.astype(np.float16)
    xf = base16.astype(np.float32)
    d = (queries ** 2).sum(1)[:, None] + (xf ** 2).sum(1)[None, :] - 2.0 * queries @ xf.T
    gt = np.argsort(d, axis=1, kind="stable")[:, :10]
    g, ep = ref.build(base16, "l2", 64, 128, alpha=1.2, threads=8)
    out["build_synthetic_f16_recall_w64"] = np.float64(
        recall_at_k(oracle.index(base16, g, ep, "l2").search(queries, 10, 64, 64)[0], gt))
    np.savez_compressed(f"{OUT}/ref_checks.npz", **out)
    print("ref_checks.npz", os.path.getsize(f"{OUT}/ref_checks.npz") // 1024, "KiB")


if __name__ == "__main__":
    main()
