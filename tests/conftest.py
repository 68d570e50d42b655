import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")
    # The product library is built in-tree (git-ignored); compile it if this checkout has not been built yet
    # (nvcc cross-compiles sm_100a without a GPU).  Never a fallback: tests still go through libsvsb200.so.
    lib = os.path.join(ROOT, "scalablevectorsearch_b200", "libsvsb200.so")
    if not os.path.exists(lib) and os.path.exists("/usr/local/cuda/bin/nvcc"):
        import subprocess
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "scalablevectorsearch_b200", "csrc"), "-j", "6"],
                              stdout=subprocess.DEVNULL)


class Dataset:
    """The reference's data/test_dataset fixtures, from the committed tests/golden/test_dataset.npz."""

    def __init__(self):
        z = np.load(os.path.join(GOLDEN, "test_dataset.npz"))
        self.data = z["data"].astype(np.float32)       # 10000 x 128, integer valued
        self.queries = z["queries"].astype(np.float32)  # 1000 x 128
        self.graph = z["graph"]                         # uint32[10000][129], degree first
        self.entry_point = int(z["entry_point"])
        self.gt = {"l2": z["gt_l2"], "ip": z["gt_ip"], "cosine": z["gt_cosine"]}

    def variant(self, name):
        """(queries, data) for a '<qtype>_<dtype>' pair, as tests/golden/make_golden.py built them."""
        q, x = self.queries, self.data
        return {
            "f32_f32": (q, x),
            "f32_f16": (q, x.astype(np.float16)), "f16_f16": (q.astype(np.float16), x.astype(np.float16)),
            "f16_f32": (q.astype(np.float16), x), "f32_i8": (q, x.astype(np.int8)),
            "i8_i8": (q.astype(np.int8), x.astype(np.int8)), "f32_u8": (q, (x + 127).astype(np.uint8)),
            "u8_u8": ((q + 127).astype(np.uint8), (x + 127).astype(np.uint8)),
        }[name]


@pytest.fixture(scope="session")
def dataset():
    return Dataset()


@pytest.fixture(scope="session")
def ref_outputs():
    return np.load(os.path.join(GOLDEN, "ref_outputs.npz"))


@pytest.fixture(scope="session")
def ref_checks():
    """What the compiled reference computed for the oracle and graph-builder tests (tests/golden/make_golden.py)."""
    return np.load(os.path.join(GOLDEN, "ref_checks.npz"))


@pytest.fixture(scope="session")
def golden_recalls():
    return json.load(open(os.path.join(GOLDEN, "golden_recalls.json")))


@pytest.fixture(scope="session")
def oracle():
    from oracle.bindings import OracleLib
    import subprocess
    if not OracleLib.available():
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"])
    return OracleLib()


@pytest.fixture(scope="session")
def reflib():
    """The compiled reference, when it is present and this CPU runs its AVX-512 kernels."""
    from oracle.bindings import RefLib
    if not RefLib.available():
        pytest.skip("oracle/_ref/libsvsref.so not built (needs /root/reference)")
    try:
        lib = RefLib()
    except OSError as e:
        pytest.skip(f"libsvsref.so does not load here: {e}")
    if not lib.avx512():
        pytest.skip("host lacks AVX-512F: the reference would take its AVX2 expression tree")
    return lib


def recall_at_k(ids, gt, k=10):
    """k_recall_at_n with k == n (core/recall.h:48-59)."""
    hits = 0
    for row, truth in zip(ids[:, :k], gt[:, :k]):
        hits += len(set(row.tolist()) & set(truth.tolist()))
    return hits / (k * len(ids))


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def knn_graph(data, max_degree, rng, extra_random=4):
    """Small brute-force kNN graph + a few random long edges (degree-first reference layout)."""
    x = data.astype(np.float32)
    n = x.shape[0]
    sq = (x * x).sum(1)
    d = sq[:, None] + sq[None, :] - 2.0 * (x @ x.T)
    np.fill_diagonal(d, np.inf)
    graph = np.zeros((n, max_degree + 1), dtype=np.uint32)
    near = np.argsort(d, axis=1, kind="stable")[:, : max_degree - extra_random]
    for i in range(n):
        deg = int(rng.integers(max(1, max_degree // 2), max_degree + 1))
        nb = list(near[i][: max(1, deg - extra_random)])
        while len(nb) < deg:
            c = int(rng.integers(0, n))
            if c != i and c not in nb:
                nb.append(c)
        graph[i, 0] = len(nb)
        graph[i, 1:1 + len(nb)] = nb
    return graph
