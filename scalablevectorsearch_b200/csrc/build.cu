// build.cu -- host side of the GPU Vamana graph builder (SURVEY.md §8 f1) + its small helper kernels.
// Replaces index::vamana::auto_build / VamanaBuilder::construct (index/vamana/index.h:404-440,968-994,
// vamana_build.h:221-310) for float32 / float16 data with L2 or inner-product distance.
#include "build_kernels.cuh"

#include <vector>

namespace svsb200 {

// add_reverse_edges, first half (vamana_build.h:484-501): one thread per new edge v -> u.
__global__ void reverse_insert_kernel(uint32_t first, uint32_t count, uint32_t* __restrict__ graph, uint32_t* __restrict__ deg,
                                      uint32_t gstride, uint32_t max_degree, int* __restrict__ head, int* __restrict__ next,
                                      uint32_t* __restrict__ pair_v, uint32_t* __restrict__ pair_count,
                                      uint32_t* __restrict__ touched, uint32_t* __restrict__ touched_count,
                                      uint32_t pair_cap) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t i = idx / max_degree, j = idx % max_degree;
    if (i >= count) return;
    const uint32_t v = first + i;
    if (j >= min(deg[v], max_degree)) return;
    const uint32_t u = graph[size_t(v) * gstride + j];
    if (u == kNoNeighbor || u == v) return;
    // graph.add_edge(u, v) keeps rows free of repeats (core/graph/graph.h:211-260)
    uint32_t* urow = graph + size_t(u) * gstride;
    const uint32_t du = min(deg[u], max_degree);
    for (uint32_t z = 0; z < du; ++z)
        if (urow[z] == v) return;
    const uint32_t slot = atomicAdd(deg + u, 1u);
    if (slot < max_degree) {
        urow[slot] = v;
        return;
    }
    atomicSub(deg + u, 1u);
    const uint32_t e = atomicAdd(pair_count, 1u);
    if (e >= pair_cap) return;
    pair_v[e] = v;
    const int old = atomicExch(head + u, int(e));
    next[e] = old;
    if (old < 0) touched[atomicAdd(touched_count, 1u)] = u;
}

__global__ void reset_heads_kernel(const uint32_t* __restrict__ touched, const uint32_t* __restrict__ touched_count,
                                   int* __restrict__ head) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < *touched_count) head[touched[i]] = -1;
}

// ---- medoid (core/medioid.h:232-330): mean in double, then the row closest to it in double ----
template <int ROWT>
__global__ void column_sum_kernel(const char* __restrict__ vectors, uint32_t n, uint32_t dim, uint32_t row_stride,
                                  double* __restrict__ sums) {
    const uint32_t rows_per_block = 256;
    const uint32_t r0 = blockIdx.x * rows_per_block;
    for (uint32_t d = threadIdx.x; d < dim; d += blockDim.x) {
        double acc = 0.0;
        for (uint32_t r = r0; r < min(n, r0 + rows_per_block); ++r) {
            const char* row = vectors + size_t(r) * row_stride;
            if constexpr (ROWT == SVSB200_F32) acc += double(reinterpret_cast<const float*>(row)[d]);
            else acc += double(__half2float(reinterpret_cast<const __half*>(row)[d]));
        }
        atomicAdd(sums + d, acc);
    }
}

template <int ROWT>
__global__ void medoid_distance_kernel(const char* __restrict__ vectors, uint32_t n, uint32_t dim, uint32_t row_stride,
                                       const double* __restrict__ sums, double* __restrict__ best_d,
                                       uint32_t* __restrict__ best_i) {
    // one warp per row; block-level argmin, one (distance, id) pair per block
    __shared__ double sd[8];
    __shared__ uint32_t si[8];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t r = blockIdx.x * 8 + warp;
    double acc = 0.0;
    if (r < n) {
        const char* row = vectors + size_t(r) * row_stride;
        for (uint32_t d = lane; d < dim; d += 32) {
            double x;
            if constexpr (ROWT == SVSB200_F32) x = double(reinterpret_cast<const float*>(row)[d]);
            else x = double(__half2float(reinterpret_cast<const __half*>(row)[d]));
            const double diff = sums[d] / double(n) - x;
            acc += diff * diff;
        }
    }
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
    if (lane == 0) {
        sd[warp] = r < n ? acc : 1e300;
        si[warp] = r;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double bd = sd[0];
        uint32_t bi = si[0];
        for (int w2 = 1; w2 < 8; ++w2)
            if (sd[w2] < bd) {
                bd = sd[w2];
                bi = si[w2];
            }
        best_d[blockIdx.x] = bd;
        best_i[blockIdx.x] = bi;
    }
}

// neighbours-first device rows -> the reference's in-memory layout (degree first, core/graph/graph.h:103-114)
__global__ void export_graph_kernel(const uint32_t* __restrict__ graph, const uint32_t* __restrict__ deg, uint32_t n,
                                    uint32_t gstride, uint32_t max_degree, uint32_t* __restrict__ out) {
    const uint32_t row = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const uint32_t lane = threadIdx.x & 31;
    if (row >= n) return;
    const uint32_t d = min(deg[row], max_degree);
    uint32_t* o = out + size_t(row) * (max_degree + 1);
    if (lane == 0) o[0] = d;
    for (uint32_t j = lane; j < max_degree; j += 32) o[1 + j] = j < d ? graph[size_t(row) * gstride + j] : 0u;
}

// batch rows [first, first+count) as prepared fp32 queries (exact conversion, zero padding)
template <int ROWT>
__global__ void batch_queries_kernel(const char* __restrict__ vectors, uint32_t row_stride, uint32_t dim, uint32_t qstride,
                                     uint32_t first, uint32_t count, float* __restrict__ qf, float* __restrict__ qaux) {
    const uint32_t q = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const uint32_t lane = threadIdx.x & 31;
    if (q >= count) return;
    const char* row = vectors + size_t(first + q) * row_stride;
    float sq = 0.f;
    for (uint32_t i = lane; i < qstride; i += 32) {
        float v = 0.f;
        if (i < dim) {
            if constexpr (ROWT == SVSB200_F32) v = reinterpret_cast<const float*>(row)[i];
            else v = __half2float(reinterpret_cast<const __half*>(row)[i]);
        }
        qf[size_t(q) * qstride + i] = v;
        sq = fmaf(v, v, sq);
    }
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xFFFFFFFFu, sq, o);
    if (lane == 0) {   // {a_norm, unused}: the cosine query norm (cosine.h:117-119)
        qaux[2 * size_t(q)] = sqrtf(sq);
        qaux[2 * size_t(q) + 1] = 0.f;
    }
}

__global__ void fill_u32_kernel(uint32_t* p, size_t n, uint32_t v) {
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace svsb200

using namespace svsb200;

extern "C" int svsb200_build_vamana(const void* vectors, int dtype, size_t n, size_t dim, size_t row_stride_bytes, int metric,
                                    float alpha, size_t graph_max_degree, size_t window_size,
                                    size_t max_candidate_pool_size, size_t prune_to, int device, uint32_t* graph_rows_out,
                                    uint32_t* entry_point_out) {
    if (!vectors || !graph_rows_out || !entry_point_out) return set_error("svsb200_build_vamana: NULL argument");
    if (dtype != SVSB200_F32 && dtype != SVSB200_F16) return set_error("svsb200_build_vamana: float32 / float16 data only");
    if (metric < SVSB200_L2 || metric > SVSB200_COSINE) return set_error("svsb200_build_vamana: bad metric");
    if (n < 2 || dim == 0 || n >= (size_t(1) << 31)) return set_error("svsb200_build_vamana: bad shape");
    if (graph_max_degree == 0 || graph_max_degree > 32u * kFastMaxGW) return set_error("svsb200_build_vamana: graph_max_degree must be in [1, 128]");
    if (window_size == 0) return set_error("svsb200_build_vamana: window_size must be positive");
    // verify_and_set_default_index_parameters (index/vamana/index.h:1079-1110)
    if (max_candidate_pool_size == 0) max_candidate_pool_size = 3 * window_size;
    if (prune_to == 0) prune_to = graph_max_degree >= 16 ? graph_max_degree - 4 : graph_max_degree;
    if (prune_to > graph_max_degree) return set_error("svsb200_build_vamana: prune_to must be <= graph_max_degree");
    if (alpha == 0.f) alpha = metric == SVSB200_L2 ? 1.2f : 0.95f;
    if (metric == SVSB200_L2 ? alpha < 1.0f : alpha > 1.0f) return set_error("svsb200_build_vamana: alpha on the wrong side of 1 for this metric");
    const uint32_t R = uint32_t(graph_max_degree);
    const uint32_t gstride = gstride_for(R);
    const uint32_t hist_cap = kPoolMax - gstride;
    if (window_size + 32 > hist_cap) return set_error("svsb200_build_vamana: window_size too large for the candidate pool");
    const int ndev = svsb200_device_count();
    if (ndev == 0) return set_error("svsb200_build_vamana: no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return set_error("svsb200_build_vamana: bad device ordinal");
    cudaDeviceProp prop;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess)
        return set_error("svsb200_build_vamana: cannot select the device");
    if (prop.major != 10 || prop.minor != 0) return set_error("svsb200_build_vamana: device is not sm_100");

    const size_t row_bytes = dim * esize(dtype);
    const size_t src_stride = row_stride_bytes ? row_stride_bytes : row_bytes;
    const uint32_t row_stride = row_stride_for(SVSB200_PLAIN, dtype, dim);
    const uint32_t qstride = qstride_for(dim);
    // batches (vamana_build.h:229-240)
    size_t num_batches = std::max<size_t>(40, (n + 4095) / 4096);
    if (num_batches > n) num_batches = n;
    const size_t batchsize = (n + num_batches - 1) / num_batches;
    const size_t pair_cap = batchsize * R;
    const int grid_sm = prop.multiProcessorCount;
    const unsigned nblk = unsigned((n + 7) / 8);   // blocks of the medoid search

    cudaStream_t stream = nullptr;
    CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    StreamOwner stream_owner(stream, cudaStreamDestroy);   // (declared first: destroyed after every buffer is freed)
    DeviceBuffer<char> d_vectors;
    DeviceBuffer<uint32_t> d_graph, d_deg, d_hist_count, d_pair_v, d_counts, d_touched, d_best_i, d_export;
    DeviceBuffer<int> d_head, d_next;
    DeviceBuffer<uint2> d_hist;
    DeviceBuffer<float> d_qf, d_qaux;
    DeviceBuffer<double> d_sums, d_best_d;
    DeviceBuffer<unsigned int> d_work;
    CUDA_TRY(d_vectors.ensure(n * size_t(row_stride)));
    CUDA_TRY(cudaMemset(d_vectors.ptr, 0, n * size_t(row_stride)));
    CUDA_TRY(cudaMemcpy2D(d_vectors.ptr, row_stride, vectors, src_stride, row_bytes, n, cudaMemcpyHostToDevice));
    CUDA_TRY(d_graph.ensure(n * size_t(gstride)));
    CUDA_TRY(d_deg.ensure(n));
    CUDA_TRY(cudaMemset(d_deg.ptr, 0, n * 4));
    CUDA_TRY(d_head.ensure(n));
    CUDA_TRY(cudaMemset(d_head.ptr, 0xFF, n * 4));
    CUDA_TRY(d_next.ensure(pair_cap));
    CUDA_TRY(d_pair_v.ensure(pair_cap));
    CUDA_TRY(d_touched.ensure(pair_cap));
    CUDA_TRY(d_counts.ensure(2));
    CUDA_TRY(d_hist.ensure(batchsize * size_t(hist_cap)));
    CUDA_TRY(d_hist_count.ensure(batchsize));
    CUDA_TRY(d_qf.ensure(batchsize * size_t(qstride)));
    CUDA_TRY(d_qaux.ensure(batchsize * 2));
    CUDA_TRY(cudaMemset(d_qaux.ptr, 0, batchsize * 2 * 4));
    CUDA_TRY(d_work.ensure(1));
    CUDA_TRY(d_sums.ensure(dim));
    CUDA_TRY(cudaMemset(d_sums.ptr, 0, dim * 8));
    {
        const size_t cnt = n * size_t(gstride);
        fill_u32_kernel<<<unsigned((cnt + 255) / 256), 256, 0, stream>>>(d_graph.ptr, cnt, kNoNeighbor);
        count_launch();
    }
    // ---- entry point = medoid (index.h:986-990, core/medioid.h:292-330) ----
    uint32_t entry_point = 0;
    {
        CUDA_TRY(d_best_d.ensure(nblk));
        CUDA_TRY(d_best_i.ensure(nblk));
        if (dtype == SVSB200_F32) {
            column_sum_kernel<SVSB200_F32><<<unsigned((n + 255) / 256), 128, 0, stream>>>(d_vectors.ptr, uint32_t(n), uint32_t(dim), row_stride, d_sums.ptr);
            medoid_distance_kernel<SVSB200_F32><<<nblk, 256, 0, stream>>>(d_vectors.ptr, uint32_t(n), uint32_t(dim), row_stride, d_sums.ptr, d_best_d.ptr, d_best_i.ptr);
        } else {
            column_sum_kernel<SVSB200_F16><<<unsigned((n + 255) / 256), 128, 0, stream>>>(d_vectors.ptr, uint32_t(n), uint32_t(dim), row_stride, d_sums.ptr);
            medoid_distance_kernel<SVSB200_F16><<<nblk, 256, 0, stream>>>(d_vectors.ptr, uint32_t(n), uint32_t(dim), row_stride, d_sums.ptr, d_best_d.ptr, d_best_i.ptr);
        }
        count_launch();
        count_launch();
        CUDA_TRY(cudaGetLastError());
        std::vector<double> bd(nblk);
        std::vector<uint32_t> bi(nblk);
        CUDA_TRY(cudaMemcpyAsync(bd.data(), d_best_d.ptr, size_t(nblk) * 8, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaMemcpyAsync(bi.data(), d_best_i.ptr, size_t(nblk) * 4, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        size_t best = 0;
        for (size_t b = 1; b < nblk; ++b)
            if (bd[b] < bd[best]) best = b;
        entry_point = bi[best];
    }

    SearchParams p{};
    p.vectors = d_vectors.ptr;
    p.graph = d_graph.ptr;
    p.ref_degree = nullptr;
    p.n = uint32_t(n);
    p.dim = uint32_t(dim);
    p.row_stride = row_stride;
    p.gstride = gstride;
    p.entry_point = entry_point;
    p.greater = metric != SVSB200_L2;
    p.scale = 1.f;
    p.qf = d_qf.ptr;
    p.qcodes = nullptr;
    p.qaux = d_qaux.ptr;
    p.qstride = qstride;
    p.k = 0;
    p.window = uint32_t(window_size);
    p.capacity = uint32_t(window_size);
    p.cap_pad = uint32_t(round_up(window_size, 32));
    p.deg_pad = gstride;
    p.id_bytes = 4;
    p.work_counter = d_work.ptr;
    p.hist = d_hist.ptr;
    p.hist_count = d_hist_count.ptr;
    p.hist_cap = hist_cap;
    // visited filter of the lean kernel at its default size, grown as n needs for exact tags
    const LeanFilterPlan filter = lean_filter_plan(n, dim, window_size, p.deg_pad, 2048);
    p.filter_slots = filter.slots;
    p.filter_shift = filter.shift;
    p.filter_tag16 = 1;
    LaunchConfig cfg{};
    cfg.warps_per_cta = 1;
    cfg.smem_bytes = filter.smem_bytes;
    cfg.stream = stream;
    cfg.grid = -grid_sm;
    if (cfg.smem_bytes > 227 * 1024) return set_error("svsb200_build_vamana: window_size too large for shared memory");
    const int op = metric == SVSB200_L2 ? OP_L2F : metric == SVSB200_IP ? OP_IPF : OP_COSF;

    BuildParams bp{};
    bp.hist = d_hist.ptr;
    bp.hist_count = d_hist_count.ptr;
    bp.hist_cap = hist_cap;
    bp.head = d_head.ptr;
    bp.next = d_next.ptr;
    bp.pair_v = d_pair_v.ptr;
    bp.graph = d_graph.ptr;
    bp.deg = d_deg.ptr;
    bp.gstride = gstride;
    bp.max_degree = R;
    bp.max_candidates = uint32_t(std::min<size_t>(max_candidate_pool_size, kPoolMax));
    bp.iterative = metric != SVSB200_L2;
    bp.work_counter = d_work.ptr;
    bp.count_ptr = d_counts.ptr + 1;
    bp.nodes = d_touched.ptr;
    const int prune_grid = grid_sm * 16;

    // ---- two passes (index.h:436-439): reverse pruning with alpha 1, then with the configured alpha ----
    for (int pass = 0; pass < 2; ++pass) {
        const float reverse_alpha = pass == 0 ? 1.0f : alpha;
        for (size_t b = 0; b < num_batches; ++b) {
            const size_t start = std::min(n, batchsize * b), stop = std::min(n, batchsize * (b + 1));
            if (stop == start) continue;
            const uint32_t B = uint32_t(stop - start);
            // 1. generate_neighbors: search ...
            if (dtype == SVSB200_F32)
                batch_queries_kernel<SVSB200_F32><<<(B + 7) / 8, 256, 0, stream>>>(d_vectors.ptr, row_stride, uint32_t(dim), qstride, uint32_t(start), B, d_qf.ptr, d_qaux.ptr);
            else
                batch_queries_kernel<SVSB200_F16><<<(B + 7) / 8, 256, 0, stream>>>(d_vectors.ptr, row_stride, uint32_t(dim), qstride, uint32_t(start), B, d_qf.ptr, d_qaux.ptr);
            count_launch();
            CUDA_TRY(cudaMemsetAsync(d_work.ptr, 0, 4, stream));
            p.nq = B;
            CUDA_TRY(dtype == SVSB200_F32 ? launch_build_search<SVSB200_F32>(op, p, cfg) : launch_build_search<SVSB200_F16>(op, p, cfg));
            // ... pool + prune (always with the configured alpha, vamana_build.h:268-272)
            CUDA_TRY(cudaMemsetAsync(d_work.ptr, 0, 4, stream));
            bp.reverse = 0;
            bp.first = uint32_t(start);
            bp.count = B;
            bp.limit = R;
            bp.alpha = alpha;
            CUDA_TRY(dtype == SVSB200_F32 ? launch_build_prune_op<SVSB200_F32>(op, p, bp, std::min<int>(prune_grid, int(B)), stream)
                                          : launch_build_prune_op<SVSB200_F16>(op, p, bp, std::min<int>(prune_grid, int(B)), stream));
            // 2. add_reverse_edges
            CUDA_TRY(cudaMemsetAsync(d_counts.ptr, 0, 8, stream));
            reverse_insert_kernel<<<unsigned((size_t(B) * R + 255) / 256), 256, 0, stream>>>(
                uint32_t(start), B, d_graph.ptr, d_deg.ptr, gstride, R, d_head.ptr, d_next.ptr, d_pair_v.ptr, d_counts.ptr,
                d_touched.ptr, d_counts.ptr + 1, uint32_t(pair_cap));
            count_launch();
            CUDA_TRY(cudaMemsetAsync(d_work.ptr, 0, 4, stream));
            bp.reverse = 1;
            bp.limit = uint32_t(prune_to);
            bp.alpha = reverse_alpha;
            CUDA_TRY(dtype == SVSB200_F32 ? launch_build_prune_op<SVSB200_F32>(op, p, bp, prune_grid, stream)
                                          : launch_build_prune_op<SVSB200_F16>(op, p, bp, prune_grid, stream));
            reset_heads_kernel<<<unsigned((pair_cap + 255) / 256), 256, 0, stream>>>(d_touched.ptr, d_counts.ptr + 1, d_head.ptr);
            count_launch();
            CUDA_TRY(cudaGetLastError());
        }
    }
    // ---- export in the reference's layout ----
    CUDA_TRY(d_export.ensure(n * size_t(R + 1)));
    export_graph_kernel<<<unsigned((n + 7) / 8), 256, 0, stream>>>(d_graph.ptr, d_deg.ptr, uint32_t(n), gstride, R, d_export.ptr);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(graph_rows_out, d_export.ptr, n * size_t(R + 1) * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    *entry_point_out = entry_point;
    return 0;
}
