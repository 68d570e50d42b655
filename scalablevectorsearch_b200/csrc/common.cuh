// common.cuh -- shared definitions for libsvsb200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>

#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <memory>
#include <string>

#include "../../include/svsb200.h"

namespace svsb200 {

constexpr uint32_t kNoNeighbor = 0xFFFFFFFFu;   // padding of adjacency rows in HBM
constexpr uint32_t kVisitedBit = 0x80000000u;   // SearchNeighbor::visited packed into the id
constexpr uint32_t kIdMask = 0x7FFFFFFFu;

// Internal row kinds of the search kernel: the four ABI element types plus LVQ-8 rows
// (uint8 codes followed by the per-vector {delta, lower} as two float16; DESIGN.md §10).
constexpr int ROW_LVQ8 = 4;

// Distance operator of the search kernel.
//   *F: the reference's fp32 expression tree (generic_simd_op, simd_utils.h:204-252)
//   *I: exact int32 arithmetic for (int8,int8)/(uint8,uint8) (L2VNNIOp/IPVNNIOp)
enum Op : int { OP_L2F = 0, OP_IPF = 1, OP_COSF = 2, OP_L2I = 3, OP_IPI = 4, OP_COSI = 5 };

// Everything the search kernel needs; passed by value (__grid_constant__).
struct SearchParams {
    // index
    const void* vectors;       // HBM, row-major, `row_stride` bytes apart (multiple of 16)
    const uint32_t* graph;     // HBM, uint32[n][gstride], neighbours then kNoNeighbor padding
    const uint16_t* ref_degree; // HBM, out-degree as the reference stores it (repeats included); counters only
    uint32_t n;
    uint32_t dim;
    uint32_t row_stride;
    uint32_t lvq_const_offset;  // LVQ-8: byte offset of {delta, lower} (2 x f16) inside a row
    uint32_t gstride;
    uint32_t entry_point;
    const uint32_t* entry_points;   // more than one entry point (index/vamana/index.h:304-312 holds a vector): device array
    uint32_t n_entry;               // 0 or 1: `entry_point` alone
    // distance post-processing
    int greater;               // comparator std::greater (IP / cosine): keys are negated
    int sq;                    // rows are scalar-quantised codes
    int lvq;                   // rows are LVQ-8 (mean-removed, per-vector delta/lower)
    // (scale_sq first: with scale and bias on one 8-byte boundary nvcc pairs their loads, and the search kernels'
    // register allocation shifts)
    float scale_sq, scale, bias;
    // prepared queries (output of prepare_queries)
    const float* qf;           // [nq][qstride] fp32 operands of the float tree
    const uint8_t* qcodes;     // [nq][qstride] int8/uint8 operands of the integer kernels
    const float* qaux;         // [nq][2]: {a_norm | offset, float(sum x*x)}
    uint32_t qstride;          // elements; multiple of 16
    uint32_t nq;
    // search buffer configuration
    uint32_t k, window, capacity;
    uint32_t cap_pad;          // capacity+1 rounded up to 32
    uint32_t deg_pad;          // gstride rounded up to 32
    uint32_t filter_slots;     // per-query exact visited filter (power of two, 0 = off)
    uint32_t filter_shift;     // tag = id >> filter_shift: log2(sets) = log2(filter_slots / 2) in tag16 mode,
                               // log2(filter_slots) (unused: full ids are stored) otherwise
    uint32_t filter_tag16;     // 1: two 16-bit tags per 32-bit set (exact while (n-1) >> filter_shift < 0xFFFF)
    // outputs
    void* out_ids;
    int id_bytes;
    uint64_t id_offset;        // added to every valid 64-bit output id (this index is a shard of a larger one)
    float* out_dists;
    // bookkeeping
    unsigned int* work_counter;  // dynamic query scheduler
    uint32_t* hops;              // optional per-query counters
    uint32_t* evals;
    uint32_t* fetched;           // rows actually read from HBM (after the visited filter)
    const int* cancel;           // optional device flag: non-zero stops the batch (polled per query and per hop)
    uint32_t exh_split;          // exhaustive scan: base rows are cut into this many ranges, one work item per (query, range)
    // graph builder only (HIST kernels): per query, every expanded node {key bits, id}
    uint2* hist;
    uint32_t* hist_count;
    uint32_t hist_cap;
};

struct LaunchConfig {
    int grid;
    int warps_per_cta;
    size_t smem_bytes;
    cudaStream_t stream;
};

// Per-warp shared-memory footprint of the search kernel (bytes), mirrored on the host.
__host__ __device__ inline size_t warp_smem_bytes(uint32_t qstride, uint32_t cap_pad, uint32_t deg_pad,
                                                  uint32_t filter_bytes) {
    // query (fp32 or bytes, reserve fp32) + buffer keys/ids + candidate keys/ids +
    // survivor keys/pos/ids/final-pos + visited filter
    // + two staged adjacency rows
    return size_t(qstride) * 4 + size_t(cap_pad) * 8 + size_t(deg_pad) * 8 + size_t(deg_pad) * 16 +
           size_t(filter_bytes) + size_t(deg_pad) * 8;
}

// Per-CTA (= per-warp = per-query) shared memory of the fast kernel, mirrored on the host.
__host__ __device__ inline size_t fast_smem_bytes(uint32_t qstride, uint32_t cap_pad, uint32_t deg_pad,
                                                  uint32_t filter_bytes) {
    // filter | query | buffer {key,id} | candidate keys | candidate ids
    return size_t((filter_bytes + 15u) & ~15u) + size_t(qstride) * 4 + size_t(cap_pad) * 8 + size_t(deg_pad) * 8;
}

constexpr int kFastMaxGW = 4;   // adjacency rows up to 128 neighbours (4 x 32) are register-staged

// One launcher per (row type, op); defined in search_<type>.cu.
template <int ROWT> cudaError_t launch_search(int op, const SearchParams& p, const LaunchConfig& cfg, int rows_in_flight);
// The lean one-warp-per-CTA form of the same search (search_fast.cuh); defined in fast_<type>.cu.
template <int ROWT> cudaError_t launch_search_fast(int op, const SearchParams& p, const LaunchConfig& cfg);
// Exhaustive scan with the same distance code (ground truth / flat search).
template <int ROWT> cudaError_t launch_search_exhaustive(int op, const SearchParams& p, const LaunchConfig& cfg);

// Tensor-core exhaustive search (flat.cu)
cudaError_t flat_tile_rows(int srct, const void* src, uint32_t row_stride, uint32_t n, uint32_t dim, uint32_t tile_rows,
                           float scale, int l2, void* dst_tiles, float* bias, float* norms, unsigned int* max_norm_bits,
                           cudaStream_t stream);
cudaError_t flat_gemm_topk(const void* a_tiles, const void* b_tiles, const float* b_bias, uint32_t KB, uint32_t ntiles,
                           uint32_t mtiles, uint32_t ctas, uint32_t share, uint32_t nlists, float key_scale, float* cand_key,
                           uint32_t* cand_id, uint32_t* progress, cudaStream_t stream);
struct SearchParams;
void flat_plan(uint32_t mtiles, uint32_t ntiles, uint32_t sm_count, uint32_t* ctas, uint32_t* share, uint32_t* nlists);
cudaError_t flat_rescore(int rowt, int op, const SearchParams& p, const float* cand_key, const uint32_t* cand_id, uint32_t nsplit,
                         uint32_t nq, uint32_t k, const float* qnorm, const unsigned int* xmax_bits, uint64_t* out_ids,
                         float* out_dists, uint32_t* unverified, uint32_t* n_unverified, cudaStream_t stream);
cudaError_t flat_move_rows(const void* src, void* dst, const uint32_t* idx, const uint32_t* count, uint32_t max_count,
                           uint32_t row_bytes, int scatter, cudaStream_t stream);
uint32_t flat_kc();

void count_launch();
int set_error(const std::string& msg);   // records the calling thread's svsb200_last_error(); returns 1

// A failed CUDA call becomes the calling thread's error, and the enclosing function returns 1.
#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t err__ = (expr);                                                            \
        if (err__ != cudaSuccess) {                                                            \
            return set_error(std::string(#expr) + ": " + cudaGetErrorString(err__));           \
        }                                                                                      \
    } while (0)

// Owns one device allocation.  The owner selects the allocation's device before the destructor runs.
template <typename T> struct DeviceBuffer {
    T* ptr = nullptr;
    size_t count = 0;
    DeviceBuffer() = default;
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    DeviceBuffer(DeviceBuffer&& o) noexcept : ptr(o.ptr), count(o.count) {
        o.ptr = nullptr;
        o.count = 0;
    }
    ~DeviceBuffer() { release(); }
    // Room for at least n elements; the old contents are not kept.
    cudaError_t ensure(size_t n) {
        if (n <= count) return cudaSuccess;
        release();   // (cudaFree synchronises the device: safe against work still using the old block)
        cudaError_t err = cudaMalloc(&ptr, n * sizeof(T));
        if (err == cudaSuccess) count = n;
        else ptr = nullptr;
        return err;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        count = 0;
    }
};

// Owns a stream: StreamOwner owner(stream, cudaStreamDestroy).
using StreamOwner = std::unique_ptr<CUstream_st, cudaError_t (*)(cudaStream_t)>;

inline size_t esize(int dtype) { return dtype == SVSB200_F32 ? 4 : dtype == SVSB200_F16 ? 2 : 1; }
inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

// ---- index layout in HBM, shared by the search library and the graph builder ----
// Bytes from one vector to the next: LVQ-8 rows use the ABI's stride, other rows are padded to 16 bytes.
inline uint32_t row_stride_for(int storage, int dtype, size_t dim) {
    return uint32_t(storage == SVSB200_LVQ8 ? svsb200_lvq8_row_stride(dim) : round_up(dim * esize(dtype), 16));
}
// Words from one adjacency row to the next.  Rows of up to 128 neighbours are padded to whole 32-word groups (one
// coalesced load per group and lane in the lean kernel, no per-lane bounds checks); wider rows stay 16-byte aligned.
inline uint32_t gstride_for(size_t max_degree) {
    return uint32_t(round_up(max_degree, max_degree <= 32u * kFastMaxGW ? 32 : 4));
}
// Elements from one prepared query to the next.
inline uint32_t qstride_for(size_t dim) { return uint32_t(round_up(dim, 16)); }

// Visited filter of the lean kernel: sets of eight 16-bit tags, `slots` of them (0 = off, else at least 64), doubled
// until every id >> shift fits below the 0xFFFF "empty" tag, so that the filter is exact.
struct LeanFilterPlan {
    uint32_t slots, shift;
    size_t smem_bytes;   // per CTA
};
inline LeanFilterPlan lean_filter_plan(size_t n, size_t dim, size_t capacity, uint32_t deg_pad, uint32_t slots) {
    if (slots && slots < 64) slots = 64;
    uint32_t shift = 0;
    while ((8u << shift) < slots) ++shift;   // log2(sets)
    while (slots && (uint64_t(n - 1) >> shift) >= 0xFFFFull && shift < 20) {
        ++shift;
        slots <<= 1;
    }
    return {slots, shift, fast_smem_bytes(qstride_for(dim), uint32_t(round_up(capacity, 32)), deg_pad, slots * 2u)};
}

}  // namespace svsb200
