// svsb200.cu -- C ABI (include/svsb200.h) of the B200 Vamana search library: index upload to one or
// several GPUs, query preparation (the device-side maybe_fix_argument), launch plumbing, result gather.
//
// Host-side structure (the reference's thread pool -> CUDA streams, index/vamana/index.h:455-470,564-611):
//   * an index owns one Replica per device (graph + vectors in that device's HBM);
//   * every search call checks a Scratch (stream + prepared-query buffers + work counter + cancel flag) out
//     of the replica's pool, so concurrent host threads search concurrently on their own streams;
//   * a multi-replica index splits a batch with threads::balance (lib/threads/types.h:311-329), one slice per
//     device, results landing in disjoint rows of the caller's arrays (SURVEY.md 8e mode A);
//   * svsb200_search_sharded runs every query on every shard index and merges G*k -> k on one device with
//     the reference's TotalOrder (mode B); with NVLink peer access the shards' search kernels write their
//     rows straight into the merging device's buffer.
//
// No CPU fallback lives here: every entry point either runs CUDA kernels on an sm_100 device or fails.
#include "common.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <type_traits>
#include <vector>

#include <sys/stat.h>

namespace svsb200 {

static thread_local std::string g_error;
static std::atomic<uint64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static int fail(const std::string& msg) {
    g_error = msg;
    return 1;
}
int set_error(const std::string& msg) { return fail(msg); }
// Everything one in-flight search needs on one device: the analogue of the reference's per-thread scratch
// space (index/vamana/index.h:455-470).
struct Scratch {
    int device = 0;
    cudaStream_t stream = nullptr;   // own non-blocking stream (blocking API) or the caller's (device API)
    cudaStream_t ctl = nullptr;      // side stream that raises the cancel flag while `stream` is busy
    bool owns_stream = false;
    DeviceBuffer<unsigned char> q_raw, q_codes, ids;
    DeviceBuffer<float> q_f32, q_aux, dists;
    DeviceBuffer<uint32_t> hops, evals, fetched;
    DeviceBuffer<uint64_t> exh_ids;                    // exhaustive scan split over base ranges: per-range top-k
    DeviceBuffer<float> exh_dists;
    DeviceBuffer<unsigned char> flat_a, flat_q2;       // tensor-core flat search: query tiles, gathered queries
    DeviceBuffer<float> flat_qnorm, flat_ckey, flat_d2;
    DeviceBuffer<uint32_t> flat_cid, flat_unv;         // candidates, unverified list (+ its counter in slot 0)
    DeviceBuffer<uint32_t> flat_progress;              // per CTA of the flat GEMM: tiles started (keeps row groups in step)
    DeviceBuffer<uint64_t> flat_i2;
    DeviceBuffer<uint64_t> gather_ids, merged_ids;     // sharded search (on the merging device)
    DeviceBuffer<float> gather_dists, merged_dists;
    DeviceBuffer<unsigned int> d_counter;
    DeviceBuffer<int> d_cancel;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_done = nullptr;
    bool timed = false;
    bool poll_cancel = false;        // this search was given a cancellation predicate: the kernels poll the flag
    size_t counted_nq = 0;
    int last_kernel = 0;
    ~Scratch() {   // (the buffers are freed after this body, on the device it selects)
        cudaSetDevice(device);
        if (ev_start) cudaEventDestroy(ev_start);
        if (ev_stop) cudaEventDestroy(ev_stop);
        if (ev_done) cudaEventDestroy(ev_done);
        if (ctl) cudaStreamDestroy(ctl);
        if (owns_stream && stream) cudaStreamDestroy(stream);
    }
};

// One copy of the index in one device's HBM.
struct Replica {
    int device = 0;
    int sm_count = 0;
    DeviceBuffer<char> d_vectors;
    DeviceBuffer<uint32_t> d_graph;
    DeviceBuffer<uint16_t> d_ref_degree;
    DeviceBuffer<float> d_mean;          // LVQ-8: dataset mean
    DeviceBuffer<uint32_t> d_entry;      // entry points when there are several
    // tensor-core flat search: the base vectors as fp16 UMMA tiles + per-row bias, built on first use
    DeviceBuffer<char> flat_b;
    DeviceBuffer<float> flat_bias;
    DeviceBuffer<unsigned int> flat_xmax;
    std::mutex mu;
    std::vector<Scratch*> idle;                      // pool for the blocking API
    std::map<cudaStream_t, Scratch*> by_stream;      // one per caller stream for the enqueue-only API
    std::vector<std::unique_ptr<Scratch>> all;       // (declared last: destroyed before the arrays above)
    ~Replica() { cudaSetDevice(device); }
};

}  // namespace svsb200

using namespace svsb200;

struct svsb200_index {
    int dtype = 0, metric = 0, storage = 0;
    size_t n = 0, dim = 0, max_degree = 0;
    uint32_t row_stride = 0, gstride = 0, entry_point = 0;
    float scale = 1.f, bias = 0.f;
    uint32_t lvq_const_offset = 0;
    size_t device_bytes = 0;          // per replica
    uint64_t id_offset = 0;           // added to every 64-bit output id (shard of a larger index)
    uint32_t n_entry = 1;             // entry points (the first one is `entry_point`)
    long cfg_window = 0, cfg_capacity = 0, cfg_visited = 0;   // search parameters of the TOML an index was assembled from
    std::vector<std::unique_ptr<Replica>> reps;
    int counting = 0;
    // options
    long warps_per_cta = 0, ctas_per_sm = 0, rows_in_flight = 0, filter_slots = -1;
    long generic_kernel = 0;          // 1: force the generic (round-1) kernel instead of the lean one
    long host_chunks = 0;             // host-buffer searches: pieces per device whose copies overlap the kernels (0 = auto)
    std::mutex mu;
    Scratch* last = nullptr;          // scratch of the most recent search: counters, kernel time, kernel kind
};

namespace svsb200 {

// A new scratch set of the replica (null, with the error recorded, when it cannot be made).
static Scratch* new_scratch(Replica* rep, cudaStream_t caller_stream) {
    auto sc = std::make_unique<Scratch>();
    sc->device = rep->device;
    cudaError_t e = cudaSuccess;
    if (caller_stream) {
        sc->stream = caller_stream;
    } else {
        e = cudaStreamCreateWithFlags(&sc->stream, cudaStreamNonBlocking);
        sc->owns_stream = true;
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&sc->ctl, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = sc->d_counter.ensure(1);
    if (e == cudaSuccess) e = sc->d_cancel.ensure(1);
    if (e == cudaSuccess) e = cudaMemset(sc->d_cancel.ptr, 0, sizeof(int));
    if (e == cudaSuccess) e = cudaEventCreate(&sc->ev_start);
    if (e == cudaSuccess) e = cudaEventCreate(&sc->ev_stop);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sc->ev_done, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        fail(std::string("scratch allocation: ") + cudaGetErrorString(e));
        return nullptr;
    }
    Scratch* raw = sc.get();
    rep->all.push_back(std::move(sc));
    return raw;
}

// Enqueue-only API: the scratch bound to the caller's stream (work on one stream is ordered, so it is reusable).
static Scratch* scratch_for_stream(Replica* rep, cudaStream_t stream) {
    std::lock_guard<std::mutex> lock(rep->mu);
    auto it = rep->by_stream.find(stream);
    if (it != rep->by_stream.end()) return it->second;
    Scratch* sc = new_scratch(rep, stream);
    if (sc) rep->by_stream[stream] = sc;
    return sc;
}

// The scratch set of one blocking call.  With a caller stream it is the one bound to that stream; without, it is an
// idle one of the replica's pool (a new one if all are busy -- one per concurrent caller), which goes back to the pool
// when the lease ends.  take() also selects the replica's device.
struct ScratchLease {
    Scratch* sc = nullptr;
    Replica* pool = nullptr;   // set while `sc` is checked out of this replica's pool
    ScratchLease() = default;
    ScratchLease(ScratchLease&& o) noexcept : sc(o.sc), pool(o.pool) { o.pool = nullptr; }
    ~ScratchLease() {
        if (!pool) return;
        std::lock_guard<std::mutex> lock(pool->mu);
        pool->idle.push_back(sc);
    }
    int take(Replica* rep, cudaStream_t caller_stream) {
        CUDA_TRY(cudaSetDevice(rep->device));
        if (caller_stream) {
            sc = scratch_for_stream(rep, caller_stream);
        } else {
            std::lock_guard<std::mutex> lock(rep->mu);
            if (rep->idle.empty()) {
                sc = new_scratch(rep, nullptr);
            } else {
                sc = rep->idle.back();
                rep->idle.pop_back();
            }
            if (sc) pool = rep;
        }
        return sc ? 0 : 1;
    }
};

// The scratch set of an enqueue-only call: the one bound to the caller's stream (NULL: a stream the index keeps for
// that purpose) on the index's only device, which is selected.
static int device_api_scratch(const char* who, svsb200_index* ix, void* stream, Scratch** sc) {
    if (ix->reps.size() != 1) return fail(std::string(who) + ": the index must live on exactly one device");
    CUDA_TRY(cudaSetDevice(ix->reps[0]->device));
    *sc = scratch_for_stream(ix->reps[0].get(), static_cast<cudaStream_t>(stream));
    return *sc ? 0 : 1;
}

// threads::balance (lib/threads/types.h:311-329): contiguous ranges whose sizes differ by at most one.
static void balance(size_t n, size_t parts, size_t i, size_t* lo, size_t* hi) {
    const size_t base = n / parts, rem = n % parts;
    *lo = i * base + (i < rem ? i : rem);
    *hi = *lo + base + (i < rem ? 1 : 0);
}

}  // namespace svsb200

namespace svsb200 {

// ---------------------------------------------------------------------------------------
// Upload kernels
// ---------------------------------------------------------------------------------------

// Reference adjacency rows (degree first, core/graph/graph.h:103-114) -> HBM layout:
// neighbours first, kNoNeighbor padding, row length a multiple of 4 words so rows stay
// 16-byte aligned.  Repeated ids inside a row keep their first occurrence only: the
// reference's insert() rejects the later copy as a duplicate (search_buffer.h:380-391) or
// drops it off the end, so removing it up front cannot change any result.
__global__ void repack_graph_kernel(const uint32_t* __restrict__ src, size_t row_len, uint32_t n,
                                    uint32_t* __restrict__ dst, uint32_t gstride, uint16_t* __restrict__ ref_degree,
                                    int* __restrict__ bad) {
    const uint32_t row = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const uint32_t* in = src + size_t(row) * row_len;
    uint32_t* out = dst + size_t(row) * gstride;
    const uint32_t deg = in[0];
    if (deg > row_len - 1) {
        if (lane == 0) atomicExch(bad, 1);
        return;
    }
    if (lane == 0) ref_degree[row] = uint16_t(deg);
    uint32_t written = 0;
    for (uint32_t j0 = 0; j0 < deg; j0 += 32) {
        const uint32_t j = j0 + lane;
        uint32_t id = j < deg ? in[1 + j] : kNoNeighbor;
        bool keep = j < deg;
        if (keep && id >= n) {
            atomicExch(bad, 2);
            keep = false;
        }
        if (keep) {
            for (uint32_t i = 0; i < j; ++i) {
                if (in[1 + i] == id) {
                    keep = false;
                    break;
                }
            }
        }
        const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
        if (keep) out[written + __popc(m & ((1u << lane) - 1u))] = id;
        written += __popc(m);
    }
    for (uint32_t j = written + lane; j < gstride; j += 32) out[j] = kNoNeighbor;
}

// ---------------------------------------------------------------------------------------
// Query preparation == distance::maybe_fix_argument for the whole batch
// (concepts/distance.h:90-130), one warp per query.
// ---------------------------------------------------------------------------------------
enum PrepMode : int {
    PREP_FLOAT = 0,   // float tree: operands converted exactly like the SIMD loads
    PREP_INT = 1,     // exact integer kernels: raw int8/uint8 query
    PREP_SQ_L2 = 2,   // EuclideanCompressed::fix_argument  (scalar.h:75-82)
    PREP_SQ_IP = 3,   // InnerProductCompressed::fix_argument (scalar.h:123-131)
    PREP_SQ_COS = 4,  // CosineSimilarityCompressed::fix_argument (scalar.h:168-171)
    PREP_LVQ_L2 = 5,  // LVQ-8, L2: query with the dataset mean removed (own spec, DESIGN.md §10)
    PREP_LVQ_IP = 6,  // LVQ-8, IP: raw query + <q, mean>
};

// Float16 -> float the way non-SIMD reference code does it (lib/float16.h:45-52):
// subnormals flush to signed zero.
__device__ __forceinline__ float f16_scalar(uint16_t x) {
    if ((x & 0x7C00u) == 0) return __uint_as_float(uint32_t(x & 0x8000u) << 16);
    return __half2float(__ushort_as_half(x));
}

template <int QT> __device__ __forceinline__ float q_simd(const void* q, uint32_t i) {
    if constexpr (QT == SVSB200_F32) return static_cast<const float*>(q)[i];
    if constexpr (QT == SVSB200_F16) return __half2float(__ushort_as_half(static_cast<const uint16_t*>(q)[i]));
    if constexpr (QT == SVSB200_I8) return float(static_cast<const int8_t*>(q)[i]);
    return float(static_cast<const uint8_t*>(q)[i]);
}
template <int QT> __device__ __forceinline__ float q_scalar(const void* q, uint32_t i) {
    if constexpr (QT == SVSB200_F16) return f16_scalar(static_cast<const uint16_t*>(q)[i]);
    return q_simd<QT>(q, i);
}

template <int QT>
__global__ void prepare_queries_kernel(const void* __restrict__ queries, uint32_t nq, uint32_t dim, uint32_t qstride,
                                       int mode, int metric, int code_type, float scale, float bias,
                                       const float* __restrict__ mean, float* __restrict__ qf,
                                       uint8_t* __restrict__ qcodes, float* __restrict__ qaux) {
    const uint32_t q = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x & 31;
    if (q >= nq) return;
    constexpr size_t QES = QT == SVSB200_F32 ? 4 : QT == SVSB200_F16 ? 2 : 1;
    const void* src = static_cast<const char*>(queries) + size_t(q) * dim * QES;
    float* f = qf + size_t(q) * qstride;
    uint8_t* c = qcodes + size_t(q) * qstride;

    for (uint32_t i = lane; i < qstride; i += 32) {
        float fv = 0.f;
        uint8_t cv = 0;
        if (i < dim) {
            if (mode == PREP_FLOAT || mode == PREP_LVQ_IP) {
                fv = q_simd<QT>(src, i);
            } else if (mode == PREP_LVQ_L2) {
                fv = __fsub_rn(q_simd<QT>(src, i), mean[i]);
            } else if (mode == PREP_INT) {
                if constexpr (QT == SVSB200_I8 || QT == SVSB200_U8) cv = static_cast<const uint8_t*>(src)[i];
            } else if (mode == PREP_SQ_L2) {
                // detail::compress (scalar.h:38-42)
                const float lo = code_type == SVSB200_I8 ? -128.f : 0.f, hi = code_type == SVSB200_I8 ? 127.f : 255.f;
                float r = roundf(__fdiv_rn(__fsub_rn(q_scalar<QT>(src, i), bias), scale));
                r = fminf(fmaxf(r, lo), hi);
                cv = code_type == SVSB200_I8 ? uint8_t(int8_t(int(r))) : uint8_t(int(r));
            } else {
                fv = q_scalar<QT>(src, i);
            }
        }
        f[i] = fv;
        c[i] = cv;
    }
    __syncwarp();
    if (lane != 0) return;

    float aux0 = 0.f, aux1 = 0.f;
    if (mode == PREP_INT || mode == PREP_SQ_L2) {
        int xx = 0;
        const bool is_signed = (mode == PREP_INT) ? (QT == SVSB200_I8) : (code_type == SVSB200_I8);
        for (uint32_t i = 0; i < dim; ++i) {
            int v = is_signed ? int(int8_t(c[i])) : int(c[i]);
            xx += v * v;
        }
        aux1 = __int_as_float(xx);
    }
    const bool need_norm = (metric == SVSB200_COSINE) && (mode == PREP_FLOAT || mode == PREP_INT || mode == PREP_SQ_COS);
    if (need_norm) {
        // distance::norm (distance_core.h:45-66): sequential fp32 `accum += v * v`, sqrt.
        float acc = 0.f;
        for (uint32_t i = 0; i < dim; ++i) {
            float sq;
            if constexpr (QT == SVSB200_I8 || QT == SVSB200_U8) {
                int v = QT == SVSB200_I8 ? int(static_cast<const int8_t*>(src)[i]) : int(static_cast<const uint8_t*>(src)[i]);
                sq = float(v * v);
            } else {
                float v = q_scalar<QT>(src, i);
                sq = __fmul_rn(v, v);
            }
            acc = __fadd_rn(acc, sq);
        }
        aux0 = __fsqrt_rn(acc);
    } else if (mode == PREP_LVQ_IP) {
        float acc = 0.f;
        for (uint32_t i = 0; i < dim; ++i) acc = __fmaf_rn(f[i], mean[i], acc);
        aux0 = acc;
    } else if (mode == PREP_SQ_IP) {
        // std::reduce over the fp32 query (libstdc++: four at a time, then the tail).
        float acc = 0.f;
        uint32_t i = 0;
        for (; i + 4 <= dim; i += 4) {
            float v1 = __fadd_rn(f[i], f[i + 1]);
            float v2 = __fadd_rn(f[i + 2], f[i + 3]);
            acc = __fadd_rn(acc, __fadd_rn(v1, v2));
        }
        for (; i < dim; ++i) acc = __fadd_rn(acc, f[i]);
        aux0 = __fmul_rn(bias, acc);
    }
    qaux[2 * size_t(q)] = aux0;
    qaux[2 * size_t(q) + 1] = aux1;
}

// ---------------------------------------------------------------------------------------
// Cross-shard top-k merge with TotalOrder (lib/neighbor.h:143-155): distance, then id.
// ---------------------------------------------------------------------------------------
// One warp per query selects the k smallest (key, id) pairs among all nshards * k candidates by repeated
// "smallest entry greater than the previous output" -- a full TotalOrder sort of the candidates' prefix, so
// the result does not depend on how ties are ordered inside a shard's list (they come out of the search
// buffer in insertion order, not id order).  Padding entries (id = all-ones) are ignored.
__device__ __forceinline__ uint32_t total_order_key(float d, int greater) {
    float k = greater ? -d : d;
    k = __fadd_rn(k, 0.0f);                       // -0 == +0 under operator<
    const uint32_t u = __float_as_uint(k);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);   // monotone float -> uint
}
__global__ void merge_topk_kernel(const uint64_t* __restrict__ ids, const float* __restrict__ dists, uint32_t nshards,
                                  uint32_t nq, uint32_t k, int greater, uint64_t* __restrict__ out_ids,
                                  float* __restrict__ out_dists) {
    const uint32_t q = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x & 31;
    if (q >= nq) return;
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const uint32_t n = nshards * k;
    // (key, id) of the previous output; "nothing yet" sorts before everything
    bool have_last = false;
    uint32_t last_key = 0;
    uint64_t last_id = 0;
    for (uint32_t j = 0; j < k; ++j) {
        uint32_t best_key = 0xFFFFFFFFu;
        uint64_t best_id = ~uint64_t(0);
        float best_d = 0.f;
        bool found = false;
        for (uint32_t c = lane; c < n; c += 32) {
            const uint32_t sh = c / k, jj = c - sh * k;
            const size_t o = (size_t(sh) * nq + q) * k + jj;
            const uint64_t id = ids[o];
            if (id == ~uint64_t(0)) continue;
            const float d = dists[o];
            const uint32_t key = total_order_key(d, greater);
            if (have_last && (key < last_key || (key == last_key && id <= last_id))) continue;
            if (!found || key < best_key || (key == best_key && id < best_id)) {
                best_key = key;
                best_id = id;
                best_d = d;
                found = true;
            }
        }
        // warp argmin over (found, key, id)
        for (int off = 16; off; off >>= 1) {
            const uint32_t okey = __shfl_xor_sync(FULL, best_key, off);
            const uint64_t oid = __shfl_xor_sync(FULL, best_id, off);
            const float od = __shfl_xor_sync(FULL, best_d, off);
            const bool ofound = __shfl_xor_sync(FULL, int(found), off) != 0;
            if (ofound && (!found || okey < best_key || (okey == best_key && oid < best_id))) {
                best_key = okey;
                best_id = oid;
                best_d = od;
                found = true;
            }
        }
        if (lane == 0) {
            const size_t o = size_t(q) * k + j;
            out_ids[o] = found ? best_id : ~uint64_t(0);
            out_dists[o] = found ? best_d : (greater ? -INFINITY : INFINITY);
        }
        if (!found) {
            for (uint32_t r = j + 1 + lane; r < k; r += 32) {   // nothing left: pad the tail
                out_ids[size_t(q) * k + r] = ~uint64_t(0);
                out_dists[size_t(q) * k + r] = greater ? -INFINITY : INFINITY;
            }
            return;
        }
        have_last = true;
        last_key = best_key;
        last_id = best_id;
    }
}

static cudaError_t launch_merge_topk(const uint64_t* ids, const float* dists, size_t nshards, size_t nq, size_t k, int greater,
                                     uint64_t* out_ids, float* out_dists, cudaStream_t stream) {
    const unsigned warps = 4;
    merge_topk_kernel<<<unsigned((nq + warps - 1) / warps), warps * 32, 0, stream>>>(
        ids, dists, uint32_t(nshards), uint32_t(nq), uint32_t(k), greater, out_ids, out_dists);
    count_launch();
    return cudaGetLastError();
}

// LVQ-8 encoder (own specification, DESIGN.md §10), one warp per vector:
//   r_i = x_i - mean_i;  lower = min r, upper = max r;  delta = (upper - lower) / 255
//   {delta, lower} are stored as float16 (round to nearest even) and the codes are computed against
//   the *stored* constants:  c_i = clamp(rint((r_i - lower16) / delta16), 0, 255)   (0 when delta16 == 0)
// so that decode y_i = fma(delta16, c_i, lower16) is the nearest representable grid point.
__global__ void lvq8_compress_kernel(const float* __restrict__ data, uint32_t n, uint32_t dim,
                                     const float* __restrict__ mean, uint8_t* __restrict__ rows, uint32_t stride,
                                     uint32_t const_offset) {
    const uint32_t row = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const float* x = data + size_t(row) * dim;
    uint8_t* out = rows + size_t(row) * stride;
    float lo = INFINITY, hi = -INFINITY;
    for (uint32_t i = lane; i < dim; i += 32) {
        const float r = __fsub_rn(x[i], mean[i]);
        lo = fminf(lo, r);
        hi = fmaxf(hi, r);
    }
    for (int o = 16; o; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
    }
    const __half dh = __float2half_rn(__fdiv_rn(__fsub_rn(hi, lo), 255.0f));
    const __half lh = __float2half_rn(lo);
    const float d = __half2float(dh), l = __half2float(lh);
    for (uint32_t i = lane; i < stride; i += 32) {
        uint8_t c = 0;
        if (i < dim && d > 0.0f) {
            const float r = __fsub_rn(x[i], mean[i]);
            float q = rintf(__fdiv_rn(__fsub_rn(r, l), d));
            q = fminf(fmaxf(q, 0.0f), 255.0f);
            c = uint8_t(int(q));
        }
        if (i < const_offset || i >= const_offset + 4) out[i] = c;
    }
    if (lane == 0) {
        __half2 h = __halves2half2(dh, lh);
        *reinterpret_cast<__half2*>(out + const_offset) = h;
    }
}

// Filtered search (bindings/cpp/src/vamana_index_impl.h:139-218): out of a query's `kk` search results (sorted), keep
// the first k whose id is a member of the filter bitmap; `found[q]` = how many there were.
__global__ void filter_topk_kernel(const uint64_t* __restrict__ ids, const float* __restrict__ dists, uint32_t nq, uint32_t kk,
                                   uint32_t k, const uint32_t* __restrict__ bitmap, uint64_t* __restrict__ out_ids,
                                   float* __restrict__ out_dists, uint32_t* __restrict__ found, uint32_t* __restrict__ unfinished) {
    const uint32_t q = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const uint32_t lane = threadIdx.x & 31;
    if (q >= nq) return;
    uint32_t cnt = 0;
    bool exhausted = false;   // the search returned fewer than kk valid entries: nothing more to find
    for (uint32_t j0 = 0; j0 < kk && cnt < k; j0 += 32) {
        const uint32_t j = j0 + lane;
        const uint64_t id = j < kk ? ids[size_t(q) * kk + j] : ~uint64_t(0);
        const bool valid = id != ~uint64_t(0);
        const bool pass = valid && ((bitmap[id >> 5] >> (id & 31)) & 1u);
        const unsigned m = __ballot_sync(0xFFFFFFFFu, pass);
        const uint32_t o = cnt + __popc(m & ((1u << lane) - 1u));
        if (pass && o < k) {
            out_ids[size_t(q) * k + o] = id;
            out_dists[size_t(q) * k + o] = dists[size_t(q) * kk + j];
        }
        cnt += __popc(m);
        if (__any_sync(0xFFFFFFFFu, j < kk && !valid)) exhausted = true;
    }
    cnt = min(cnt, k);
    if (lane == 0) {
        found[q] = cnt;
        if (cnt < k && !exhausted) atomicAdd(unfinished, 1u);
    }
}

// Range search (vamana_index_impl.h:227-300): number of a query's sorted results inside the radius; a query whose
// last result is still inside needs a longer list.
__global__ void range_count_kernel(const float* __restrict__ dists, const uint64_t* __restrict__ ids, uint32_t nq, uint32_t kk,
                                   float radius, int greater, uint32_t* __restrict__ counts, uint32_t* __restrict__ unfinished) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    uint32_t c = 0;
    bool exhausted = false;
    for (; c < kk; ++c) {
        if (ids[size_t(q) * kk + c] == ~uint64_t(0)) {
            exhausted = true;
            break;
        }
        const float d = dists[size_t(q) * kk + c];
        if (greater ? !(d > radius) : !(d < radius)) break;
    }
    counts[q] = c;
    if (c == kk && !exhausted) atomicAdd(unfinished, 1u);
}

// Prepares the batch's queries for the search kernels (the device-side maybe_fix_argument) into sc's query buffers.
static int prepare_queries(const svsb200_index* ix, const Replica* rep, Scratch* sc, const void* d_queries, int qdtype,
                           size_t nq, int mode, cudaStream_t stream) {
    const uint32_t qstride = qstride_for(ix->dim);
    CUDA_TRY(sc->q_f32.ensure(nq * qstride));
    CUDA_TRY(sc->q_codes.ensure(nq * qstride));
    CUDA_TRY(sc->q_aux.ensure(nq * 2));
    auto launch = [&](auto kernel) {
        const int warps = 8;
        kernel<<<unsigned((nq + warps - 1) / warps), warps * 32, 0, stream>>>(
            d_queries, uint32_t(nq), uint32_t(ix->dim), qstride, mode, ix->metric, ix->dtype, ix->scale, ix->bias,
            rep->d_mean.ptr, sc->q_f32.ptr, sc->q_codes.ptr, sc->q_aux.ptr);
    };
    switch (qdtype) {
        case SVSB200_F32: launch(prepare_queries_kernel<SVSB200_F32>); break;
        case SVSB200_F16: launch(prepare_queries_kernel<SVSB200_F16>); break;
        case SVSB200_I8: launch(prepare_queries_kernel<SVSB200_I8>); break;
        default: launch(prepare_queries_kernel<SVSB200_U8>);
    }
    count_launch();
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// Calls f(std::integral_constant<int, ROWT>()) for the search kernels' row type `rowt`.
template <typename F> static cudaError_t with_row_type(int rowt, F&& f) {
    switch (rowt) {
        case ROW_LVQ8: return f(std::integral_constant<int, ROW_LVQ8>());
        case SVSB200_F32: return f(std::integral_constant<int, SVSB200_F32>());
        case SVSB200_F16: return f(std::integral_constant<int, SVSB200_F16>());
        case SVSB200_I8: return f(std::integral_constant<int, SVSB200_I8>());
        default: return f(std::integral_constant<int, SVSB200_U8>());
    }
}

}  // namespace svsb200

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" {

const char* svsb200_last_error(void) { return g_error.c_str(); }
int svsb200_version(void) { return SVSB200_VERSION; }
uint64_t svsb200_launch_count(void) { return g_launches.load(); }

int svsb200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int svsb200_device_sm(int device, int* sm) {
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (sm) *sm = prop.major * 10 + prop.minor;
    return 0;
}

// -----------------------------------------------------------------------------------------------------------------
// Assembling an index from files, streamed straight into HBM (SURVEY.md 8 f3).  Replaces
// index::vamana::auto_assemble (index/vamana/index.h:1022-1050) + the native / vecs readers
// (core/io/native.h:315-345, core/io/vecs.h:137-273) + the TOML load of VamanaIndexParameters
// (index/vamana/index.h:53-178, lib/saveload/load.h:829-878).
// -----------------------------------------------------------------------------------------------------------------
namespace {

// A TOML subset sufficient for the reference's saved configurations: comments, [tables] with dotted names,
// [[arrays of tables]] (skipped), key = value with integers, floats, booleans, 'literal' / "basic" strings,
// dates as bare tokens.  Returns "table.key" -> raw value text (strings unquoted).
bool parse_toml_subset(const std::string& text, std::map<std::string, std::string>& out, std::string& err) {
    std::string table;
    bool skip = false;
    size_t line_no = 0, pos = 0;
    while (pos <= text.size()) {
        size_t eol = text.find('\n', pos);
        if (eol == std::string::npos) eol = text.size();
        std::string line = text.substr(pos, eol - pos);
        pos = eol + 1;
        ++line_no;
        // strip comments outside strings
        bool in_s = false, in_d = false;
        for (size_t i = 0; i < line.size(); ++i) {
            const char c = line[i];
            if (c == '\'' && !in_d) in_s = !in_s;
            else if (c == '"' && !in_s && (i == 0 || line[i - 1] != '\\')) in_d = !in_d;
            else if (c == '#' && !in_s && !in_d) {
                line.resize(i);
                break;
            }
        }
        auto trim = [](std::string& v) {
            const size_t b = v.find_first_not_of(" \t\r");
            if (b == std::string::npos) {
                v.clear();
                return;
            }
            v = v.substr(b, v.find_last_not_of(" \t\r") - b + 1);
        };
        trim(line);
        if (line.empty()) continue;
        if (line[0] == '[') {
            if (line.size() > 1 && line[1] == '[') {   // array of tables: not needed for index parameters
                skip = true;
                continue;
            }
            const size_t close = line.find(']');
            if (close == std::string::npos) {
                err = "line " + std::to_string(line_no) + ": unterminated table header";
                return false;
            }
            table = line.substr(1, close - 1);
            trim(table);
            skip = false;
            continue;
        }
        if (skip) continue;
        const size_t eq = line.find('=');
        if (eq == std::string::npos) {
            err = "line " + std::to_string(line_no) + ": expected key = value";
            return false;
        }
        std::string key = line.substr(0, eq), value = line.substr(eq + 1);
        trim(key);
        trim(value);
        if (key.size() >= 2 && (key.front() == '"' || key.front() == '\'')) key = key.substr(1, key.size() - 2);
        if (value.size() >= 2 && (value.front() == '\'' || value.front() == '"') && value.back() == value.front())
            value = value.substr(1, value.size() - 2);
        if (key.empty() || value.empty()) {
            err = "line " + std::to_string(line_no) + ": empty key or value";
            return false;
        }
        out[table.empty() ? key : table + "." + key] = value;
    }
    return true;
}

// Reads `path` and parses it with parse_toml_subset.
int read_toml_file(const std::string& path, std::map<std::string, std::string>& cfg) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return fail("cannot open " + path);
    std::string text;
    char buf[4096];
    size_t got;
    while ((got = fread(buf, 1, sizeof(buf), f)) > 0) text.append(buf, got);
    fclose(f);
    std::string err;
    if (!parse_toml_subset(text, cfg, err)) return fail(path + ": " + err);
    return 0;
}

struct RowFile {
    FILE* f = nullptr;
    size_t n = 0, dim = 0, esize = 0;
    size_t row_prefix = 0;     // bytes in front of every row (vecs formats: the int32 dimension)
    ~RowFile() {
        if (f) fclose(f);
    }
};

std::string resolve(const std::string& path, const char* inside) {
    struct stat st;
    if (stat(path.c_str(), &st) == 0 && S_ISDIR(st.st_mode)) return path + "/" + inside;
    return path;
}

// Opens a native v1 .svs container or a [fibh]vecs file; `esize` is the element size the caller expects.
int open_rows(const std::string& path, size_t esize, RowFile& rf) {
    rf.f = fopen(path.c_str(), "rb");
    if (!rf.f) return fail("cannot open " + path);
    rf.esize = esize;
    const size_t dot = path.rfind('.');
    const std::string ext = dot == std::string::npos ? "" : path.substr(dot);
    fseek(rf.f, 0, SEEK_END);
    const size_t bytes = size_t(ftell(rf.f));
    fseek(rf.f, 0, SEEK_SET);
    if (ext == ".fvecs" || ext == ".ivecs" || ext == ".bvecs" || ext == ".hvecs") {
        int32_t d = 0;
        if (fread(&d, 4, 1, rf.f) != 1 || d <= 0) return fail(path + ": empty or malformed vecs file");
        rf.dim = size_t(d);
        rf.row_prefix = 4;
        const size_t row = 4 + rf.dim * esize;
        if (bytes % row) return fail(path + ": size is not a multiple of the row size");
        rf.n = bytes / row;
        fseek(rf.f, 0, SEEK_SET);
        return 0;
    }
    unsigned char header[1024];
    if (fread(header, 1, 1024, rf.f) != 1024) return fail(path + ": truncated header");
    uint64_t magic, n, dims;
    memcpy(&magic, header, 8);
    memcpy(&n, header + 24, 8);
    memcpy(&dims, header + 32, 8);
    if (magic != 0xcad4a6b2579980feull) return fail(path + ": not a native v1 .svs file (bad magic)");
    if (bytes < 1024 + n * dims * esize) return fail(path + ": truncated body");
    rf.n = n;
    rf.dim = dims;
    return 0;
}

// Streams the rows of `rf` through two pinned staging buffers: while chunk i is copied host->device (asynchronously,
// strided into the padded HBM rows), chunk i+1 is read from the file.  `sink(dev_chunk_rows_ptr?, ...)` is not needed:
// rows land at dst + row * dst_stride.
int stream_rows_to_device(RowFile& rf, char* dst, size_t dst_stride, cudaStream_t stream) {
    const size_t src_row = rf.row_prefix + rf.dim * rf.esize;
    const size_t chunk_rows = std::max<size_t>(1, (size_t(32) << 20) / src_row);
    char* pinned[2] = {nullptr, nullptr};
    cudaEvent_t done[2] = {nullptr, nullptr};
    int rc = 0;
    for (int i = 0; i < 2 && rc == 0; ++i) {
        if (cudaMallocHost(&pinned[i], chunk_rows * src_row) != cudaSuccess || cudaEventCreate(&done[i]) != cudaSuccess)
            rc = fail("pinned staging buffer allocation failed");
    }
    for (size_t r0 = 0, c = 0; r0 < rf.n && rc == 0; r0 += chunk_rows, ++c) {
        const int b = int(c & 1);
        const size_t rows = std::min(chunk_rows, rf.n - r0);
        if (c >= 2 && cudaEventSynchronize(done[b]) != cudaSuccess) rc = fail("cudaEventSynchronize failed");
        if (rc == 0 && fread(pinned[b], src_row, rows, rf.f) != rows) rc = fail("short read");
        if (rc == 0 &&
            cudaMemcpy2DAsync(dst + r0 * dst_stride, dst_stride, pinned[b] + rf.row_prefix, src_row, rf.dim * rf.esize, rows,
                              cudaMemcpyHostToDevice, stream) != cudaSuccess)
            rc = fail("cudaMemcpy2DAsync failed");
        if (rc == 0) cudaEventRecord(done[b], stream);
    }
    if (cudaStreamSynchronize(stream) != cudaSuccess && rc == 0) rc = fail("stream synchronisation failed");
    for (int i = 0; i < 2; ++i) {
        if (pinned[i]) cudaFreeHost(pinned[i]);
        if (done[i]) cudaEventDestroy(done[i]);
    }
    return rc;
}

}  // namespace

// Where the first replica's bytes come from: host arrays, or (when the RowFile pointers are set) the files being
// assembled from.
struct ReplicaSource {
    const void* vectors = nullptr;
    size_t vector_stride = 0;            // bytes between host rows; 0 = packed
    const uint32_t* graph_rows = nullptr;
    const float* aux = nullptr;          // SQ: {scale, bias}; LVQ-8: mean[dim]
    RowFile* vector_file = nullptr;
    RowFile* graph_file = nullptr;
};

// Allocates the replica's arrays and fills them from `src`: the vectors into padded rows, the graph through a staging
// copy of the reference's rows that repack_graph_kernel turns into the HBM layout.
static int upload_replica(const char* who, svsb200_index* ix, Replica* rep, size_t graph_row_len, const ReplicaSource& src) {
    const size_t n = ix->n;
    CUDA_TRY(cudaSetDevice(rep->device));
    cudaStream_t stream = nullptr;
    CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    StreamOwner stream_owner(stream, cudaStreamDestroy);   // (declared first: destroyed after the staging buffers are freed)
    const size_t vbytes = n * size_t(ix->row_stride);
    const size_t gbytes = n * size_t(ix->gstride) * sizeof(uint32_t);
    CUDA_TRY(rep->d_vectors.ensure(vbytes));
    CUDA_TRY(rep->d_graph.ensure(n * size_t(ix->gstride)));
    CUDA_TRY(rep->d_ref_degree.ensure(n));
    ix->device_bytes = vbytes + gbytes + n * sizeof(uint16_t);
    CUDA_TRY(cudaMemsetAsync(rep->d_vectors.ptr, 0, vbytes, stream));
    if (src.vector_file) {
        if (int rc = stream_rows_to_device(*src.vector_file, rep->d_vectors.ptr, ix->row_stride, stream)) return rc;
    } else {
        const size_t row_bytes = ix->storage == SVSB200_LVQ8 ? ix->lvq_const_offset + 4 : ix->dim * esize(ix->dtype);
        CUDA_TRY(cudaMemcpy2DAsync(rep->d_vectors.ptr, ix->row_stride, src.vectors,
                                   src.vector_stride ? src.vector_stride : row_bytes, row_bytes, n, cudaMemcpyHostToDevice,
                                   stream));
    }
    DeviceBuffer<uint32_t> d_src;
    DeviceBuffer<int> d_bad;
    CUDA_TRY(d_src.ensure(n * graph_row_len));
    CUDA_TRY(d_bad.ensure(1));
    CUDA_TRY(cudaMemsetAsync(d_bad.ptr, 0, sizeof(int), stream));
    if (src.graph_file) {
        if (int rc = stream_rows_to_device(*src.graph_file, reinterpret_cast<char*>(d_src.ptr), graph_row_len * 4, stream))
            return rc;
    } else {
        CUDA_TRY(cudaMemcpyAsync(d_src.ptr, src.graph_rows, n * graph_row_len * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                 stream));
    }
    const int warps = 8;
    repack_graph_kernel<<<unsigned((n + warps - 1) / warps), warps * 32, 0, stream>>>(
        d_src.ptr, graph_row_len, uint32_t(n), rep->d_graph.ptr, ix->gstride, rep->d_ref_degree.ptr, d_bad.ptr);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    int bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, d_bad.ptr, sizeof(int), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    if (bad) return fail(std::string(who) + (bad == 1 ? ": adjacency row with degree > max_degree" : ": neighbour id out of range"));
    if (ix->storage == SVSB200_LVQ8) {
        CUDA_TRY(rep->d_mean.ensure(ix->dim));
        CUDA_TRY(cudaMemcpy(rep->d_mean.ptr, src.aux, ix->dim * sizeof(float), cudaMemcpyHostToDevice));
    }
    return 0;
}

// Copies an uploaded replica device to device (NVLink when peer access exists).
static int clone_replica(svsb200_index* ix, const Replica* src, Replica* dst) {
    const size_t n = ix->n;
    CUDA_TRY(cudaSetDevice(dst->device));
    const size_t vbytes = n * size_t(ix->row_stride);
    const size_t gbytes = n * size_t(ix->gstride) * sizeof(uint32_t);
    CUDA_TRY(dst->d_vectors.ensure(vbytes));
    CUDA_TRY(dst->d_graph.ensure(n * size_t(ix->gstride)));
    CUDA_TRY(dst->d_ref_degree.ensure(n));
    CUDA_TRY(cudaMemcpyPeer(dst->d_vectors.ptr, dst->device, src->d_vectors.ptr, src->device, vbytes));
    CUDA_TRY(cudaMemcpyPeer(dst->d_graph.ptr, dst->device, src->d_graph.ptr, src->device, gbytes));
    CUDA_TRY(cudaMemcpyPeer(dst->d_ref_degree.ptr, dst->device, src->d_ref_degree.ptr, src->device, n * sizeof(uint16_t)));
    if (src->d_mean.ptr) {
        CUDA_TRY(dst->d_mean.ensure(ix->dim));
        CUDA_TRY(cudaMemcpyPeer(dst->d_mean.ptr, dst->device, src->d_mean.ptr, src->device, ix->dim * sizeof(float)));
    }
    return 0;
}

// Argument checks that create and assemble share, in the order both make them.
static int check_index_kind(const char* who, const int* devices, size_t ndevices, int dtype, int metric) {
    const std::string w(who);
    if (!devices || ndevices == 0) return fail(w + ": empty device list");
    if (dtype < SVSB200_F32 || dtype > SVSB200_U8) return fail(w + ": bad dtype");
    if (metric < SVSB200_L2 || metric > SVSB200_COSINE) return fail(w + ": bad metric");
    return 0;
}
static int check_index_size(const char* who, size_t n, size_t dim) {
    if (n == 0 || dim == 0) return fail(std::string(who) + ": empty dataset");
    if (n >= (size_t(1) << 31)) return fail(std::string(who) + ": more than 2^31-1 vectors per index");
    return 0;
}

// The index over checked arguments: its fields and layout, then one replica per listed device, the first uploaded from
// `src` and the others copied from it.
static int make_index(const char* who, int dtype, int metric, int storage, size_t n, size_t dim, size_t graph_row_len,
                      uint32_t entry_point, const int* devices, size_t ndevices, const ReplicaSource& src,
                      std::unique_ptr<svsb200_index>& ix) {
    const std::string w(who);
    const int ndev = svsb200_device_count();
    if (ndev == 0) return fail(w + ": no CUDA device (there is no CPU fallback)");
    ix.reset(new svsb200_index());
    ix->dtype = dtype;
    ix->metric = metric;
    ix->storage = storage;
    ix->n = n;
    ix->dim = dim;
    ix->max_degree = graph_row_len - 1;
    ix->entry_point = entry_point;
    if (storage == SVSB200_SQ) {
        ix->scale = src.aux[0];
        ix->bias = src.aux[1];
    }
    if (storage == SVSB200_LVQ8) ix->lvq_const_offset = uint32_t(round_up(dim, 4));
    ix->row_stride = row_stride_for(storage, dtype, dim);
    ix->gstride = gstride_for(ix->max_degree);

    for (size_t r = 0; r < ndevices; ++r) {
        const int device = devices[r];
        if (device < 0 || device >= ndev) return fail(w + ": bad device ordinal");
        for (size_t j = 0; j < r; ++j)
            if (devices[j] == device) return fail(w + ": device listed twice");
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10 || prop.minor != 0) return fail(w + ": device is not sm_100 (this binary holds sm_100a code only)");
        std::unique_ptr<Replica> rep(new Replica());
        rep->device = device;
        rep->sm_count = prop.multiProcessorCount;
        int rc = r == 0 ? upload_replica(who, ix.get(), rep.get(), graph_row_len, src)
                        : clone_replica(ix.get(), ix->reps[0].get(), rep.get());
        if (rc) return rc;
        ix->reps.push_back(std::move(rep));
    }
    return 0;
}

int svsb200_index_create_multi(const void* vectors, int dtype, size_t n, size_t dim, size_t row_stride_bytes,
                               const uint32_t* graph_rows, size_t graph_row_len, uint32_t entry_point, int metric,
                               int storage, const float* aux, const int* devices, size_t ndevices, svsb200_index** out) {
    const char* who = "svsb200_index_create";
    if (!out) return fail("svsb200_index_create: out is NULL");
    *out = nullptr;
    if (!vectors || !graph_rows) return fail("svsb200_index_create: NULL input");
    if (int rc = check_index_kind(who, devices, ndevices, dtype, metric)) return rc;
    if (int rc = check_index_size(who, n, dim)) return rc;
    if (graph_row_len < 2) return fail("svsb200_index_create: graph rows need a degree word and one slot");
    if (graph_row_len > 65536) return fail("svsb200_index_create: max_degree above 65535");
    if (entry_point >= n) return fail("svsb200_index_create: entry point out of range");
    if (storage == SVSB200_SQ) {
        if (dtype != SVSB200_I8 && dtype != SVSB200_U8) return fail("svsb200_index_create: SQ codes must be int8/uint8");
        if (!aux) return fail("svsb200_index_create: SQ needs aux = {scale, bias}");
    } else if (storage == SVSB200_LVQ8) {
        if (dtype != SVSB200_U8) return fail("svsb200_index_create: LVQ-8 rows are uint8 codes (dtype SVSB200_U8)");
        if (!aux) return fail("svsb200_index_create: LVQ-8 needs aux = mean[dim]");
        if (row_stride_bytes != svsb200_lvq8_row_stride(dim))
            return fail("svsb200_index_create: LVQ-8 rows must use svsb200_lvq8_row_stride(dim)");
    } else if (storage != SVSB200_PLAIN) {
        return fail("svsb200_index_create: unsupported storage kind");
    }
    ReplicaSource src;
    src.vectors = vectors;
    src.vector_stride = row_stride_bytes;
    src.graph_rows = graph_rows;
    src.aux = aux;
    std::unique_ptr<svsb200_index> ix;
    if (int rc = make_index(who, dtype, metric, storage, n, dim, graph_row_len, entry_point, devices, ndevices, src, ix))
        return rc;
    *out = ix.release();
    return 0;
}

int svsb200_index_create(const void* vectors, int dtype, size_t n, size_t dim, size_t row_stride_bytes,
                         const uint32_t* graph_rows, size_t graph_row_len, uint32_t entry_point, int metric, int storage,
                         const float* aux, int device, svsb200_index** out) {
    return svsb200_index_create_multi(vectors, dtype, n, dim, row_stride_bytes, graph_rows, graph_row_len, entry_point,
                                      metric, storage, aux, &device, 1, out);
}


int svsb200_toml_get(const char* path, const char* dotted_key, char* out, size_t capacity) {
    if (!path || !dotted_key || !out || capacity == 0) return fail("svsb200_toml_get: NULL argument");
    std::map<std::string, std::string> cfg;
    if (int rc = read_toml_file(path, cfg)) return rc;
    auto it = cfg.find(dotted_key);
    if (it == cfg.end()) return fail(std::string(path) + ": no key " + dotted_key);
    if (it->second.size() + 1 > capacity) return fail("svsb200_toml_get: value does not fit");
    memcpy(out, it->second.c_str(), it->second.size() + 1);
    return 0;
}

int svsb200_index_assemble(const char* config_path, const char* graph_path, const char* data_path, int dtype,
                           size_t expected_dims, int metric, const int* devices, size_t ndevices, svsb200_index** out) {
    const char* who = "svsb200_index_assemble";
    if (!out) return fail("svsb200_index_assemble: out is NULL");
    *out = nullptr;
    if (!config_path || !graph_path || !data_path) return fail("svsb200_index_assemble: NULL path");
    if (int rc = check_index_kind(who, devices, ndevices, dtype, metric)) return rc;
    // ---- VamanaIndexParameters from TOML ----
    const std::string cfg_file = resolve(config_path, "svs_config.toml");
    std::map<std::string, std::string> cfg;
    if (int rc = read_toml_file(cfg_file, cfg)) return rc;
    auto cfg_long = [&](const char* key, long dflt) {
        auto it = cfg.find(key);
        if (it == cfg.end()) return dflt;
        if (it->second == "true") return 1l;
        if (it->second == "false") return 0l;
        return strtol(it->second.c_str(), nullptr, 10);
    };
    if (cfg.find("object.entry_point") == cfg.end()) return fail(cfg_file + ": no entry_point in [object]");
    const long entry_point = cfg_long("object.entry_point", 0);
    // ---- files ----
    RowFile data, graph;
    int rc = open_rows(resolve(data_path, "data_0.svs"), esize(dtype), data);
    if (rc) return rc;
    rc = open_rows(resolve(graph_path, "graph_0.svs"), 4, graph);
    if (rc) return rc;
    if (expected_dims && data.dim != expected_dims)
        return fail("svsb200_index_assemble: the data file holds " + std::to_string(data.dim) + "-dimensional vectors, " +
                    std::to_string(expected_dims) + " expected");
    if (graph.n != data.n) return fail("Wrong sizes!");   // index/vamana/index.h:417-419
    const size_t n = data.n, graph_row_len = graph.dim;
    if ((rc = check_index_size(who, n, data.dim))) return rc;
    if (graph_row_len < 2 || graph_row_len > 65536) return fail("svsb200_index_assemble: bad graph row length");
    if (entry_point < 0 || size_t(entry_point) >= n) return fail("svsb200_index_assemble: entry point out of range");
    ReplicaSource src;
    src.vector_file = &data;
    src.graph_file = &graph;
    std::unique_ptr<svsb200_index> ix;
    rc = make_index(who, dtype, metric, SVSB200_PLAIN, n, data.dim, graph_row_len, uint32_t(entry_point), devices, ndevices,
                    src, ix);
    if (rc) return rc;
    ix->cfg_window = cfg_long("object.search_parameters.search_window_size", 0);
    ix->cfg_capacity = cfg_long("object.search_parameters.search_buffer_capacity", 0);
    ix->cfg_visited = cfg_long("object.search_parameters.search_buffer_visited_set", 0);
    *out = ix.release();
    return 0;
}

int svsb200_index_destroy(svsb200_index* ix) {
    delete ix;   // Replica / Scratch destructors release the device memory
    return 0;
}

size_t svsb200_index_size(const svsb200_index* ix) { return ix ? ix->n : 0; }
size_t svsb200_index_dimensions(const svsb200_index* ix) { return ix ? ix->dim : 0; }
size_t svsb200_index_max_degree(const svsb200_index* ix) { return ix ? ix->max_degree : 0; }
size_t svsb200_index_device_bytes(const svsb200_index* ix) { return ix ? ix->device_bytes : 0; }
int svsb200_index_device(const svsb200_index* ix) { return ix && !ix->reps.empty() ? ix->reps[0]->device : -1; }
size_t svsb200_index_num_devices(const svsb200_index* ix) { return ix ? ix->reps.size() : 0; }

int svsb200_set_counting(svsb200_index* ix, int enabled) {
    if (!ix) return fail("svsb200_set_counting: NULL index");
    ix->counting = enabled;
    return 0;
}

int svsb200_set_entry_points(svsb200_index* ix, const uint32_t* entry_points, size_t count) {
    if (!ix || !entry_points) return fail("svsb200_set_entry_points: NULL argument");
    if (count == 0 || count > 32) return fail("svsb200_set_entry_points: 1..32 entry points");
    for (size_t i = 0; i < count; ++i)
        if (entry_points[i] >= ix->n) return fail("svsb200_set_entry_points: entry point out of range");
    for (auto& rep : ix->reps) {
        CUDA_TRY(cudaSetDevice(rep->device));
        CUDA_TRY(cudaDeviceSynchronize());
        CUDA_TRY(rep->d_entry.ensure(32));
        CUDA_TRY(cudaMemcpy(rep->d_entry.ptr, entry_points, count * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    ix->entry_point = entry_points[0];
    ix->n_entry = uint32_t(count);
    return 0;
}

int svsb200_set_id_offset(svsb200_index* ix, uint64_t offset) {
    if (!ix) return fail("svsb200_set_id_offset: NULL index");
    ix->id_offset = offset;
    return 0;
}

int svsb200_set_option(svsb200_index* ix, const char* name, long value) {
    if (!ix || !name) return fail("svsb200_set_option: NULL argument");
    const std::string key(name);
    if (key == "warps_per_cta") {
        if (value < 0 || value > 8) return fail("warps_per_cta must be in [0, 8]");
        ix->warps_per_cta = value;
    } else if (key == "ctas_per_sm") {
        if (value < 0 || value > 32) return fail("ctas_per_sm must be in [0, 32]");
        ix->ctas_per_sm = value;
    } else if (key == "rows_in_flight") {
        if (value < 0 || value > 2) return fail("rows_in_flight must be in [0, 2]");
        ix->rows_in_flight = value;
    } else if (key == "generic_kernel") {
        ix->generic_kernel = value;
    } else if (key == "host_chunks") {
        if (value < 0 || value > 16) return fail("host_chunks must be in [0, 16]");
        ix->host_chunks = value;
    } else if (key == "visited_filter_slots") {
        // -1 = default; 0 = off; otherwise a power of two
        if (value > 0 && (value & (value - 1))) return fail("visited_filter_slots must be a power of two");
        // the filter words sit in front of 16-byte aligned arrays in shared memory
        if (value > 0 && value < 8) return fail("visited_filter_slots must be 0 (off) or at least 8");
        if (value > 16384) return fail("visited_filter_slots must be <= 16384");
        ix->filter_slots = value;
    } else {
        return fail("svsb200_set_option: unknown option " + key);
    }
    return 0;
}

int svsb200_get_option(svsb200_index* ix, const char* name, long* value) {
    if (!ix || !name || !value) return fail("svsb200_get_option: NULL argument");
    const std::string key(name);
    if (key == "last_kernel") {          // 1 = lean kernel, 0 = generic kernel
        std::lock_guard<std::mutex> lock(ix->mu);
        *value = ix->last ? ix->last->last_kernel : 0;
    } else if (key == "warps_per_cta") *value = ix->warps_per_cta;
    else if (key == "ctas_per_sm") *value = ix->ctas_per_sm;
    else if (key == "rows_in_flight") *value = ix->rows_in_flight;
    else if (key == "visited_filter_slots") *value = ix->filter_slots;
    else if (key == "generic_kernel") *value = ix->generic_kernel;
    else if (key == "host_chunks") *value = ix->host_chunks;
    else if (key == "config_search_window_size") *value = ix->cfg_window;
    else if (key == "config_search_buffer_capacity") *value = ix->cfg_capacity;
    else if (key == "config_search_buffer_visited_set") *value = ix->cfg_visited;
    else if (key == "entry_point") *value = long(ix->entry_point);
    else if (key == "streams") {         // scratch sets (= streams) created so far over all replicas
        long c = 0;
        for (auto& rep : ix->reps) {
            std::lock_guard<std::mutex> lock(rep->mu);
            c += long(rep->all.size());
        }
        *value = c;
    } else return fail("svsb200_get_option: unknown option " + key);
    return 0;
}

// Shared body of every search entry point: everything on one device, enqueued on `stream`.
static int search_on_device(svsb200_index* ix, Replica* rep, Scratch* sc, const void* d_queries, int qdtype, size_t nq,
                            size_t k, size_t window, size_t capacity, void* d_out_ids, int id_bytes, float* d_out_dists,
                            cudaStream_t stream, bool exhaustive = false) {
    if (id_bytes != 4 && id_bytes != 8) return fail("id_bytes must be 4 or 8");
    if (qdtype < SVSB200_F32 || qdtype > SVSB200_U8) return fail("bad query dtype");
    if (window > capacity) {
        // SearchBufferConfig::check_invariants (search_buffer.h:87-96)
        return fail("Improper configuration for search buffer! search window size cannot exceed capacity");
    }
    if (capacity < k) window = capacity = k;   // index/vamana/index.h:590-592
    if (capacity == 0) return fail("search buffer capacity is zero");
    if (nq == 0) return 0;
    if (nq >= (size_t(1) << 31)) return fail("too many queries in one batch");

    // Which (query, data) pairs exist, mirroring the SIMD specialisations
    // (euclidean.h:293-358) and the SQ CPOs (extensions/vamana/scalar.h:32-43).
    int op, mode;
    const int metric = ix->metric;
    if (ix->storage == SVSB200_LVQ8) {
        if (qdtype != SVSB200_F32 && qdtype != SVSB200_F16) return fail("LVQ-8 datasets take float32/float16 queries");
        if (metric == SVSB200_COSINE) return fail("LVQ-8: cosine is not supported (L2 and MIP are)");
        op = metric == SVSB200_L2 ? OP_L2F : OP_IPF;
        mode = metric == SVSB200_L2 ? PREP_LVQ_L2 : PREP_LVQ_IP;
    } else if (ix->storage == SVSB200_SQ) {
        if (qdtype != SVSB200_F32 && qdtype != SVSB200_F16) return fail("SQ datasets take float32/float16 queries");
        op = metric == SVSB200_L2 ? OP_L2I : metric == SVSB200_IP ? OP_IPF : OP_COSF;
        mode = metric == SVSB200_L2 ? PREP_SQ_L2 : metric == SVSB200_IP ? PREP_SQ_IP : PREP_SQ_COS;
    } else if (qdtype == SVSB200_I8 || qdtype == SVSB200_U8) {
        if (qdtype != ix->dtype) return fail("int8/uint8 queries need a dataset of the same type");
        op = metric == SVSB200_L2 ? OP_L2I : metric == SVSB200_IP ? OP_IPI : OP_COSI;
        mode = PREP_INT;
    } else {
        if (qdtype == SVSB200_F16 && ix->dtype != SVSB200_F32 && ix->dtype != SVSB200_F16)
            return fail("float16 queries need a float32/float16 dataset");
        op = metric == SVSB200_L2 ? OP_L2F : metric == SVSB200_IP ? OP_IPF : OP_COSF;
        mode = PREP_FLOAT;
    }

    const bool counting = ix->counting != 0;
    if (counting) {
        CUDA_TRY(sc->hops.ensure(nq));
        CUDA_TRY(sc->evals.ensure(nq));
        CUDA_TRY(sc->fetched.ensure(nq));
        sc->counted_nq = nq;
    }
    if (int rc = prepare_queries(ix, rep, sc, d_queries, qdtype, nq, mode, stream)) return rc;
    CUDA_TRY(cudaMemsetAsync(sc->d_counter.ptr, 0, sizeof(unsigned int), stream));
    // (sc->d_cancel is zero here: only wait_kernels raises it, and lowers it again once the kernels have finished)

    SearchParams p{};
    p.vectors = rep->d_vectors.ptr;
    p.graph = rep->d_graph.ptr;
    p.ref_degree = rep->d_ref_degree.ptr;
    p.n = uint32_t(ix->n);
    p.dim = uint32_t(ix->dim);
    p.row_stride = ix->row_stride;
    p.gstride = ix->gstride;
    p.entry_point = ix->entry_point;
    p.entry_points = rep->d_entry.ptr;
    // push_back drops entry points once the buffer is full (search_buffer.h:311-316): only the first `capacity` count
    p.n_entry = rep->d_entry.ptr ? uint32_t(std::min<size_t>(ix->n_entry, capacity)) : 1;
    p.greater = metric != SVSB200_L2;
    p.sq = ix->storage == SVSB200_SQ;
    p.lvq = ix->storage == SVSB200_LVQ8;
    p.lvq_const_offset = ix->lvq_const_offset;
    p.scale = ix->scale;
    p.bias = ix->bias;
    p.scale_sq = ix->scale * ix->scale;   // EuclideanCompressed ctor (scalar.h:68-72)
    p.qf = sc->q_f32.ptr;
    p.qcodes = sc->q_codes.ptr;
    p.qaux = sc->q_aux.ptr;
    p.qstride = qstride_for(ix->dim);
    p.nq = uint32_t(nq);
    p.k = uint32_t(k);
    p.window = uint32_t(window);
    p.capacity = uint32_t(capacity);
    p.cap_pad = uint32_t(round_up(capacity + 1, 32));
    p.deg_pad = uint32_t(round_up(ix->gstride, 32));
    p.out_ids = d_out_ids;
    p.id_bytes = id_bytes;
    p.id_offset = id_bytes == 8 ? ix->id_offset : 0;
    p.out_dists = d_out_dists;
    p.work_counter = sc->d_counter.ptr;
    p.cancel = sc->poll_cancel ? sc->d_cancel.ptr : nullptr;   // (no predicate: no per-hop poll in the kernel)
    p.hops = counting ? sc->hops.ptr : nullptr;
    p.evals = counting ? sc->evals.ptr : nullptr;
    p.fetched = counting ? sc->fetched.ptr : nullptr;
    p.filter_slots = exhaustive ? 0u : (ix->filter_slots < 0 ? 4096u : uint32_t(ix->filter_slots));
    // generic kernel: 16-bit tags (two per 32-bit set, 2-way LRU) are exact as long as every id >> log2(sets) fits
    // below the 0xFFFF "empty" mark; larger indexes fall back to direct-mapped 32-bit entries.
    p.filter_shift = 0;
    while ((2u << p.filter_shift) < p.filter_slots) ++p.filter_shift;   // log2(sets) with sets = slots / 2
    p.filter_tag16 = p.filter_slots >= 2 && ((uint64_t(ix->n - 1) >> p.filter_shift) < 0xFFFFull);
    if (!p.filter_tag16) {
        p.filter_shift = 0;
        while ((1u << p.filter_shift) < p.filter_slots) ++p.filter_shift;
    }

    LaunchConfig cfg{};
    const size_t smem_limit = 227 * 1024;
    // The lean kernel (search_fast.cuh) covers the common shape: 16-bit-tag filter on, adjacency rows of up to
    // 128 neighbours; anything else (and the exhaustive scan) runs on the generic kernel.
    // Its filter: default 256 sets (4 KB).
    const LeanFilterPlan fast = lean_filter_plan(ix->n, ix->dim, capacity, p.deg_pad,
                                                 ix->filter_slots < 0 ? 2048u : uint32_t(ix->filter_slots));
    const bool use_fast = !exhaustive && !ix->generic_kernel && fast.slots >= 64 &&
                          (uint64_t(ix->n - 1) >> fast.shift) < 0xFFFFull && p.deg_pad <= 32u * kFastMaxGW &&
                          p.gstride % 32u == 0 && fast.smem_bytes <= smem_limit;
    sc->last_kernel = use_fast ? 1 : 0;
    const int nrows = ix->rows_in_flight ? int(ix->rows_in_flight) : 2;
    if (use_fast) {
        p.cap_pad = uint32_t(round_up(capacity, 32));
        p.filter_slots = fast.slots;
        p.filter_shift = fast.shift;
        p.filter_tag16 = 1;
        cfg.warps_per_cta = 1;
        cfg.smem_bytes = fast.smem_bytes;
        cfg.stream = stream;
        cfg.grid = ix->ctas_per_sm ? rep->sm_count * int(ix->ctas_per_sm) : -rep->sm_count;
    } else {
        const size_t per_warp = warp_smem_bytes(p.qstride, p.cap_pad, p.deg_pad, p.filter_slots * (p.filter_tag16 ? 2u : 4u));
        int warps = ix->warps_per_cta ? int(ix->warps_per_cta) : 4;
        while (warps > 1 && per_warp * warps > smem_limit) warps >>= 1;
        if (per_warp * warps > smem_limit) return fail("search buffer capacity too large for shared memory");
        cfg.warps_per_cta = warps;
        cfg.smem_bytes = per_warp * warps;
        cfg.stream = stream;
        // grid: persistent CTAs; the launcher clamps to what is resident.  ctas_per_sm == 0
        // means "as many as fit" (computed by the launcher through the occupancy API).
        cfg.grid = rep->sm_count * (ix->ctas_per_sm ? int(ix->ctas_per_sm) : 0);
        if (cfg.grid == 0 || exhaustive) cfg.grid = -rep->sm_count;   // negative: launcher multiplies by occupancy
    }

    CUDA_TRY(cudaEventRecord(sc->ev_start, stream));
    const int rowt = ix->storage == SVSB200_LVQ8 ? ROW_LVQ8 : ix->dtype;
    cudaError_t err;
    if (exhaustive) {
        // few queries: cut the base rows into ranges so that (query, range) work items fill the GPU; the per-range
        // top-k lists are merged with TotalOrder (== the scan's own order: key, then id)
        const size_t want_items = size_t(rep->sm_count) * 32;
        uint32_t split = uint32_t(std::min<size_t>(64, std::max<size_t>(1, want_items / nq)));
        while (split > 1 && ix->n / split < 4 * k + 64) --split;
        if (split > 1) {
            CUDA_TRY(sc->exh_ids.ensure(size_t(split) * nq * k));
            CUDA_TRY(sc->exh_dists.ensure(size_t(split) * nq * k));
            p.out_ids = sc->exh_ids.ptr;
            p.out_dists = sc->exh_dists.ptr;
            p.exh_split = split;
        }
        err = with_row_type(rowt, [&](auto t) { return launch_search_exhaustive<decltype(t)::value>(op, p, cfg); });
        if (err == cudaSuccess && split > 1)
            err = launch_merge_topk(sc->exh_ids.ptr, sc->exh_dists.ptr, split, nq, k, metric != SVSB200_L2,
                                    static_cast<uint64_t*>(d_out_ids), d_out_dists, stream);
    } else if (use_fast) {
        err = with_row_type(rowt, [&](auto t) { return launch_search_fast<decltype(t)::value>(op, p, cfg); });
    } else {
        err = with_row_type(rowt, [&](auto t) { return launch_search<decltype(t)::value>(op, p, cfg, nrows); });
    }
    CUDA_TRY(err);
    CUDA_TRY(cudaEventRecord(sc->ev_stop, stream));
    sc->timed = true;
    {
        std::lock_guard<std::mutex> lock(ix->mu);
        ix->last = sc;
    }
    return 0;
}

int svsb200_search_device(svsb200_index* ix, const void* d_queries, int qdtype, size_t nq, size_t k, size_t window,
                          size_t capacity, int use_visited_set, void* d_out_ids, int id_bytes, float* d_out_dists,
                          void* stream_) {
    (void)use_visited_set;   // performance-only in the reference (search_buffer.h:420); results identical
    if (!ix) return fail("svsb200_search_device: NULL index");
    if (nq && (!d_queries || !d_out_ids || !d_out_dists)) return fail("svsb200_search_device: NULL buffer");
    Scratch* sc = nullptr;
    if (int rc = device_api_scratch("svsb200_search_device", ix, stream_, &sc)) return rc;
    return search_on_device(ix, ix->reps[0].get(), sc, d_queries, qdtype, nq, k, window, capacity, d_out_ids, id_bytes, d_out_dists,
                            sc->stream);
}

// Waits for the search kernels of `scs` (their ev_stop events); with a cancel callback it polls the callback
// meanwhile and raises the device flags the kernels poll per query and per hop (greedy_search.h:155,
// extensions.h:579).
static int wait_kernels(const std::vector<ScratchLease>& scs, int (*cancel)(void*), void* cancel_arg) {
    if (!cancel) return 0;   // nothing to poll for: the stream order of the copies behind the kernels is enough
    bool raised = false;
    int rc = 0;
    for (;;) {
        bool busy = false;
        for (const ScratchLease& l : scs) {
            Scratch* sc = l.sc;
            if (!sc->timed) continue;
            cudaSetDevice(sc->device);
            cudaError_t q = cudaEventQuery(sc->ev_stop);
            if (q == cudaErrorNotReady) busy = true;
            else if (q != cudaSuccess) rc = fail(std::string("cudaEventQuery: ") + cudaGetErrorString(q));
        }
        if (!busy || rc) break;
        if (!raised && cancel(cancel_arg)) {
            raised = true;
            for (const ScratchLease& l : scs) {
                cudaSetDevice(l.sc->device);
                cudaError_t e = cudaMemsetAsync(l.sc->d_cancel.ptr, 1, sizeof(int), l.sc->ctl);
                if (e != cudaSuccess) rc = fail(std::string("cudaMemsetAsync: ") + cudaGetErrorString(e));
            }
        }
        std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
    if (raised) {   // the kernels are done (or failed): lower the flags for the next search of these scratch sets
        for (const ScratchLease& l : scs) {
            cudaSetDevice(l.sc->device);
            cudaStreamSynchronize(l.sc->stream);
            cudaMemsetAsync(l.sc->d_cancel.ptr, 0, sizeof(int), l.sc->ctl);
            cudaStreamSynchronize(l.sc->ctl);
        }
    }
    return rc;
}
static int wait_all(const std::vector<ScratchLease>& scs) {
    for (const ScratchLease& l : scs) {
        cudaSetDevice(l.sc->device);
        CUDA_TRY(cudaStreamSynchronize(l.sc->stream));
    }
    return 0;
}

int svsb200_search_cancellable(svsb200_index* ix, const void* queries, int qdtype, size_t nq, size_t k, size_t window,
                               size_t capacity, int use_visited_set, void* out_ids, int id_bytes, float* out_dists,
                               void* stream_, int (*cancel)(void*), void* cancel_arg) {
    (void)use_visited_set;
    if (!ix) return fail("svsb200_search: NULL index");
    if (nq == 0) return 0;
    if (!queries || !out_ids || !out_dists) return fail("svsb200_search: NULL buffer");
    if (qdtype < SVSB200_F32 || qdtype > SVSB200_U8) return fail("bad query dtype");
    if (id_bytes != 4 && id_bytes != 8) return fail("id_bytes must be 4 or 8");
    const size_t R = ix->reps.size();
    if (stream_ && R != 1) return fail("svsb200_search: a caller stream needs a single-device index");
    if (cancel && cancel(cancel_arg)) return 0;   // index.h:575 checks before any work
    const size_t qrow = ix->dim * esize(qdtype);
    std::vector<ScratchLease> used;
    std::vector<size_t> used_lo, used_m;
    int rc = 0;
    // Every device's share is cut into C pieces, each on its own stream: the host-to-device copy of piece i+1 and the
    // device-to-host copy of piece i-1 run under the kernel of piece i (the kernels of consecutive pieces overlap
    // too -- the next one's CTAs start as the previous one's retire).  C = 1 on a caller's stream (enqueue order is
    // the caller's) and for small shares.
    size_t C = 1;
    if (!stream_ && !ix->counting && !cancel) {   // (the diagnostic counters describe one launch; a predicate: one piece)
        const size_t share = (nq + R - 1) / R;
        // (measured on C2: 1 piece 6.5 M QPS end to end, 4 pieces 7.1 M, 8 pieces 6.8-6.9 M -- the enqueue calls of a piece
        // cost the host about as much as 1 000 queries cost the GPU)
        C = ix->host_chunks > 0 ? size_t(ix->host_chunks) : (share >= 4096 ? 4 : share >= 1024 ? 2 : 1);
        C = std::min(C, share);
    }
    for (size_t part = 0; part < R * C && rc == 0; ++part) {
        const size_t r = part / C;
        size_t lo, hi;
        balance(nq, R * C, part, &lo, &hi);
        if (hi == lo) continue;
        Replica* rep = ix->reps[r].get();
        ScratchLease lease;
        if ((rc = lease.take(rep, static_cast<cudaStream_t>(stream_)))) break;
        Scratch* sc = lease.sc;
        used.push_back(std::move(lease));
        const size_t m = hi - lo;
        used_lo.push_back(lo);
        used_m.push_back(m);
        sc->timed = false;
        sc->poll_cancel = cancel != nullptr;
        auto step = [&]() -> int {
            CUDA_TRY(sc->q_raw.ensure(m * qrow));
            CUDA_TRY(sc->ids.ensure(m * k * size_t(id_bytes)));
            CUDA_TRY(sc->dists.ensure(m * k));
            CUDA_TRY(cudaMemcpyAsync(sc->q_raw.ptr, static_cast<const char*>(queries) + lo * qrow, m * qrow,
                                     cudaMemcpyHostToDevice, sc->stream));
            return search_on_device(ix, rep, sc, sc->q_raw.ptr, qdtype, m, k, window, capacity, sc->ids.ptr, id_bytes,
                                    sc->dists.ptr, sc->stream);
        };
        rc = step();
    }
    std::string first_error = g_error;
    // the kernels of every replica are in flight: poll the predicate until they finish (a copy into pageable host
    // memory would block this thread, so the device-to-host copies are only enqueued afterwards)
    int rc_wait = wait_kernels(used, cancel, cancel_arg);
    for (size_t i = 0; i < used.size() && rc == 0 && rc_wait == 0; ++i) {
        Scratch* sc = used[i].sc;
        if (!sc->timed) continue;
        auto copy_out = [&]() -> int {
            CUDA_TRY(cudaSetDevice(sc->device));
            CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out_ids) + used_lo[i] * k * size_t(id_bytes), sc->ids.ptr,
                                     used_m[i] * k * size_t(id_bytes), cudaMemcpyDeviceToHost, sc->stream));
            CUDA_TRY(cudaMemcpyAsync(out_dists + used_lo[i] * k, sc->dists.ptr, used_m[i] * k * sizeof(float),
                                     cudaMemcpyDeviceToHost, sc->stream));
            return 0;
        };
        rc = copy_out();
        if (rc) first_error = g_error;
    }
    if (rc_wait == 0) rc_wait = wait_all(used);
    for (const ScratchLease& l : used) l.sc->poll_cancel = false;
    if (rc) {
        g_error = first_error;
        return rc;
    }
    return rc_wait;
}

int svsb200_search(svsb200_index* ix, const void* queries, int qdtype, size_t nq, size_t k, size_t window,
                   size_t capacity, int use_visited_set, void* out_ids, int id_bytes, float* out_dists, void* stream_) {
    return svsb200_search_cancellable(ix, queries, qdtype, nq, k, window, capacity, use_visited_set, out_ids, id_bytes,
                                      out_dists, stream_, nullptr, nullptr);
}

// Searches the queries in sc->q_raw with result lists of `kk` entries (window = capacity = max(window, kk)) into the
// scratch's own id / distance blocks; `check(kk)` enqueues the kernel that counts the queries that need longer lists
// into *d_unfinished.  The lists grow (x4) until no query is unfinished, like the reference's batch iterator asks for
// further batches (vamana_index_impl.h:183-205).  *kk is the length of the last lists.
extern "C++" template <typename Check>
int search_growing_lists(svsb200_index* ix, Replica* rep, Scratch* sc, int qdtype, size_t nq, size_t window,
                         uint32_t* d_unfinished, size_t* kk, Check check) {
    for (;;) {
        *kk = std::min(*kk, ix->n);
        CUDA_TRY(sc->ids.ensure(nq * *kk * 8));
        CUDA_TRY(sc->dists.ensure(nq * *kk));
        const size_t w = std::max(window, *kk);
        int rc = search_on_device(ix, rep, sc, sc->q_raw.ptr, qdtype, nq, *kk, w, w, sc->ids.ptr, 8, sc->dists.ptr, sc->stream);
        if (rc) return rc;
        CUDA_TRY(cudaMemsetAsync(d_unfinished, 0, 4, sc->stream));
        check(*kk);
        count_launch();
        CUDA_TRY(cudaGetLastError());
        uint32_t unfinished = 0;
        CUDA_TRY(cudaMemcpyAsync(&unfinished, d_unfinished, 4, cudaMemcpyDeviceToHost, sc->stream));
        CUDA_TRY(cudaStreamSynchronize(sc->stream));
        if (unfinished == 0 || *kk >= ix->n || *kk >= 16384) return 0;
        *kk *= 4;
    }
}

int svsb200_search_filtered(svsb200_index* ix, const void* queries, int qdtype, size_t nq, size_t k, size_t window,
                            const uint32_t* id_bitmap, uint64_t* out_ids, float* out_dists, uint32_t* out_found) {
    if (!ix) return fail("svsb200_search_filtered: NULL index");
    if (nq == 0) return 0;
    if (!queries || !id_bitmap || !out_ids || !out_dists) return fail("svsb200_search_filtered: NULL buffer");
    if (k == 0) return fail("k must be greater than 0");
    if (qdtype < SVSB200_F32 || qdtype > SVSB200_U8) return fail("bad query dtype");
    Replica* rep = ix->reps[0].get();
    ScratchLease lease;   // (declared first: returned after the buffers below are freed)
    if (int rc = lease.take(rep, nullptr)) return rc;
    Scratch* sc = lease.sc;
    DeviceBuffer<uint32_t> d_bitmap, d_found;
    DeviceBuffer<uint64_t> d_oi;
    DeviceBuffer<float> d_od;
    const size_t words = (ix->n + 31) / 32;
    const size_t qbytes = nq * ix->dim * esize(qdtype);
    CUDA_TRY(d_bitmap.ensure(words));
    CUDA_TRY(d_found.ensure(nq + 1));
    CUDA_TRY(d_oi.ensure(nq * k));
    CUDA_TRY(d_od.ensure(nq * k));
    CUDA_TRY(sc->q_raw.ensure(qbytes));
    CUDA_TRY(cudaMemcpyAsync(d_bitmap.ptr, id_bitmap, words * 4, cudaMemcpyHostToDevice, sc->stream));
    CUDA_TRY(cudaMemcpyAsync(sc->q_raw.ptr, queries, qbytes, cudaMemcpyHostToDevice, sc->stream));
    CUDA_TRY(cudaMemsetAsync(d_oi.ptr, 0xFF, nq * k * 8, sc->stream));
    // lists grow until every query has k members or its search is exhausted
    size_t kk = std::max(k, window);
    int rc = search_growing_lists(ix, rep, sc, qdtype, nq, window, d_found.ptr + nq, &kk, [&](size_t len) {
        filter_topk_kernel<<<unsigned((nq + 3) / 4), 128, 0, sc->stream>>>(
            reinterpret_cast<const uint64_t*>(sc->ids.ptr), sc->dists.ptr, uint32_t(nq), uint32_t(len), uint32_t(k),
            d_bitmap.ptr, d_oi.ptr, d_od.ptr, d_found.ptr, d_found.ptr + nq);
    });
    if (rc) return rc;
    std::vector<uint32_t> found(nq);
    CUDA_TRY(cudaMemcpyAsync(found.data(), d_found.ptr, nq * 4, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaMemcpyAsync(out_ids, d_oi.ptr, nq * k * 8, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaMemcpyAsync(out_dists, d_od.ptr, nq * k * 4, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    for (size_t q = 0; q < nq; ++q) {   // pad like the reference: unspecified id (all-ones), +inf distance
        for (size_t j = found[q]; j < k; ++j) {
            out_ids[q * k + j] = ~uint64_t(0);
            out_dists[q * k + j] = INFINITY;
        }
        if (out_found) out_found[q] = found[q];
    }
    return 0;
}

int svsb200_range_search(svsb200_index* ix, const void* queries, int qdtype, size_t nq, float radius, size_t window,
                         uint32_t* out_counts, uint64_t** out_ids, float** out_dists) {
    if (!ix) return fail("svsb200_range_search: NULL index");
    if (nq == 0) return 0;
    if (!queries || !out_counts || !out_ids || !out_dists) return fail("svsb200_range_search: NULL buffer");
    if (qdtype < SVSB200_F32 || qdtype > SVSB200_U8) return fail("bad query dtype");
    *out_ids = nullptr;
    *out_dists = nullptr;
    Replica* rep = ix->reps[0].get();
    ScratchLease lease;   // (declared first: returned after the buffer below is freed)
    if (int rc = lease.take(rep, nullptr)) return rc;
    Scratch* sc = lease.sc;
    DeviceBuffer<uint32_t> d_counts;
    const size_t qbytes = nq * ix->dim * esize(qdtype);
    CUDA_TRY(d_counts.ensure(nq + 1));
    CUDA_TRY(sc->q_raw.ensure(qbytes));
    CUDA_TRY(cudaMemcpyAsync(sc->q_raw.ptr, queries, qbytes, cudaMemcpyHostToDevice, sc->stream));
    // lists grow until every query's last result lies outside the radius or its search is exhausted
    size_t kk = std::max<size_t>(window, 16);
    int rc = search_growing_lists(ix, rep, sc, qdtype, nq, window, d_counts.ptr + nq, &kk, [&](size_t len) {
        range_count_kernel<<<unsigned((nq + 127) / 128), 128, 0, sc->stream>>>(
            sc->dists.ptr, reinterpret_cast<const uint64_t*>(sc->ids.ptr), uint32_t(nq), uint32_t(len), radius,
            ix->metric != SVSB200_L2, d_counts.ptr, d_counts.ptr + nq);
    });
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_counts, d_counts.ptr, nq * 4, cudaMemcpyDeviceToHost, sc->stream));
    std::vector<uint64_t> ids(nq * kk);
    std::vector<float> dd(nq * kk);
    CUDA_TRY(cudaMemcpyAsync(ids.data(), sc->ids.ptr, nq * kk * 8, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaMemcpyAsync(dd.data(), sc->dists.ptr, nq * kk * 4, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    size_t total = 0;
    for (size_t q = 0; q < nq; ++q) total += out_counts[q];
    uint64_t* oi = static_cast<uint64_t*>(malloc(std::max<size_t>(total, 1) * 8));
    float* od = static_cast<float*>(malloc(std::max<size_t>(total, 1) * 4));
    if (!oi || !od) {
        free(oi);
        free(od);
        return fail("svsb200_range_search: out of host memory");
    }
    size_t o = 0;
    for (size_t q = 0; q < nq; ++q)
        for (size_t j = 0; j < out_counts[q]; ++j, ++o) {
            oi[o] = ids[q * kk + j];
            od[o] = dd[q * kk + j];
        }
    *out_ids = oi;
    *out_dists = od;
    return 0;
}

void svsb200_free(void* p) { free(p); }

int svsb200_search_sharded(svsb200_index* const* shards, size_t nshards, const void* queries, int qdtype, size_t nq,
                           size_t k, size_t window, size_t capacity, uint64_t* out_ids, float* out_dists) {
    if (!shards || nshards == 0) return fail("svsb200_search_sharded: no shards");
    if (nshards > 1024) return fail("svsb200_search_sharded: at most 1024 shards");
    if (nq == 0) return 0;
    if (!queries || !out_ids || !out_dists) return fail("svsb200_search_sharded: NULL buffer");
    if (qdtype < SVSB200_F32 || qdtype > SVSB200_U8) return fail("bad query dtype");
    for (size_t s = 0; s < nshards; ++s) {
        if (!shards[s] || shards[s]->reps.size() != 1) return fail("svsb200_search_sharded: every shard is a single-device index");
        if (shards[s]->dim != shards[0]->dim || shards[s]->metric != shards[0]->metric)
            return fail("svsb200_search_sharded: shards disagree on dimension or metric");
    }
    const size_t qbytes = nq * shards[0]->dim * esize(qdtype);
    const size_t cnt = nq * k;
    std::vector<ScratchLease> scs(nshards);
    for (size_t s = 0; s < nshards; ++s) {
        if (int rc = scs[s].take(shards[s]->reps[0].get(), nullptr)) return rc;
    }
    // the merging device is shard 0's; its scratch holds the [nshards][nq][k] gather block
    Replica* rep0 = shards[0]->reps[0].get();
    Scratch* sc0 = scs[0].sc;
    auto body = [&]() -> int {
        CUDA_TRY(cudaSetDevice(rep0->device));
        CUDA_TRY(sc0->gather_ids.ensure(nshards * cnt));
        CUDA_TRY(sc0->gather_dists.ensure(nshards * cnt));
        CUDA_TRY(sc0->merged_ids.ensure(cnt));
        CUDA_TRY(sc0->merged_dists.ensure(cnt));
        for (size_t s = 0; s < nshards; ++s) {
            Replica* rep = shards[s]->reps[0].get();
            Scratch* sc = scs[s].sc;
            CUDA_TRY(cudaSetDevice(rep->device));
            CUDA_TRY(sc->q_raw.ensure(qbytes));
            CUDA_TRY(cudaMemcpyAsync(sc->q_raw.ptr, queries, qbytes, cudaMemcpyHostToDevice, sc->stream));
            // With peer access the shard's kernel writes its rows straight into the merging device's block over
            // NVLink (the gather is fused into the search kernel's copy-out); otherwise it writes locally and the
            // block is moved by a peer copy.
            bool direct = rep->device == rep0->device;
            if (!direct) {
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, rep->device, rep0->device) == cudaSuccess && can) {
                    cudaError_t pe = cudaDeviceEnablePeerAccess(rep0->device, 0);
                    direct = pe == cudaSuccess || pe == cudaErrorPeerAccessAlreadyEnabled;
                    cudaGetLastError();
                }
            }
            uint64_t* ids_dst = sc0->gather_ids.ptr + s * cnt;
            float* d_dst = sc0->gather_dists.ptr + s * cnt;
            if (!direct) {
                CUDA_TRY(sc->ids.ensure(cnt * 8));
                CUDA_TRY(sc->dists.ensure(cnt));
            }
            int rc = search_on_device(shards[s], rep, sc, sc->q_raw.ptr, qdtype, nq, k, window, capacity,
                                      direct ? static_cast<void*>(ids_dst) : static_cast<void*>(sc->ids.ptr), 8,
                                      direct ? d_dst : sc->dists.ptr, sc->stream);
            if (rc) return rc;
            CUDA_TRY(cudaEventRecord(sc->ev_done, sc->stream));
            if (s != 0) {
                CUDA_TRY(cudaSetDevice(rep0->device));
                CUDA_TRY(cudaStreamWaitEvent(sc0->stream, sc->ev_done, 0));
                if (!direct) {
                    CUDA_TRY(cudaMemcpyPeerAsync(ids_dst, rep0->device, sc->ids.ptr, rep->device, cnt * 8, sc0->stream));
                    CUDA_TRY(cudaMemcpyPeerAsync(d_dst, rep0->device, sc->dists.ptr, rep->device, cnt * 4, sc0->stream));
                }
            }
        }
        CUDA_TRY(cudaSetDevice(rep0->device));
        CUDA_TRY(launch_merge_topk(sc0->gather_ids.ptr, sc0->gather_dists.ptr, nshards, nq, k, shards[0]->metric != SVSB200_L2,
                                   sc0->merged_ids.ptr, sc0->merged_dists.ptr, sc0->stream));
        CUDA_TRY(cudaMemcpyAsync(out_ids, sc0->merged_ids.ptr, cnt * 8, cudaMemcpyDeviceToHost, sc0->stream));
        CUDA_TRY(cudaMemcpyAsync(out_dists, sc0->merged_dists.ptr, cnt * 4, cudaMemcpyDeviceToHost, sc0->stream));
        return 0;
    };
    int rc = body();
    const std::string first_error = g_error;
    int rc_wait = wait_all(scs);
    if (rc) {
        g_error = first_error;
        return rc;
    }
    return rc_wait;
}

static Scratch* last_scratch(svsb200_index* ix) {
    std::lock_guard<std::mutex> lock(ix->mu);
    return ix->last;
}

int svsb200_get_fetched(svsb200_index* ix, size_t nq, uint32_t* fetched) {
    if (!ix || !fetched) return fail("svsb200_get_fetched: NULL argument");
    Scratch* sc = last_scratch(ix);
    if (!ix->counting || !sc || sc->counted_nq < nq) return fail("svsb200_get_fetched: counting was not enabled for that many queries");
    CUDA_TRY(cudaSetDevice(sc->device));
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(fetched, sc->fetched.ptr, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return 0;
}

int svsb200_get_counters(svsb200_index* ix, size_t nq, uint32_t* hops, uint32_t* evals) {
    if (!ix) return fail("svsb200_get_counters: NULL index");
    Scratch* sc = last_scratch(ix);
    if (!ix->counting || !sc || sc->counted_nq < nq) return fail("svsb200_get_counters: counting was not enabled for that many queries");
    CUDA_TRY(cudaSetDevice(sc->device));
    CUDA_TRY(cudaDeviceSynchronize());
    if (hops) CUDA_TRY(cudaMemcpy(hops, sc->hops.ptr, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (evals) CUDA_TRY(cudaMemcpy(evals, sc->evals.ptr, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return 0;
}

int svsb200_last_kernel_ms(svsb200_index* ix, float* ms) {
    if (!ix || !ms) return fail("svsb200_last_kernel_ms: NULL argument");
    Scratch* sc = last_scratch(ix);
    if (!sc || !sc->timed) return fail("svsb200_last_kernel_ms: no search has run yet");
    CUDA_TRY(cudaSetDevice(sc->device));
    CUDA_TRY(cudaEventSynchronize(sc->ev_stop));
    CUDA_TRY(cudaEventElapsedTime(ms, sc->ev_start, sc->ev_stop));
    return 0;
}

int svsb200_merge_topk_device(const uint64_t* d_ids, const float* d_dists, size_t nshards, size_t nq, size_t k, int metric,
                              uint64_t* d_out_ids, float* d_out_dists, int device, void* stream) {
    if (nshards == 0 || nshards > 1024) return fail("svsb200_merge_topk_device: 1..1024 shards supported");
    if (nq == 0 || k == 0) return 0;
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(launch_merge_topk(d_ids, d_dists, nshards, nq, k, metric != SVSB200_L2, d_out_ids, d_out_dists,
                               static_cast<cudaStream_t>(stream)));
    return 0;
}

size_t svsb200_lvq8_row_stride(size_t dim) { return round_up(round_up(dim, 4) + 4, 32); }

int svsb200_lvq8_compress(const float* data, size_t n, size_t dim, const float* mean, void* out_rows, int device) {
    if (!data || !mean || !out_rows) return fail("svsb200_lvq8_compress: NULL argument");
    if (n == 0 || dim == 0 || n >= (size_t(1) << 31)) return fail("svsb200_lvq8_compress: bad shape");
    if (svsb200_device_count() == 0) return fail("svsb200_lvq8_compress: no CUDA device (there is no CPU fallback)");
    CUDA_TRY(cudaSetDevice(device));
    const size_t stride = svsb200_lvq8_row_stride(dim);
    DeviceBuffer<float> d_data, d_mean;
    DeviceBuffer<uint8_t> d_rows;
    CUDA_TRY(d_data.ensure(n * dim));
    CUDA_TRY(d_mean.ensure(dim));
    CUDA_TRY(d_rows.ensure(n * stride));
    CUDA_TRY(cudaMemcpy(d_data.ptr, data, n * dim * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_mean.ptr, mean, dim * sizeof(float), cudaMemcpyHostToDevice));
    const int warps = 8;
    lvq8_compress_kernel<<<unsigned((n + warps - 1) / warps), warps * 32>>>(d_data.ptr, uint32_t(n), uint32_t(dim), d_mean.ptr,
                                                                          d_rows.ptr, uint32_t(stride),
                                                                          uint32_t(round_up(dim, 4)));
    count_launch();
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(out_rows, d_rows.ptr, n * stride, cudaMemcpyDeviceToHost));
    return 0;
}

// Shared body of the tensor-core flat search: device buffers in, device buffers out, enqueued on sc->stream except
// for one synchronisation (the count of queries that need the exact-scan fallback).
static int flat_on_device(svsb200_index* ix, Replica* rep, Scratch* sc, const void* d_queries, int qdtype, size_t nq, size_t k,
                          uint64_t* d_out_ids, float* d_out_dists, uint32_t* fallback_queries) {
    if (fallback_queries) *fallback_queries = 0;
    if (nq == 0) return 0;
    cudaStream_t stream = sc->stream;
    const bool gemm_ok = ix->storage == SVSB200_PLAIN && (ix->dtype == SVSB200_F32 || ix->dtype == SVSB200_F16) &&
                         ix->metric != SVSB200_COSINE && (qdtype == SVSB200_F32 || qdtype == SVSB200_F16) &&
                         k + 8 <= flat_kc() && ix->n >= 512;
    if (!gemm_ok) {   // shapes outside the GEMM path: the exact scan
        if (fallback_queries) *fallback_queries = uint32_t(nq);
        return search_on_device(ix, rep, sc, d_queries, qdtype, nq, k, k, k, d_out_ids, 8, d_out_dists, stream, true);
    }
    const uint32_t n = uint32_t(ix->n), dim = uint32_t(ix->dim);
    const uint32_t KB = (dim + 31) / 32, ntiles = (n + 255) / 256, mtiles = uint32_t((nq + 127) / 128);
    const int l2 = ix->metric == SVSB200_L2;
    {   // base tiles, once per replica
        std::lock_guard<std::mutex> lock(rep->mu);
        if (!rep->flat_b.ptr) {
            CUDA_TRY(rep->flat_b.ensure(size_t(ntiles) * 256 * KB * 32 * 2));
            CUDA_TRY(rep->flat_bias.ensure(size_t(ntiles) * 256));
            CUDA_TRY(rep->flat_xmax.ensure(1));
            CUDA_TRY(cudaMemsetAsync(rep->flat_xmax.ptr, 0, 4, stream));
            CUDA_TRY(flat_tile_rows(ix->dtype, rep->d_vectors.ptr, ix->row_stride, n, dim, 256, 1.0f, l2, rep->flat_b.ptr,
                                    rep->flat_bias.ptr, nullptr, rep->flat_xmax.ptr, stream));
            CUDA_TRY(cudaStreamSynchronize(stream));
        }
    }
    // one CTA per SM over equal runs of output tiles; `nsplit` = candidate lists per query (flat.cu: flat_plan)
    uint32_t flat_ctas = 1, flat_share = 1, nsplit = 2;
    flat_plan(mtiles, ntiles, uint32_t(rep->sm_count), &flat_ctas, &flat_share, &nsplit);
    const size_t qrow = size_t(dim) * esize(qdtype);
    CUDA_TRY(sc->flat_a.ensure(size_t(mtiles) * 128 * KB * 32 * 2));
    CUDA_TRY(sc->flat_qnorm.ensure(size_t(mtiles) * 128));
    CUDA_TRY(sc->flat_ckey.ensure(size_t(mtiles) * 128 * nsplit * flat_kc()));
    CUDA_TRY(sc->flat_cid.ensure(size_t(mtiles) * 128 * nsplit * flat_kc()));
    CUDA_TRY(sc->flat_unv.ensure(nq + 1));
    CUDA_TRY(sc->flat_progress.ensure(flat_ctas));
    CUDA_TRY(cudaMemsetAsync(sc->flat_progress.ptr, 0, size_t(flat_ctas) * 4, stream));
    CUDA_TRY(flat_tile_rows(qdtype, d_queries, uint32_t(qrow), uint32_t(nq), dim, 128, 1.0f, 0, sc->flat_a.ptr, nullptr,
                            sc->flat_qnorm.ptr, nullptr, stream));
    CUDA_TRY(flat_gemm_topk(sc->flat_a.ptr, rep->flat_b.ptr, rep->flat_bias.ptr, KB, ntiles, mtiles, flat_ctas, flat_share, nsplit, l2 ? -2.0f : -1.0f,
                            sc->flat_ckey.ptr, sc->flat_cid.ptr, sc->flat_progress.ptr, stream));
    // exact re-scoring with the search path's distance code: prepared queries as for a search
    if (int rc = prepare_queries(ix, rep, sc, d_queries, qdtype, nq, PREP_FLOAT, stream)) return rc;
    SearchParams p{};
    p.vectors = rep->d_vectors.ptr;
    p.n = n;
    p.dim = dim;
    p.row_stride = ix->row_stride;
    p.greater = !l2;
    p.scale = 1.f;
    p.qf = sc->q_f32.ptr;
    p.qaux = sc->q_aux.ptr;
    p.qstride = qstride_for(dim);
    p.nq = uint32_t(nq);
    p.k = uint32_t(k);
    CUDA_TRY(cudaMemsetAsync(sc->flat_unv.ptr, 0, 4, stream));
    // rounding terms of E(q) (flat.cu header): the query is always rounded to fp16, float32 data too
    p.scale = (qdtype == SVSB200_F32 ? 1.0f : 0.0f) + (ix->dtype == SVSB200_F32 ? 1.0f : 0.0f);   // number of rounded operands
    CUDA_TRY(flat_rescore(ix->dtype, l2 ? OP_L2F : OP_IPF, p, sc->flat_ckey.ptr, sc->flat_cid.ptr, nsplit, uint32_t(nq), uint32_t(k),
                          sc->flat_qnorm.ptr, rep->flat_xmax.ptr, d_out_ids, d_out_dists, sc->flat_unv.ptr + 1, sc->flat_unv.ptr, stream));
    // queries whose bound did not verify: exact scan, results scattered over the rescored rows
    uint32_t nunv = 0;
    CUDA_TRY(cudaMemcpyAsync(&nunv, sc->flat_unv.ptr, 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    if (fallback_queries) *fallback_queries = nunv;
    if (nunv) {
        CUDA_TRY(sc->flat_q2.ensure(size_t(nunv) * qrow));
        CUDA_TRY(sc->flat_i2.ensure(size_t(nunv) * k));
        CUDA_TRY(sc->flat_d2.ensure(size_t(nunv) * k));
        CUDA_TRY(flat_move_rows(d_queries, sc->flat_q2.ptr, sc->flat_unv.ptr + 1, sc->flat_unv.ptr, nunv, uint32_t(qrow), 0, stream));
        int rc = search_on_device(ix, rep, sc, sc->flat_q2.ptr, qdtype, nunv, k, k, k, sc->flat_i2.ptr, 8, sc->flat_d2.ptr, stream, true);
        if (rc) return rc;
        CUDA_TRY(flat_move_rows(sc->flat_i2.ptr, d_out_ids, sc->flat_unv.ptr + 1, sc->flat_unv.ptr, nunv, uint32_t(k * 8), 1, stream));
        CUDA_TRY(flat_move_rows(sc->flat_d2.ptr, d_out_dists, sc->flat_unv.ptr + 1, sc->flat_unv.ptr, nunv, uint32_t(k * 4), 1, stream));
    }
    return 0;
}

int svsb200_flat_search_device(svsb200_index* ix, const void* d_queries, int qdtype, size_t nq, size_t k, uint64_t* d_out_ids,
                               float* d_out_dists, void* stream_, uint32_t* fallback_queries) {
    if (!ix) return fail("svsb200_flat_search_device: NULL index");
    if (nq && (!d_queries || !d_out_ids || !d_out_dists)) return fail("svsb200_flat_search_device: NULL buffer");
    if (k == 0 || k > 1024) return fail("svsb200_flat_search_device: k must be in [1, 1024]");
    if (qdtype < SVSB200_F32 || qdtype > SVSB200_U8) return fail("bad query dtype");
    Scratch* sc = nullptr;
    if (int rc = device_api_scratch("svsb200_flat_search_device", ix, stream_, &sc)) return rc;
    return flat_on_device(ix, ix->reps[0].get(), sc, d_queries, qdtype, nq, k, d_out_ids, d_out_dists, fallback_queries);
}

int svsb200_flat_search(svsb200_index* ix, const void* queries, int qdtype, size_t nq, size_t k, uint64_t* out_ids,
                        float* out_dists) {
    if (!ix) return fail("svsb200_flat_search: NULL index");
    if (nq == 0) return 0;
    if (!queries || !out_ids || !out_dists) return fail("svsb200_flat_search: NULL buffer");
    if (k == 0 || k > 1024) return fail("svsb200_flat_search: k must be in [1, 1024]");
    if (qdtype < SVSB200_F32 || qdtype > SVSB200_U8) return fail("bad query dtype");
    Replica* rep = ix->reps[0].get();
    ScratchLease lease;
    if (int rc = lease.take(rep, nullptr)) return rc;
    Scratch* sc = lease.sc;
    const size_t qbytes = nq * ix->dim * esize(qdtype);
    CUDA_TRY(sc->q_raw.ensure(qbytes));
    CUDA_TRY(sc->ids.ensure(nq * k * 8));
    CUDA_TRY(sc->dists.ensure(nq * k));
    CUDA_TRY(cudaMemcpyAsync(sc->q_raw.ptr, queries, qbytes, cudaMemcpyHostToDevice, sc->stream));
    int rc = flat_on_device(ix, rep, sc, sc->q_raw.ptr, qdtype, nq, k, reinterpret_cast<uint64_t*>(sc->ids.ptr), sc->dists.ptr,
                            nullptr);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_ids, sc->ids.ptr, nq * k * 8, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaMemcpyAsync(out_dists, sc->dists.ptr, nq * k * 4, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    return 0;
}

int svsb200_exhaustive_device(svsb200_index* ix, const void* d_queries, int qdtype, size_t nq, size_t k, uint64_t* d_out_ids,
                              float* d_out_dists, void* stream_) {
    if (!ix) return fail("svsb200_exhaustive_device: NULL index");
    if (nq && (!d_queries || !d_out_ids || !d_out_dists)) return fail("svsb200_exhaustive_device: NULL buffer");
    if (k == 0 || k > 1024) return fail("svsb200_exhaustive_device: k must be in [1, 1024]");
    Scratch* sc = nullptr;
    if (int rc = device_api_scratch("svsb200_exhaustive_device", ix, stream_, &sc)) return rc;
    return search_on_device(ix, ix->reps[0].get(), sc, d_queries, qdtype, nq, k, k, k, d_out_ids, 8, d_out_dists, sc->stream, true);
}

}  // extern "C"
