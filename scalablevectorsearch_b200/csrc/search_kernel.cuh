// search_kernel.cuh -- the Vamana batched greedy search as one persistent sm_100a kernel.
//
// Replaces, for a whole query batch (file:line under /root/reference/include/svs):
//   index/vamana/index.h:564-611        VamanaIndex::search       (thread pool -> grid)
//   index/vamana/greedy_search.h:124-203 greedy_search            (one warp per query)
//   index/vamana/search_buffer.h:104-497 SearchBuffer             (sorted buffer in smem)
//   core/distance/simd_utils.h:204-252   generic_simd_op + L2/IP/Cosine ops (bit-exact)
//
// Mapping
//   * one warp owns one query at a time and pulls query indices from a global counter
//     (persistent CTAs, grid = SMs x resident CTAs);
//   * per expanded node the warp reads the adjacency row (coalesced), then evaluates the
//     neighbours' distances GROUPS rows at a time: a row is owned by G = 16/LPT adjacent
//     threads, thread t of the group holding logical AVX-512 lanes [LPT*t, LPT*t+LPT) of
//     every 16-element chunk, so each thread issues 128-bit (f32/f16) loads of its own
//     row and keeps the reference's 16-lane x 4-accumulator FMA tree entirely in
//     registers; the 8/4/2/1 reduction is two xor-shuffle levels plus in-thread adds;
//   * the <= max_degree candidates of a node are then merged into the sorted buffer in one
//     step.  The merge reproduces the result of the reference's sequential
//     `for id in neighbours: buffer.insert(...)` exactly (DESIGN.md §merge): stable order
//     (new after equal old, adjacency order among equal new), duplicate-id rejection over
//     the equal-distance run, truncation at capacity, and the best-unvisited cursor.
#pragma once

#include "common.cuh"

namespace svsb200 {

// ---------------------------------------------------------------------------------------
// Row access: how one thread fetches its LPT lanes of one 16-element chunk.
// ---------------------------------------------------------------------------------------
template <int ROWT> struct Row;

template <> struct Row<SVSB200_F32> {
    static constexpr int LPT = 4, ESIZE = 4;
    using raw_t = float4;
    __device__ static __forceinline__ raw_t load(const char* p) {
        return __ldg(reinterpret_cast<const float4*>(p));
    }
    __device__ static __forceinline__ void cvt(const raw_t& r, float (&y)[4]) {
        y[0] = r.x; y[1] = r.y; y[2] = r.z; y[3] = r.w;
    }
};
template <> struct Row<SVSB200_F16> {
    static constexpr int LPT = 8, ESIZE = 2;
    using raw_t = uint4;
    __device__ static __forceinline__ raw_t load(const char* p) {
        return __ldg(reinterpret_cast<const uint4*>(p));
    }
    __device__ static __forceinline__ void cvt(const raw_t& r, float (&y)[8]) {
        // __half2float is exact and honours subnormals, like vcvtph2ps (simd_utils.h:270).
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
            y[2 * i] = __low2float(h);
            y[2 * i + 1] = __high2float(h);
        }
    }
};
template <> struct Row<SVSB200_I8> {
    static constexpr int LPT = 8, ESIZE = 1;
    using raw_t = uint2;
    __device__ static __forceinline__ raw_t load(const char* p) {
        return __ldg(reinterpret_cast<const uint2*>(p));
    }
    __device__ static __forceinline__ void cvt(const raw_t& r, float (&y)[8]) {
        const uint32_t w[2] = {r.x, r.y};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            y[i] = float(int(int8_t((w[i >> 2] >> (8 * (i & 3))) & 0xFF)));
        }
    }
};
template <> struct Row<SVSB200_U8> {
    static constexpr int LPT = 8, ESIZE = 1;
    using raw_t = uint2;
    __device__ static __forceinline__ raw_t load(const char* p) {
        return __ldg(reinterpret_cast<const uint2*>(p));
    }
    __device__ static __forceinline__ void cvt(const raw_t& r, float (&y)[8]) {
        const uint32_t w[2] = {r.x, r.y};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            y[i] = float((w[i >> 2] >> (8 * (i & 3))) & 0xFF);
        }
    }
};

// LVQ-8 rows: uint8 codes; decompression y = fma(delta, code, lower) happens in float_rows.
template <> struct Row<ROW_LVQ8> : Row<SVSB200_U8> {};

// Fire-and-forget L2 prefetch: costs no registers, so the bytes in flight per warp are not
// bounded by the register file; the later 128-bit loads then hit L2 instead of HBM.
__device__ __forceinline__ void prefetch_l2(const void* p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// One accumulate step of the op (euclidean.h:247-250, inner_product.h:206-208,
// cosine.h:238-241).  Explicit _rn intrinsics: never contracted, never reordered.
template <int OP> __device__ __forceinline__ void accumulate(float& s, float& nrm, float x, float y) {
    if constexpr (OP == OP_L2F) {
        float c = __fsub_rn(x, y);
        s = __fmaf_rn(c, c, s);
    } else {
        s = __fmaf_rn(x, y, s);
        if constexpr (OP == OP_COSF) {
            nrm = __fmaf_rn(y, y, nrm);
        }
    }
}

// Blackwell packs two IEEE fp32 operations into one instruction (PTX add/sub/fma.rn.f32x2 ->
// SASS FADD2 / FFMA2): each half rounds exactly like the scalar _rn form, so the expression
// tree -- and every bit of the result -- is unchanged while the FP instruction count halves.
__device__ __forceinline__ float2 fsub2_rn(float2 a, float2 b) {
    unsigned long long d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 fadd2_rn(float2 a, float2 b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 ffma2_rn(float2 a, float2 b, float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)), "l"(*reinterpret_cast<unsigned long long*>(&c)));
    return *reinterpret_cast<float2*>(&d);
}
template <int OP> __device__ __forceinline__ void accumulate2(float2& s, float2& nrm, float2 x, float2 y) {
    if constexpr (OP == OP_L2F) {
        float2 c = fsub2_rn(x, y);
        s = ffma2_rn(c, c, s);
    } else {
        s = ffma2_rn(x, y, s);
        if constexpr (OP == OP_COSF) {
            nrm = ffma2_rn(y, y, nrm);
        }
    }
}

// _mm512_reduce_add_ps over the 16 logical lanes spread across the G threads of a group.
template <int LPT> __device__ __forceinline__ float reduce_lanes(float (&s)[LPT]) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    if constexpr (LPT == 4) {
        // lanes L and L+8 live in threads t and t^2, same slot.
        float v[4], w[4];
#pragma unroll
        for (int l = 0; l < 4; ++l) v[l] = __fadd_rn(__shfl_xor_sync(FULL, s[l], 2), s[l]);
        // lanes L and L+4 (L<4) live in threads 0 and 1.
#pragma unroll
        for (int l = 0; l < 4; ++l) w[l] = __fadd_rn(__shfl_xor_sync(FULL, v[l], 1), v[l]);
        return __fadd_rn(__fadd_rn(w[0], w[2]), __fadd_rn(w[1], w[3]));
    } else {
        static_assert(LPT == 8, "unsupported lane split");
        float v[8], w[4];
#pragma unroll
        for (int l = 0; l < 8; ++l) v[l] = __fadd_rn(__shfl_xor_sync(FULL, s[l], 1), s[l]);
#pragma unroll
        for (int l = 0; l < 4; ++l) w[l] = __fadd_rn(v[l + 4], v[l]);
        return __fadd_rn(__fadd_rn(w[0], w[2]), __fadd_rn(w[1], w[3]));
    }
}

// ---------------------------------------------------------------------------------------
// Float-tree distance of NROWS rows against the query staged in shared memory.
//   rowp[r]   this thread group's row base pointers (nullptr = inactive slot)
//   t         thread index inside the group
// Returns the *raw* reduced sums (op, norm) -- identical in every thread of the group.
// ---------------------------------------------------------------------------------------
template <int ROWT, int OP, int DS, int NROWS, bool DENSE = false>
__device__ __forceinline__ void float_rows(
    const SearchParams& p, const float* __restrict__ q_s, const char* const (&rowp)[NROWS], int t,
    float (&sum)[NROWS], float (&nrm)[NROWS]) {
    using R = Row<ROWT>;
    constexpr int LPT = R::LPT;
    const int D = DS ? DS : int(p.dim);
    const bool sqcos = (OP == OP_COSF) && p.sq;
    // LVQ-8: per-vector constants, two float16 right behind the codes.
    float lvq_delta[NROWS], lvq_lower[NROWS];
    if constexpr (ROWT == ROW_LVQ8) {
#pragma unroll
        for (int r = 0; r < NROWS; ++r) {
            lvq_delta[r] = 0.f;
            lvq_lower[r] = 0.f;
            if (DENSE || rowp[r]) {
                const uint32_t c = __ldg(reinterpret_cast<const uint32_t*>(rowp[r] + p.lvq_const_offset));
                const __half2 h = *reinterpret_cast<const __half2*>(&c);
                lvq_delta[r] = __low2float(h);
                lvq_lower[r] = __high2float(h);
            }
        }
    }
    // element as the distance tree sees it
    auto element = [&](int r, float y) -> float {
        if constexpr (ROWT == ROW_LVQ8) {
            return __fmaf_rn(lvq_delta[r], y, lvq_lower[r]);
        } else {
            return sqcos ? __fadd_rn(__fmul_rn(p.scale, y), p.bias) : y;
        }
    };

    constexpr int HP = LPT / 2;   // lane pairs: packed f32x2 arithmetic
    float2 s[NROWS][4][HP];
    float2 n[NROWS][4][HP];
#pragma unroll
    for (int r = 0; r < NROWS; ++r)
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int l = 0; l < HP; ++l) {
                s[r][k][l] = make_float2(0.0f, 0.0f);
                n[r][k][l] = make_float2(0.0f, 0.0f);
            }

    const int thread_elem = LPT * t;                 // first element of this thread in a chunk
    const int nblk = D >> 6;                         // 64-element main blocks
    int base = 0;                                    // element offset of the current chunk group
#pragma unroll(DS ? 16 : 1)
    for (int b = 0; b < nblk; ++b, base += 64) {
        typename R::raw_t raw[NROWS][4];
#pragma unroll
        for (int r = 0; r < NROWS; ++r)
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (DENSE || rowp[r]) raw[r][k] = R::load(rowp[r] + size_t(base + 16 * k + thread_elem) * R::ESIZE);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float x[LPT];
#pragma unroll
            for (int l = 0; l < LPT; l += 4) {
                float4 qv = *reinterpret_cast<const float4*>(q_s + base + 16 * k + thread_elem + l);
                x[l] = qv.x; x[l + 1] = qv.y; x[l + 2] = qv.z; x[l + 3] = qv.w;
            }
#pragma unroll
            for (int r = 0; r < NROWS; ++r) {
                if (!DENSE && !rowp[r]) continue;
                float y[LPT];
                R::cvt(raw[r][k], y);
#pragma unroll
                for (int l = 0; l < HP; ++l) {
                    accumulate2<OP>(s[r][k][l], n[r][k][l], make_float2(x[2 * l], x[2 * l + 1]),
                                    make_float2(element(r, y[2 * l]), element(r, y[2 * l + 1])));
                }
            }
        }
    }
    if (nblk > 0) {
        // s0 = (s0 + s1) + (s2 + s3)   (simd_utils.h:238)
#pragma unroll
        for (int r = 0; r < NROWS; ++r)
#pragma unroll
            for (int l = 0; l < HP; ++l) {
                s[r][0][l] = fadd2_rn(fadd2_rn(s[r][0][l], s[r][1][l]), fadd2_rn(s[r][2][l], s[r][3][l]));
                if constexpr (OP == OP_COSF)
                    n[r][0][l] = fadd2_rn(fadd2_rn(n[r][0][l], n[r][1][l]), fadd2_rn(n[r][2][l], n[r][3][l]));
            }
    }
    // Up to three full 16-wide chunks plus one masked remainder, all into s0, in order
    // (simd_utils.h:242-250).  Elements >= D are inactive lanes: the accumulator is kept.
    if (base < D) {
        typename R::raw_t raw[NROWS][4];
#pragma unroll
        for (int r = 0; r < NROWS; ++r)
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if ((DENSE || rowp[r]) && base + 16 * k + thread_elem < D)
                    raw[r][k] = R::load(rowp[r] + size_t(base + 16 * k + thread_elem) * R::ESIZE);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int e0 = base + 16 * k + thread_elem;
            if (e0 < D) {
                float x[LPT];
#pragma unroll
                for (int l = 0; l < LPT; l += 4) {
                    float4 qv = *reinterpret_cast<const float4*>(q_s + e0 + l);
                    x[l] = qv.x; x[l + 1] = qv.y; x[l + 2] = qv.z; x[l + 3] = qv.w;
                }
#pragma unroll
                for (int r = 0; r < NROWS; ++r) {
                    if (!DENSE && !rowp[r]) continue;
                    float y[LPT];
                    R::cvt(raw[r][k], y);
#pragma unroll
                    for (int l = 0; l < HP; ++l) {
                        if (e0 + 2 * l + 1 < D) {
                            accumulate2<OP>(s[r][0][l], n[r][0][l], make_float2(x[2 * l], x[2 * l + 1]),
                                            make_float2(element(r, y[2 * l]), element(r, y[2 * l + 1])));
                        } else if (e0 + 2 * l < D) {   // odd dimension: only the low half is a live lane
                            accumulate<OP>(s[r][0][l].x, n[r][0][l].x, x[2 * l], element(r, y[2 * l]));
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < NROWS; ++r) {
        float sl[LPT], nl[LPT];
#pragma unroll
        for (int l = 0; l < HP; ++l) {
            sl[2 * l] = s[r][0][l].x;
            sl[2 * l + 1] = s[r][0][l].y;
            nl[2 * l] = n[r][0][l].x;
            nl[2 * l + 1] = n[r][0][l].y;
        }
        sum[r] = reduce_lanes<LPT>(sl);
        if constexpr (OP == OP_COSF) nrm[r] = reduce_lanes<LPT>(nl);
    }
}

// ---------------------------------------------------------------------------------------
// Wide rows (dim >= 256).  The four accumulators s0..s3 of the main loop are independent fma
// chains until the single combine (s0+s1)+(s2+s3), so a row is spread over 4 x G threads:
// thread (kk, tl) owns accumulator kk of lanes [LPT*tl, LPT*tl+LPT) and reads only the
// chunks 4b+kk.  Four times more threads per row = four times shorter dependent chains and
// finer-grained passes when only a handful of (large) rows pass the visited filter.
// Same expression tree, same bits.
// ---------------------------------------------------------------------------------------
template <int ROWT, int OP, int NROWS, bool DENSE = false>
__device__ __forceinline__ void float_rows_split(
    const SearchParams& p, const float* __restrict__ q_s, const char* const (&rowp)[NROWS], int t,
    float (&sum)[NROWS], float (&nrm)[NROWS]) {
    using R = Row<ROWT>;
    constexpr int LPT = R::LPT;
    constexpr int G = 16 / LPT;
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const int tl = t % G, kk = t / G;
    const int D = int(p.dim);
    const bool sqcos = (OP == OP_COSF) && p.sq;
    float lvq_delta[NROWS], lvq_lower[NROWS];
    if constexpr (ROWT == ROW_LVQ8) {
#pragma unroll
        for (int r = 0; r < NROWS; ++r) {
            lvq_delta[r] = 0.f;
            lvq_lower[r] = 0.f;
            if (DENSE || rowp[r]) {
                const uint32_t c = __ldg(reinterpret_cast<const uint32_t*>(rowp[r] + p.lvq_const_offset));
                const __half2 h = *reinterpret_cast<const __half2*>(&c);
                lvq_delta[r] = __low2float(h);
                lvq_lower[r] = __high2float(h);
            }
        }
    }
    auto element = [&](int r, float y) -> float {
        if constexpr (ROWT == ROW_LVQ8) {
            return __fmaf_rn(lvq_delta[r], y, lvq_lower[r]);
        } else {
            return sqcos ? __fadd_rn(__fmul_rn(p.scale, y), p.bias) : y;
        }
    };
    constexpr int HP = LPT / 2;   // lane pairs: packed f32x2 arithmetic (same bits, see accumulate2)
    float2 s[NROWS][HP], n[NROWS][HP];
#pragma unroll
    for (int r = 0; r < NROWS; ++r)
#pragma unroll
        for (int l = 0; l < HP; ++l) {
            s[r][l] = make_float2(0.0f, 0.0f);
            n[r][l] = make_float2(0.0f, 0.0f);
        }
    const int thread_elem = LPT * tl;
    const int nblk = D >> 6;
    auto step = [&](const typename R::raw_t (&raw)[NROWS], int e0, int limit) {
        float x[LPT];
#pragma unroll
        for (int l = 0; l < LPT; l += 4) {
            float4 qv = *reinterpret_cast<const float4*>(q_s + e0 + l);
            x[l] = qv.x; x[l + 1] = qv.y; x[l + 2] = qv.z; x[l + 3] = qv.w;
        }
#pragma unroll
        for (int r = 0; r < NROWS; ++r) {
            if (!DENSE && !rowp[r]) continue;
            float y[LPT];
            R::cvt(raw[r], y);
#pragma unroll
            for (int l = 0; l < HP; ++l) {
                if (e0 + 2 * l + 1 < limit) {
                    accumulate2<OP>(s[r][l], n[r][l], make_float2(x[2 * l], x[2 * l + 1]),
                                    make_float2(element(r, y[2 * l]), element(r, y[2 * l + 1])));
                } else if (e0 + 2 * l < limit) {   // odd dimension: only the low half is a live lane
                    accumulate<OP>(s[r][l].x, n[r][l].x, x[2 * l], element(r, y[2 * l]));
                }
            }
        }
    };
    // main loop: this thread's accumulator sees chunks kk, kk+4, kk+8, ... in order;
    // four blocks of loads are put in flight before they are consumed.
    int b = 0;
    for (; b + 4 <= nblk; b += 4) {
        typename R::raw_t raw[4][NROWS];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int r = 0; r < NROWS; ++r)
                if (DENSE || rowp[r]) raw[u][r] = R::load(rowp[r] + size_t((b + u) * 64 + 16 * kk + thread_elem) * R::ESIZE);
#pragma unroll
        for (int u = 0; u < 4; ++u) step(raw[u], (b + u) * 64 + 16 * kk + thread_elem, D);
    }
    for (; b < nblk; ++b) {
        typename R::raw_t raw[NROWS];
#pragma unroll
        for (int r = 0; r < NROWS; ++r)
            if (DENSE || rowp[r]) raw[r] = R::load(rowp[r] + size_t(b * 64 + 16 * kk + thread_elem) * R::ESIZE);
        step(raw, b * 64 + 16 * kk + thread_elem, D);
    }
    if (nblk > 0) {
        // s0 = (s0 + s1) + (s2 + s3): partners kk^1 then kk^2 (fp add is commutative)
#pragma unroll
        for (int r = 0; r < NROWS; ++r)
#pragma unroll
            for (int l = 0; l < HP; ++l) {
                auto xchg = [&](float2 v, int d) {
                    return make_float2(__shfl_xor_sync(FULL, v.x, d), __shfl_xor_sync(FULL, v.y, d));
                };
                float2 v = fadd2_rn(s[r][l], xchg(s[r][l], G));
                s[r][l] = fadd2_rn(v, xchg(v, 2 * G));
                if constexpr (OP == OP_COSF) {
                    float2 w = fadd2_rn(n[r][l], xchg(n[r][l], G));
                    n[r][l] = fadd2_rn(w, xchg(w, 2 * G));
                }
            }
    }
    // tail chunks go into s0 in order; every kk replica computes the same values
    for (int e = nblk * 64; e < D; e += 16) {
        typename R::raw_t raw[NROWS];
        const int e0 = e + thread_elem;
#pragma unroll
        for (int r = 0; r < NROWS; ++r)
            if ((DENSE || rowp[r]) && e0 < D) raw[r] = R::load(rowp[r] + size_t(e0) * R::ESIZE);
        if (e0 < D) step(raw, e0, D);
    }
#pragma unroll
    for (int r = 0; r < NROWS; ++r) {
        float sl[LPT], nl[LPT];
#pragma unroll
        for (int l = 0; l < HP; ++l) {
            sl[2 * l] = s[r][l].x;
            sl[2 * l + 1] = s[r][l].y;
            nl[2 * l] = n[r][l].x;
            nl[2 * l + 1] = n[r][l].y;
        }
        sum[r] = reduce_lanes<LPT>(sl);
        if constexpr (OP == OP_COSF) nrm[r] = reduce_lanes<LPT>(nl);
    }
}

// Exact integer sums for (int8,int8)/(uint8,uint8): groups of 4 threads, 16-byte loads,
// dp4a.  Order-free (integer), so any lane split is bit-exact.
template <int ROWT, int NROWS, bool DENSE = false>
__device__ __forceinline__ void int_rows(
    const SearchParams& p, const uint8_t* __restrict__ q_s, const char* const (&rowp)[NROWS], int t,
    int (&xy)[NROWS], int (&yy)[NROWS]) {
    const int nvec = (int(p.dim) + 15) >> 4;   // rows and query are zero-padded to 16 bytes
#pragma unroll
    for (int r = 0; r < NROWS; ++r) {
        xy[r] = 0;
        yy[r] = 0;
    }
    for (int v = t; v < nvec; v += 4) {
        uint4 qv = *reinterpret_cast<const uint4*>(q_s + 16 * v);
        const uint32_t qw[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
        for (int r = 0; r < NROWS; ++r) {
            if (!DENSE && !rowp[r]) continue;
            uint4 rv = __ldg(reinterpret_cast<const uint4*>(rowp[r] + 16 * v));
            const uint32_t rw[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if constexpr (ROWT == SVSB200_I8) {
                    xy[r] = __dp4a(int(qw[i]), int(rw[i]), xy[r]);
                    yy[r] = __dp4a(int(rw[i]), int(rw[i]), yy[r]);
                } else {
                    xy[r] = int(__dp4a(qw[i], rw[i], unsigned(xy[r])));
                    yy[r] = int(__dp4a(rw[i], rw[i], unsigned(yy[r])));
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < NROWS; ++r) {
        xy[r] += __shfl_xor_sync(0xFFFFFFFFu, xy[r], 2);
        xy[r] += __shfl_xor_sync(0xFFFFFFFFu, xy[r], 1);
        yy[r] += __shfl_xor_sync(0xFFFFFFFFu, yy[r], 2);
        yy[r] += __shfl_xor_sync(0xFFFFFFFFu, yy[r], 1);
    }
}

// Final scalar expression of each distance functor (after the reduction).
template <int OP>
__device__ __forceinline__ float finish_distance(const SearchParams& p, float sum, float nrm, int ixy, int iyy,
                                                 float aux0, float aux1) {
    if constexpr (OP == OP_L2F) {
        return sum;
    } else if constexpr (OP == OP_IPF) {
        // InnerProductCompressed::compute: scale * ip + offset (scalar.h:139-141).
        // LVQ-8: the rows are stored mean-removed, so <q, x> = <q, y> + <q, mean> (aux0).
        return p.sq ? __fadd_rn(__fmul_rn(p.scale, sum), aux0) : (p.lvq ? __fadd_rn(sum, aux0) : sum);
    } else if constexpr (OP == OP_COSF) {
        // cosine.h:334-335: sum / (sqrt(norm) * a_norm)
        return __fdiv_rn(sum, __fmul_rn(__fsqrt_rn(nrm), aux0));
    } else if constexpr (OP == OP_L2I) {
        // sum (x-y)^2 = xx - 2xy + yy, exact in int32; EuclideanCompressed scales by
        // scale^2 (scalar.h:92-93).
        int l2 = __float_as_int(aux1) + iyy - 2 * ixy;   // aux1 carries the int32 bits of sum x*x
        float f = float(l2);
        return p.sq ? __fmul_rn(p.scale_sq, f) : f;
    } else if constexpr (OP == OP_IPI) {
        return float(ixy);
    } else {
        // cosine.h:292-296: float(sum) / (a_norm * sqrt(float(bnorm)))
        return __fdiv_rn(float(ixy), __fmul_rn(aux0, __fsqrt_rn(float(iyy))));
    }
}

// One pass of the neighbour expansion: NR rows per thread group, GROUPS groups per warp.
// Candidate `base + r*GROUPS + g` is evaluated by group g in slot r; thread 0 of the group
// publishes the sort key into ckey[].
template <int ROWT, int OP, int DS, int NR, int KS = 1, bool DENSE = false>
__device__ __forceinline__ void eval_pass(const SearchParams& p, const float* q_s, const char* vectors,
                                          const uint32_t* cid, float* ckey, uint32_t base, uint32_t count, int g, int t,
                                          float aux0, float aux1, float ksign) {
    constexpr bool kInt = (OP >= OP_L2I);
    constexpr int G = kInt ? 4 : KS * 16 / Row<ROWT>::LPT;
    constexpr int GROUPS = 32 / G;
    const char* rowp[NR];
    uint32_t idx[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        idx[r] = base + r * GROUPS + g;
        if constexpr (DENSE) {
            // slots past the last candidate re-read the last candidate's row (already in flight in this
            // pass) instead of being predicated off: no null checks, no predicated arithmetic
            rowp[r] = vectors + size_t(cid[min(idx[r], count - 1)]) * p.row_stride;
        } else {
            rowp[r] = idx[r] < count ? vectors + size_t(cid[idx[r]]) * p.row_stride : nullptr;
        }
    }
    float sum[NR], nrm[NR];
    int ixy[NR], iyy[NR];
    if constexpr (kInt) {
        int_rows<ROWT, NR, DENSE>(p, reinterpret_cast<const uint8_t*>(q_s), rowp, t, ixy, iyy);
    } else if constexpr (KS == 4) {
        float_rows_split<ROWT, OP, NR, DENSE>(p, q_s, rowp, t, sum, nrm);
    } else {
        float_rows<ROWT, OP, DS, NR, DENSE>(p, q_s, rowp, t, sum, nrm);
    }
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const float d = finish_distance<OP>(p, kInt ? 0.f : sum[r], (OP == OP_COSF) ? nrm[r] : 0.f, kInt ? ixy[r] : 0,
                                            kInt ? iyy[r] : 0, aux0, aux1);
        if (t == 0 && (DENSE ? idx[r] < count : rowp[r] != nullptr)) ckey[idx[r]] = __fmul_rn(d, ksign);
    }
}

// 16-byte asynchronous global->shared copy (LDGSTS): no destination register, so the bytes can
// stay in flight across a whole hop.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------------------------------
// The kernel.
// ---------------------------------------------------------------------------------------
#ifndef SVSB200_MIN_BLOCKS
#define SVSB200_MIN_BLOCKS 2   // <= 128 registers: four 4-warp CTAs (16 warps) per SM
#endif
// EXH = true turns the same machinery into an exhaustive scan (the reference's flat index,
// index/flat/flat.h:159,421-465, used here for ground truth): the "neighbours" of every step
// are the next block of consecutive ids, there is no visited filter and no expansion order;
// the sorted buffer (window = capacity = k) ends up holding the exact top-k, ties by id.
template <int ROWT, int OP, int DS, int NROWS, bool EXH = false, int KS = 1>
__global__ void __launch_bounds__(256, SVSB200_MIN_BLOCKS) vamana_search_kernel(const __grid_constant__ SearchParams p) {
    constexpr bool kInt = (OP >= OP_L2I);
    constexpr int G = kInt ? 4 : KS * 16 / Row<ROWT>::LPT;     // threads per row
    constexpr int GROUPS = 32 / G;                        // rows per warp per slot
    constexpr unsigned FULL = 0xFFFFFFFFu;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int g = lane / G;      // group inside the warp
    const int t = lane % G;      // thread inside the group

    unsigned char* wbase = smem_raw + size_t(warp) * warp_smem_bytes(p.qstride, p.cap_pad, p.deg_pad, p.filter_slots * (p.filter_tag16 ? 2u : 4u));
    float* q_s = reinterpret_cast<float*>(wbase);
    float* bkey = q_s + p.qstride;                                      // [cap_pad] sort keys
    uint32_t* bid = reinterpret_cast<uint32_t*>(bkey + p.cap_pad);      // [cap_pad] id | visited
    float* ckey = reinterpret_cast<float*>(bid + p.cap_pad);            // [deg_pad] candidate keys
    uint32_t* cid = reinterpret_cast<uint32_t*>(ckey + p.deg_pad);      // [deg_pad] candidate ids
    float* skey = reinterpret_cast<float*>(cid + p.deg_pad);            // [deg_pad] survivors
    uint32_t* spos = reinterpret_cast<uint32_t*>(skey + p.deg_pad);
    uint32_t* sid = spos + p.deg_pad;
    uint32_t* sfp = sid + p.deg_pad;
    uint32_t* filt = sfp + p.deg_pad;                                   // [filter_slots] visited ids (or 16-bit tags)
    uint32_t* adj = filt + (p.filter_tag16 ? p.filter_slots / 2 : p.filter_slots);   // [2][deg_pad] staged adjacency rows

    const float ksign = p.greater ? -1.0f : 1.0f;   // keys = sign * distance, ordered by '<'
    const uint32_t C = p.capacity, W = p.window;
    const uint32_t hibit = 1u << (31 - __clz(int(C)));
    const char* vectors = reinterpret_cast<const char*>(p.vectors);

    for (;;) {
        uint32_t q = 0;
        if (lane == 0) q = atomicAdd(p.work_counter, 1u);
        q = __shfl_sync(FULL, q, 0);
        // EXH: a work item is (query, range of base rows); its top-k goes to row [range][query] of the output
        uint32_t exh_lo = 0, exh_hi = p.n, out_row = q;
        if constexpr (EXH) {
            const uint32_t splits = p.exh_split ? p.exh_split : 1u;
            if (q >= p.nq * splits) break;
            const uint32_t rg = q / p.nq;
            out_row = q;                      // == rg * nq + query
            q -= rg * p.nq;
            const uint32_t chunk = (p.n + splits - 1) / splits;
            exh_lo = min(p.n, rg * chunk);
            exh_hi = min(p.n, exh_lo + chunk);
        } else {
            if (q >= p.nq) break;
        }
        // cancellation between queries (extensions.h:579)
        if (p.cancel && *reinterpret_cast<const volatile int*>(p.cancel)) break;

        // ---- stage the prepared query (maybe_fix_argument already applied) ----
        if constexpr (kInt) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(p.qcodes + size_t(q) * p.qstride);
            uint32_t* dst = reinterpret_cast<uint32_t*>(q_s);
            for (uint32_t i = lane; i < p.qstride / 4; i += 32) dst[i] = src[i];
        } else {
            const float* src = p.qf + size_t(q) * p.qstride;
            for (uint32_t i = lane; i < p.qstride; i += 32) q_s[i] = src[i];
        }
        const float aux0 = p.qaux[2 * size_t(q)], aux1 = p.qaux[2 * size_t(q) + 1];
        // Visited filter (the reference's optional VisitedFilter, index/vamana/filter.h:49-130,
        // here direct-mapped with full ids: false negatives possible, never a false positive,
        // so skipping a hit cannot change the result -- search_buffer.h:420).
        for (uint32_t i = lane; i < (p.filter_tag16 ? p.filter_slots / 2 : p.filter_slots); i += 32) filt[i] = kNoNeighbor;
        __syncwarp();

        // ---- EntryPointInitializer (greedy_search.h:62-94): clear, push entry point ----
        const uint32_t E = p.n_entry > 1 ? min(p.n_entry, p.deg_pad) : 1u;
        uint32_t size = EXH ? 0 : 1, cursor = 0, n_hops = 0, n_evals = E, n_fetched = E;
        if constexpr (!EXH) {
            for (uint32_t i = lane; i < E; i += 32) cid[i] = E > 1 ? p.entry_points[i] : p.entry_point;
            __syncwarp();
            for (uint32_t base = 0; base < E; base += GROUPS)
                eval_pass<ROWT, OP, DS, 1, KS>(p, q_s, vectors, cid, ckey, base, E, g, t, aux0, aux1, ksign);
            __syncwarp();
            if (lane == 0) {
                // push_back every entry point, then sort (greedy_search.h:80-92); here: insertion in entry order
                // (ties keep that order, a repeated id is dropped, the list is cut at the capacity)
                size = 0;
                for (uint32_t i = 0; i < E; ++i) {
                    const float d = ckey[i];
                    const uint32_t id = cid[i];
                    bool dup = false;
                    for (uint32_t j = 0; j < size; ++j) dup |= bid[j] == id;
                    if (dup) continue;
                    uint32_t pos = size;
                    while (pos > 0 && d < bkey[pos - 1]) --pos;
                    if (pos >= C) continue;
                    const uint32_t last = min(size, C - 1);
                    for (uint32_t j = last; j > pos; --j) {
                        bkey[j] = bkey[j - 1];
                        bid[j] = bid[j - 1];
                    }
                    bkey[pos] = d;
                    bid[pos] = id;
                    size = min(size + 1, C);
                }
            }
            size = __shfl_sync(FULL, size, 0);
            __syncwarp();
        }
        uint32_t scan_base = exh_lo;   // EXH: first id of the current block
        uint32_t staged_node = kNoNeighbor;   // node whose adjacency row sits in adj[staged_buf]
        uint32_t staged_buf = 0;

        // ---- main loop: while (!buffer.done()) (greedy_search.h:153) ----
        for (;;) {
            // cancellation inside a search (greedy_search.h:155)
            if (p.cancel && *reinterpret_cast<const volatile int*>(p.cancel)) break;
            uint32_t deg = 0;
            if constexpr (EXH) {
                if (scan_base >= exh_hi) break;
                deg = min(p.deg_pad, exh_hi - scan_base);
                for (uint32_t i = lane; i < deg; i += 32) cid[i] = scan_base + i;
                scan_base += deg;
                __syncwarp();
            } else {
                // buffer.next(): first unvisited entry inside min(size, window)
                const uint32_t upper = min(size, W);
                uint32_t pos = cursor, pred_pos = 0xFFFFFFFFu;
                bool found = false;
                while (pos < upper) {
                    uint32_t j = pos + lane;
                    bool unv = (j < upper) && !(bid[j] & kVisitedBit);
                    unsigned m = __ballot_sync(FULL, unv);
                    if (m) {
                        // Once the first few hops are over, the unvisited entry right behind the
                        // chosen one is the next node to be expanded in 97% of hops (measured).
                        const unsigned m2 = m & (m - 1);
                        if (m2) pred_pos = pos + __ffs(m2) - 1;
                        pos += __ffs(m) - 1;
                        found = true;
                        break;
                    }
                    pos += 32;
                }
                if (!found) break;   // done()
                const uint32_t node = bid[pos];
                // Adjacency row of this node: staged by the previous hop if the prediction held.
                const bool have_adj = (node == staged_node);
                const uint32_t* adj_cur = adj + staged_buf * p.deg_pad;
                // (always drain: a stale copy from a missed prediction must not land later)
                cp_async_wait_all();
                __syncwarp();
                // Stage the predicted next node's adjacency row (asynchronous global->shared copy,
                // in flight during this hop's distance evaluations and merge).
                staged_node = kNoNeighbor;
                if (pred_pos != 0xFFFFFFFFu) {
                    staged_node = bid[pred_pos] & kIdMask;
                    staged_buf ^= 1u;
                    uint32_t* dst = adj + staged_buf * p.deg_pad;
                    const uint32_t* src = p.graph + size_t(staged_node) * p.gstride;
                    for (uint32_t i = lane * 4; i < p.gstride; i += 128) cp_async16(dst + i, src + i);
                    cp_async_commit();
                }
                __syncwarp();
                if (lane == 0) bid[pos] = node | kVisitedBit;
                cursor = pos + 1;

                // graph.get_node(node): adjacency row, neighbours first, kNoNeighbor padding.
                // Ids that pass the visited filter are compacted (adjacency order kept) into cid[].
                const uint32_t* grow = p.graph + size_t(node) * p.gstride;
                const uint32_t fmask = (p.filter_tag16 ? p.filter_slots / 2 : p.filter_slots) - 1;   // sets
                uint32_t ncand = 0;
                for (uint32_t j0 = 0; j0 < p.gstride; j0 += 32) {
                    uint32_t j = j0 + lane;
                    uint32_t nb = (j < p.gstride) ? (have_adj ? adj_cur[j] : __ldg(grow + j)) : kNoNeighbor;
                    bool fresh = nb != kNoNeighbor;
                    deg += __popc(__ballot_sync(FULL, fresh));
                    if (p.filter_slots && fresh) {
                        // emplace_visited (search_buffer.h:462-464): hit -> skip, else remember
                        const uint32_t slot = nb & fmask;
                        if (p.filter_tag16) {
                            // Two-way set-associative, LRU by position: a set is one 32-bit word
                            // holding two 16-bit tags (set index + tag reconstruct the full id,
                            // so a hit is exact).  A miss pushes the new tag to the front and
                            // drops the older of the two.
                            const uint32_t tag = nb >> p.filter_shift;
                            const uint32_t set = filt[slot];
                            fresh = ((set & 0xFFFFu) != tag) && ((set >> 16) != tag);
                            if (fresh) filt[slot] = (set << 16) | tag;
                        } else {
                            fresh = filt[slot] != nb;
                            if (fresh) filt[slot] = nb;
                        }
                    }
                    const unsigned m = __ballot_sync(FULL, fresh);
                    if (fresh) cid[ncand + __popc(m & ((1u << lane) - 1u))] = nb;
                    ncand += __popc(m);
                    __syncwarp();
                }
                ++n_hops;
                // tracker.visited(node, neighbors.size()) (greedy_search.h:165) counts the row as
                // the reference stores it, i.e. including the repeated ids removed at upload.
                n_evals += p.hops ? uint32_t(__ldg(p.ref_degree + node)) : deg;
                n_fetched += ncand;
                if (ncand == 0) continue;
                deg = ncand;   // from here on: the candidates that are actually evaluated

            }
            // neighbour expansion: distance of every neighbour (greedy_search.h:190-201),
            // NROWS x GROUPS candidates per pass.  (A single-row pass for small remainders was
            // measured slower: more code, more registers.)
            for (uint32_t base = 0; base < deg; base += NROWS * GROUPS)
                eval_pass<ROWT, OP, DS, NROWS, KS>(p, q_s, vectors, cid, ckey, base, deg, g, t, aux0, aux1, ksign);
            __syncwarp();

            // ---- merge the candidates into the sorted buffer (== sequential insert) ----
            const bool full = (size == C);
            const float backkey = size ? bkey[size - 1] : 0.0f;
            uint32_t S = 0, minpos = 0xFFFFFFFFu;
            for (uint32_t r0 = 0; r0 < deg; r0 += 32) {
                const uint32_t r = r0 + lane;
                const bool valid = r < deg;
                const float d = valid ? ckey[r] : 0.0f;
                const uint32_t id = valid ? cid[r] : 0;
                // can_skip (search_buffer.h:342-344): full && cmp(back, d)
                bool surv = valid && !(full && backkey < d);
                uint32_t ipos = 0;
                if (__any_sync(FULL, surv)) {
                    // lower_bound with !cmp(d, other) (search_buffer.h:364-371): number of
                    // entries that are better than or equal to d.
                    for (uint32_t step = hibit; step; step >>= 1) {
                        uint32_t j = ipos + step;
                        if (surv && j <= size && !(d < bkey[j - 1])) ipos = j;
                    }
                    // duplicate-id scan over the equal-key run (search_buffer.h:380-391)
                    if (surv) {
                        uint32_t j = ipos;
                        while (j > 0) {
                            --j;
                            if (bkey[j] < d) break;
                            if ((bid[j] & kIdMask) == id) {
                                surv = false;
                                break;
                            }
                        }
                    }
                }
                const unsigned m = __ballot_sync(FULL, surv);
                if (surv) {
                    const uint32_t ci = S + __popc(m & ((1u << lane) - 1u));
                    skey[ci] = d;
                    spos[ci] = ipos;
                    sid[ci] = id;
                    minpos = min(minpos, ipos);
                }
                S += __popc(m);
            }
            if (S == 0) continue;
            minpos = __reduce_min_sync(FULL, minpos);
            __syncwarp();

            // final position of every survivor: insertion point + stable rank among survivors
            for (uint32_t si = lane; si < S; si += 32) {
                const float md = skey[si];
                uint32_t rank = 0;
                for (uint32_t s = 0; s < S; ++s) {
                    const float ds = skey[s];
                    rank += (ds < md) || (!(md < ds) && s < si);
                }
                sfp[si] = spos[si] + rank;
            }
            // shift the old entries, top chunk first so the move is safe in place
            if (minpos < size) {
                const int chunk_lo = int(minpos >> 5);
                for (int ch = int((size - 1) >> 5); ch >= chunk_lo; --ch) {
                    const uint32_t j = uint32_t(ch) * 32 + lane;
                    const bool have = j < size;
                    const float kk = have ? bkey[j] : 0.0f;
                    const uint32_t ii = have ? bid[j] : 0;
                    uint32_t shift = 0;
                    for (uint32_t s = 0; s < S; ++s) shift += (spos[s] <= j);
                    __syncwarp();
                    if (have && shift && j + shift < C) {
                        bkey[j + shift] = kk;
                        bid[j + shift] = ii;
                    }
                    __syncwarp();
                }
            }
            __syncwarp();
            for (uint32_t si = lane; si < S; si += 32) {
                const uint32_t fp = sfp[si];
                if (fp < C) {
                    bkey[fp] = skey[si];
                    bid[fp] = sid[si];
                }
            }
            size = min(size + S, C);
            cursor = min(cursor, minpos);   // best_unvisited = min(best_unvisited, i) (:401)
            __syncwarp();
        }

        // ---- copy the first k entries out (extensions.h:588-590) ----
        for (uint32_t j = lane; j < p.k; j += 32) {
            const bool valid = j < size;
            const uint32_t id = valid ? (bid[j] & kIdMask) : 0xFFFFFFFFu;
            const float dist = valid ? __fmul_rn(bkey[j], ksign) : (p.greater ? -INFINITY : INFINITY);
            const size_t o = size_t(out_row) * p.k + j;
            if (p.id_bytes == 8)
                reinterpret_cast<uint64_t*>(p.out_ids)[o] = valid ? uint64_t(id) + p.id_offset : ~uint64_t(0);
            else
                reinterpret_cast<uint32_t*>(p.out_ids)[o] = id;
            p.out_dists[o] = dist;
        }
        if (p.hops && lane == 0) {
            p.hops[q] = n_hops;
            p.evals[q] = n_evals;
            p.fetched[q] = n_fetched;
        }
        __syncwarp();
    }
}

// Host-side launch helper shared by the per-type translation units.
template <int ROWT, int OP, int DS, int NROWS, int KS = 1>
cudaError_t launch_one(const SearchParams& p, const LaunchConfig& cfg) {
    auto kernel = vamana_search_kernel<ROWT, OP, DS, NROWS, false, KS>;
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(cfg.smem_bytes));
    if (err != cudaSuccess) return err;
    int grid = cfg.grid;
    if (grid < 0) {
        // persistent grid: SM count x resident CTAs of this instantiation
        int resident = 0;
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kernel, cfg.warps_per_cta * 32, cfg.smem_bytes);
        if (err != cudaSuccess) return err;
        grid = -grid * (resident > 0 ? resident : 1);
    }
    const int needed = int((p.nq + cfg.warps_per_cta - 1) / cfg.warps_per_cta);
    if (grid > needed) grid = needed;
    kernel<<<grid, cfg.warps_per_cta * 32, cfg.smem_bytes, cfg.stream>>>(p);
    count_launch();
    return cudaGetLastError();
}

template <int ROWT, int OP> cudaError_t launch_exhaustive(const SearchParams& p, const LaunchConfig& cfg) {
    auto kernel = vamana_search_kernel<ROWT, OP, 0, 2, true>;
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(cfg.smem_bytes));
    if (err != cudaSuccess) return err;
    int resident = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kernel, cfg.warps_per_cta * 32, cfg.smem_bytes);
    if (err != cudaSuccess) return err;
    int grid = -cfg.grid * (resident > 0 ? resident : 1);
    const int needed = int((size_t(p.nq) * (p.exh_split ? p.exh_split : 1u) + cfg.warps_per_cta - 1) / cfg.warps_per_cta);
    if (grid > needed) grid = needed;
    kernel<<<grid, cfg.warps_per_cta * 32, cfg.smem_bytes, cfg.stream>>>(p);
    count_launch();
    return cudaGetLastError();
}

template <int ROWT, int OP> cudaError_t launch_dims(const SearchParams& p, const LaunchConfig& cfg, int nrows) {
    // Static dimensions get fully unrolled loads (all of a row's loads in flight at once);
    // everything else takes the dynamic-length path.  Same expression tree either way,
    // like the reference's static-N vs Dynamic kernels (distance_core.h:31-42).
    if constexpr (OP < OP_L2I) {
        if (p.dim == 96) return nrows == 1 ? launch_one<ROWT, OP, 96, 1>(p, cfg) : launch_one<ROWT, OP, 96, 2>(p, cfg);
        if (p.dim == 128) return nrows == 1 ? launch_one<ROWT, OP, 128, 1>(p, cfg) : launch_one<ROWT, OP, 128, 2>(p, cfg);
        // wide rows: accumulators split over 4x the threads (float_rows_split)
        if (p.dim >= 256) return launch_one<ROWT, OP, 0, 2, 4>(p, cfg);
    }
    return nrows == 1 ? launch_one<ROWT, OP, 0, 1>(p, cfg) : launch_one<ROWT, OP, 0, 2>(p, cfg);
}

}  // namespace svsb200
