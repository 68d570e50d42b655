// search_fast.cuh -- the lean form of the Vamana batched greedy search (same results as
// search_kernel.cuh, far fewer instructions per expanded node).
//
// Replaces, for a whole query batch (file:line under /root/reference/include/svs):
//   index/vamana/index.h:564-611         VamanaIndex::search        (thread pool -> grid)
//   index/vamana/greedy_search.h:124-203 greedy_search              (one warp per query)
//   index/vamana/search_buffer.h:104-497 SearchBuffer               (sorted buffer in smem)
// and reuses the bit-exact distance code of search_kernel.cuh (float_rows / int_rows).
//
// What is different from vamana_search_kernel (kept as the generic fallback and as the
// exhaustive-scan kernel):
//   * ONE warp per CTA: every shared-memory address and every loop bound is CTA-uniform, so the
//     addressing lives on the uniform datapath instead of being recomputed per thread;
//   * the adjacency row of the predicted next node is prefetched into REGISTERS (one coalesced
//     32-bit load per 32 neighbours, issued a whole hop ahead) -- no cp.async staging, no
//     shared-memory round trip;
//   * the sorted buffer stores {key, id|visited} pairs (one 64-bit LDS/STS per entry) and the
//     merge is a GATHER over final slots: the survivors' final positions form a bit mask per
//     32-entry slot (one REDUX.OR), every lane derives the source of "its" slot entry from two
//     popcounts, and slots are rewritten top-down in place.  Candidates are merged in groups
//     of 32; each group is exactly equivalent to the reference's sequential
//     `for id in neighbours: buffer.insert(...)` over those candidates (DESIGN.md §4,
//     tests/test_merge_model.py), so any grouping gives the reference's result.
#pragma once

#include "search_kernel.cuh"

namespace svsb200 {

// Resident CTAs (= warps = queries) per SM the compiler must allow for: 24 (80 registers) where the
// instantiation fits without spilling, 16 (128 registers) otherwise (ptxas -v, csrc/*.ptxas.log).
template <int ROWT, int OP, int DS, int KS> constexpr int fast_min_blocks() {
#ifdef SVSB200_FAST_MIN_BLOCKS
    return SVSB200_FAST_MIN_BLOCKS;
#else
    if (ROWT == SVSB200_F32 && (DS != 0 || KS == 4)) return 24;
    if (ROWT == SVSB200_F16 && DS == 96 && OP != OP_COSF) return 24;
    return 16;
#endif
}

#ifdef SVSB200_PHASE_CLOCKS
// Diagnostic build only (scratch/build_variant.sh): SM cycles per phase of a hop, summed over all queries by lane 0.
static __device__ unsigned long long g_phase_clocks[8];   // (one copy per translation unit; fast_f32.cu exports its own)
#define PHASE_CLOCK(var) const long long var = clock64()
#else
#define PHASE_CLOCK(var)
#endif

// HIST = true is the graph builder's form (build.cu): every expanded node is appended, with its key, to the
// query's search history -- the reference's `use_full_search_history` candidate pool (vamana_build.h:344-352).
template <int ROWT, int OP, int DS, int KS, bool HIST = false>
__global__ void __launch_bounds__(32, fast_min_blocks<ROWT, OP, DS, KS>()) vamana_search_fast_kernel(const __grid_constant__ SearchParams p) {
    constexpr int NROWS = 2;
    constexpr bool kInt = (OP >= OP_L2I);
    constexpr int G = kInt ? 4 : KS * 16 / Row<ROWT>::LPT;   // threads per row
    constexpr int GROUPS = 32 / G;                            // rows per slot of a pass
    constexpr unsigned FULL = 0xFFFFFFFFu;
    constexpr uint32_t NONE = 0xFFFFFFFFu;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    const int g = lane / G;
    const int t = lane % G;
    const unsigned lt_mask = (1u << lane) - 1u;

    // Visited filter: `fsets` sets of eight 16-bit tags (one 128-bit word per set, newest tag first).  Set index
    // + tag reconstruct the full id, so a hit is exact (the host guarantees (n-1) >> filter_shift < 0xFFFF).
    const uint32_t fsets = p.filter_slots / 8;
    uint4* filt = reinterpret_cast<uint4*>(smem_raw);                        // [fsets]
    float* q_s = reinterpret_cast<float*>(filt + fsets);                     // [qstride] prepared query
    uint2* buf = reinterpret_cast<uint2*>(q_s + p.qstride);                  // [cap_pad] {key bits, id | visited}
    float* ckey = reinterpret_cast<float*>(buf + p.cap_pad);                 // [deg_pad] candidate keys
    uint32_t* cid = reinterpret_cast<uint32_t*>(ckey + p.deg_pad);           // [deg_pad] candidate ids

    const float ksign = p.greater ? -1.0f : 1.0f;   // keys = sign * distance, ordered by '<'
    const uint32_t C = p.capacity, W = p.window;
    const char* vectors = reinterpret_cast<const char*>(p.vectors);
    const uint32_t fmask = fsets - 1u;              // set index mask (fsets is a power of two)

    for (;;) {
        uint32_t q = 0;
        if (lane == 0) q = atomicAdd(p.work_counter, 1u);
        q = __shfl_sync(FULL, q, 0);
        if (q >= p.nq) break;
        // cancellation between queries (extensions.h:579)
        if (p.cancel && *reinterpret_cast<const volatile int*>(p.cancel)) break;

        // ---- stage the prepared query (maybe_fix_argument already applied), reset the filter ----
        if constexpr (kInt) {
            const uint4* src = reinterpret_cast<const uint4*>(p.qcodes + size_t(q) * p.qstride);
            uint4* dst = reinterpret_cast<uint4*>(q_s);
#pragma unroll 1
            for (uint32_t i = lane; i < p.qstride / 16; i += 32) dst[i] = __ldg(src + i);
        } else {
            const float4* src = reinterpret_cast<const float4*>(p.qf + size_t(q) * p.qstride);
            float4* dst = reinterpret_cast<float4*>(q_s);
#pragma unroll 1
            for (uint32_t i = lane; i < p.qstride / 4; i += 32) dst[i] = __ldg(src + i);
        }
        const float aux0 = p.qaux[2 * size_t(q)], aux1 = p.qaux[2 * size_t(q) + 1];
#pragma unroll 4
        for (uint32_t i = lane; i < fsets; i += 32) filt[i] = make_uint4(NONE, NONE, NONE, NONE);
        // ---- EntryPointInitializer (greedy_search.h:62-94): the entry point goes through the same
        // evaluate-and-merge code as a hop's neighbours, into the empty buffer ----
        const uint32_t E = p.n_entry > 1 ? min(p.n_entry, 32u) : 1u;   // entry points (index/vamana/index.h:304-312)
        uint32_t size = 0, cursor = 0, n_hops = 0, n_evals = E, n_fetched = E;
        uint32_t n_hist = 0;
        uint32_t staged_node = NONE;          // node whose adjacency row sits in nxt[]
        uint32_t nxt[kFastMaxGW];
#pragma unroll
        for (int w = 0; w < kFastMaxGW; ++w) nxt[w] = kNoNeighbor;
        int first = 1;
        asm volatile("" : "+r"(first));   // opaque: keeps the compiler from peeling (= duplicating) the first hop

        // ---- main loop: while (!buffer.done()) (greedy_search.h:153) ----
        for (;;) {
            // cancellation inside a search (greedy_search.h:155): polled here, consumed at the end of the hop
            const int cancelled = p.cancel ? *reinterpret_cast<const volatile int*>(p.cancel) : 0;
            uint32_t ncand = 0;
            PHASE_CLOCK(pc0);
#ifdef SVSB200_PHASE_CLOCKS
            long long pc1 = pc0, pc2 = pc0;
#endif
            if (first) {
                first = 0;
                if (uint32_t(lane) < E) cid[lane] = E > 1 ? p.entry_points[lane] : p.entry_point;
                ncand = E;
                __syncwarp();
            } else {
            // buffer.next(): first unvisited entry inside min(size, window)
            const uint32_t upper = min(size, W);
            uint32_t pos = cursor, pred_pos = NONE;
            bool found = false;
#pragma unroll 1
            while (pos < upper) {
                const uint32_t j = pos + lane;
                const bool unv = (j < upper) && !(buf[j].y & kVisitedBit);
                const unsigned m = __ballot_sync(FULL, unv);
                if (m) {
                    // the unvisited entry right behind the chosen one is the next node to be
                    // expanded in 97% of hops (measured): its adjacency row is prefetched below
                    const unsigned m2 = m & (m - 1);
                    if (m2) pred_pos = pos + __ffs(m2) - 1;
                    pos += __ffs(m) - 1;
                    found = true;
                    break;
                }
                pos += 32;
            }
            if (!found) break;   // done()
            // (masked: lane 0 sets the visited bit of this entry below, and nothing orders that store behind the other
            // lanes' read of it -- compute-sanitizer racecheck, round 2)
            const uint32_t node = buf[pos].y & kIdMask;
            // graph.get_node(node): staged in registers by the previous hop if the prediction held; a miss
            // loads into the same registers.  nb[] is copied out BEFORE the next prefetch is issued into nxt[]:
            // the write-after-read dependence keeps the prefetch loads behind every wait on this hop's row, so
            // their latency is never waited for here (they have a whole hop to land).
            if (node != staged_node) {
                const uint32_t* grow = p.graph + size_t(node) * p.gstride;
#pragma unroll
                for (int w = 0; w < kFastMaxGW; ++w)
                    if (w * 32u < p.gstride) nxt[w] = __ldg(grow + w * 32u + lane);   // gstride % 32 == 0 here
            }
            uint32_t nb[kFastMaxGW];
#pragma unroll
            for (int w = 0; w < kFastMaxGW; ++w) nb[w] = nxt[w];
            staged_node = NONE;
            if (pred_pos != NONE) {
                staged_node = buf[pred_pos].y & kIdMask;
                const uint32_t* prow = p.graph + size_t(staged_node) * p.gstride;
#pragma unroll
                for (int w = 0; w < kFastMaxGW; ++w)
                    if (w * 32u < p.gstride) nxt[w] = __ldg(prow + w * 32u + lane);
            }
            if (lane == 0) buf[pos].y = node | kVisitedBit;
            if constexpr (HIST) {
                if (lane == 0 && n_hist < p.hist_cap) p.hist[size_t(q) * p.hist_cap + n_hist] = make_uint2(buf[pos].x, node);
                n_hist += (n_hist < p.hist_cap) ? 1u : 0u;
            }
            cursor = pos + 1;
#ifdef SVSB200_PHASE_CLOCKS
            pc1 = clock64();
#endif

            // Ids that pass the visited filter are compacted (adjacency order kept) into cid[].
            // emplace_visited (search_buffer.h:462-464): hit -> skip, else remember.  Races between
            // lanes on one set can only lose an update (a later false "fresh"), never invent a hit.
#pragma unroll
            for (int w = 0; w < kFastMaxGW; ++w) {
                if (w * 32u < p.gstride) {
                    bool fresh = nb[w] != kNoNeighbor;
                    if (fresh) {   // the filter is always on here (the host routes filter-off runs to the generic kernel)
                        const uint32_t slot = nb[w] & fmask;
                        const uint32_t tag = nb[w] >> p.filter_shift;
                        const uint32_t tag2 = tag * 0x00010001u;
                        const uint4 set = filt[slot];
                        // any 16-bit half of the set equal to the tag?  x ^ tag2 has a zero half exactly then;
                        // (v - 0x00010001) & ~v & 0x80008000 is non-zero iff v has a zero half.
                        const uint32_t x0 = set.x ^ tag2, x1 = set.y ^ tag2, x2 = set.z ^ tag2, x3 = set.w ^ tag2;
                        const uint32_t hit = (((x0 - 0x00010001u) & ~x0) | ((x1 - 0x00010001u) & ~x1) |
                                              ((x2 - 0x00010001u) & ~x2) | ((x3 - 0x00010001u) & ~x3)) & 0x80008000u;
                        fresh = hit == 0u;
                        if (fresh)   // push the new tag in front, drop the oldest
                            filt[slot] = make_uint4((set.x << 16) | tag, __funnelshift_l(set.x, set.y, 16),
                                                    __funnelshift_l(set.y, set.z, 16), __funnelshift_l(set.z, set.w, 16));
                    }
                    const unsigned m = __ballot_sync(FULL, fresh);
                    if (fresh) cid[ncand + __popc(m & lt_mask)] = nb[w];
                    ncand += __popc(m);
                }
            }
            if (p.hops) {
                ++n_hops;
                // tracker.visited(node, neighbors.size()) (greedy_search.h:165) counts the row as the
                // reference stores it, i.e. including the repeated ids removed at upload.
                n_evals += uint32_t(__ldg(p.ref_degree + node));
                n_fetched += ncand;
            }
            __syncwarp();
#ifdef SVSB200_PHASE_CLOCKS
            pc2 = clock64();
#endif
            }   // !first
            if (ncand == 0) {
                if (cancelled) break;
                continue;
            }

            // neighbour expansion: distance of every fresh neighbour (greedy_search.h:190-201)
            // (two rows per thread group while more than GROUPS candidates remain, one row for the rest:
            // 69% of the hops of the C2 workload have at most 8 fresh neighbours)
#pragma unroll 1
            for (uint32_t base = 0; base < ncand;) {
                if (ncand - base > uint32_t(GROUPS)) {
                    eval_pass<ROWT, OP, DS, NROWS, KS, true>(p, q_s, vectors, cid, ckey, base, ncand, g, t, aux0, aux1, ksign);
                    base += NROWS * GROUPS;
                } else {
                    eval_pass<ROWT, OP, DS, 1, KS, true>(p, q_s, vectors, cid, ckey, base, ncand, g, t, aux0, aux1, ksign);
                    base += GROUPS;
                }
            }
            __syncwarp();
            PHASE_CLOCK(pc3);

            // ---- merge, 32 candidates at a time (each group == its sequential inserts) ----
#pragma unroll 1
            for (uint32_t r0 = 0; r0 < ncand; r0 += 32) {
                const uint32_t r = r0 + lane;
                const bool valid = r < ncand;
                const float d = valid ? ckey[r] : 0.0f;
                const uint32_t id = valid ? cid[r] : 0u;
                // can_skip (search_buffer.h:342-344): full && cmp(back, d)
                const bool full = (size == C);
                const float backkey = full ? __uint_as_float(buf[size - 1].x) : 0.0f;   // C >= 1, so full implies size >= 1
                bool surv = valid && !(full && backkey < d);
                if (!__any_sync(FULL, surv)) continue;
                // lower_bound with !cmp(d, other) (search_buffer.h:364-371): number of entries that
                // are better than or equal to d
                uint32_t ipos = 0;
#pragma unroll 1
                for (uint32_t step = size ? 1u << (31 - __clz(int(size))) : 0u; step; step >>= 1) {
                    const uint32_t j = ipos + step;
                    if (j <= size && !(d < __uint_as_float(buf[j - 1].x))) ipos = j;
                }
                // duplicate-id scan over the equal-key run (search_buffer.h:380-391)
                if (surv) {
                    uint32_t j = ipos;
                    while (j > 0) {
                        const uint2 e = buf[--j];
                        if (__uint_as_float(e.x) < d) break;
                        if ((e.y & kIdMask) == id) {
                            surv = false;
                            break;
                        }
                    }
                }
                const unsigned m = __ballot_sync(FULL, surv);
                if (m == 0) continue;
                const uint32_t S = __popc(m);
                // stable rank among the survivors: (key, adjacency order).  Their keys are compacted (adjacency
                // order) into skc[], padded with +inf, and every survivor counts the ones ordered before it.
                // (the group's own 32 candidate slots are dead once d / id sit in registers: they hold the
                // compacted keys first and the sorted survivors afterwards)
                float* skc = ckey + r0;
                uint32_t* sid = cid + r0;
                const uint32_t t_me = __popc(m & lt_mask);
                skc[lane] = INFINITY;
                __syncwarp();
                if (surv) skc[t_me] = d;
                __syncwarp();
                uint32_t rank = 0;
#pragma unroll 1
                for (uint32_t t0 = 0; t0 < S; t0 += 4) {
                    const float4 k4 = *reinterpret_cast<const float4*>(skc + t0);
                    const int rel = int(t_me) - int(t0);   // compact index of this lane relative to k4.x
                    rank += ((k4.x < d) || (k4.x == d && 0 < rel)) ? 1u : 0u;
                    rank += ((k4.y < d) || (k4.y == d && 1 < rel)) ? 1u : 0u;
                    rank += ((k4.z < d) || (k4.z == d && 2 < rel)) ? 1u : 0u;
                    rank += ((k4.w < d) || (k4.w == d && 3 < rel)) ? 1u : 0u;
                }
                // final position = insertion point + rank; unique per survivor and increasing in rank
                const uint32_t fp = surv ? ipos + rank : NONE;
                const uint32_t minpos = __reduce_min_sync(FULL, surv ? ipos : NONE);
                __syncwarp();   // every lane is done reading the compacted keys
                if (surv) {
                    skc[rank] = d;
                    sid[rank] = id;
                }
                const uint32_t newsize = min(size + S, C);
                const int top = int((newsize - 1) >> 5), lo = int(minpos >> 5);
                // Final slot f holds either the survivor with fp == f or the old entry f - #{fp < f}.  Done in
                // place, top-down, 128 entries (4 x 32) at a time: a block only reads the old buffer inside itself
                // and the 32 entries below it, so reading a block completely before writing it is enough.
                const int top4 = top >> 2, lo4 = lo >> 2;
                // survivors that land beyond the highest block (they fall off the end)
                uint32_t above = __popc(__ballot_sync(FULL, surv && fp >= 128u * uint32_t(top4 + 1)));
                __syncwarp();
#pragma unroll 1
                for (int b4 = top4; b4 >= lo4; --b4) {
                    uint2 e[4];
                    bool wr[4];
#pragma unroll
                    for (int u = 3; u >= 0; --u) {
                        const int sl = 4 * b4 + u;
                        const uint32_t f = 32u * uint32_t(sl) + lane;
                        const uint32_t Ms = __reduce_or_sync(FULL, (fp >> 5) == uint32_t(sl) ? (1u << (fp & 31u)) : 0u);
                        wr[u] = false;
                        e[u] = make_uint2(0u, 0u);
                        if (sl <= top && sl >= lo) {
                            const uint32_t before = S - (above + __popc(Ms >> lane));   // survivors with fp < f
                            const bool mine = (Ms >> lane) & 1u;
                            wr[u] = (f < newsize) && (f >= minpos);
                            if (wr[u]) e[u] = mine ? make_uint2(__float_as_uint(skc[before]), sid[before]) : buf[f - before];
                        }
                        above += __popc(Ms);
                    }
                    __syncwarp();
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (wr[u]) buf[32u * uint32_t(4 * b4 + u) + lane] = e[u];
                }
                size = newsize;
                cursor = min(cursor, minpos);   // best_unvisited = min(best_unvisited, i) (:401)
                __syncwarp();
            }
#ifdef SVSB200_PHASE_CLOCKS
            if (lane == 0) {
                const long long pc4 = clock64();
                atomicAdd(&g_phase_clocks[0], (unsigned long long)(pc1 - pc0));
                atomicAdd(&g_phase_clocks[1], (unsigned long long)(pc2 - pc1));
                atomicAdd(&g_phase_clocks[2], (unsigned long long)(pc3 - pc2));
                atomicAdd(&g_phase_clocks[3], (unsigned long long)(pc4 - pc3));
                atomicAdd(&g_phase_clocks[4], 1ull);
            }
#endif
            if (cancelled) break;
        }

        // ---- copy the first k entries out (extensions.h:588-590) ----
#pragma unroll 1
        for (uint32_t j = lane; j < p.k; j += 32) {
            const bool valid = j < size;
            const uint2 e = valid ? buf[j] : make_uint2(0u, 0u);
            const uint32_t id = valid ? (e.y & kIdMask) : 0xFFFFFFFFu;
            const float dist = valid ? __fmul_rn(__uint_as_float(e.x), ksign) : (p.greater ? -INFINITY : INFINITY);
            const size_t o = size_t(q) * p.k + j;
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
        if constexpr (HIST) {
            if (lane == 0) p.hist_count[q] = n_hist;
        }
        __syncwarp();
    }
}

template <int ROWT, int OP, int DS, int KS = 1, bool HIST = false>
cudaError_t launch_fast(const SearchParams& p, const LaunchConfig& cfg) {
    auto kernel = vamana_search_fast_kernel<ROWT, OP, DS, KS, HIST>;
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(cfg.smem_bytes));
    if (err != cudaSuccess) return err;
    int grid = cfg.grid;
    if (grid < 0) {
        // persistent grid: SM count x resident CTAs of this instantiation
        int resident = 0;
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kernel, 32, cfg.smem_bytes);
        if (err != cudaSuccess) return err;
        grid = -grid * (resident > 0 ? resident : 1);
    }
    if (uint32_t(grid) > p.nq) grid = int(p.nq);
    kernel<<<grid, 32, cfg.smem_bytes, cfg.stream>>>(p);
    count_launch();
    return cudaGetLastError();
}

template <int ROWT, int OP, bool HIST = false> cudaError_t launch_fast_dims(const SearchParams& p, const LaunchConfig& cfg) {
    // Static dimensions get fully unrolled loads; everything else takes the dynamic-length path.  Same
    // expression tree either way, like the reference's static-N vs Dynamic kernels (distance_core.h:31-42).
    if constexpr (OP < OP_L2I) {
        if (p.dim == 96) return launch_fast<ROWT, OP, 96, 1, HIST>(p, cfg);
        if (p.dim == 128 && !HIST) return launch_fast<ROWT, OP, 128, 1, HIST>(p, cfg);
        if (p.dim >= 256) return launch_fast<ROWT, OP, 0, 4, HIST>(p, cfg);
    }
    return launch_fast<ROWT, OP, 0, 1, HIST>(p, cfg);
}

}  // namespace svsb200
