// Sync-frame peak picking (decode.rs:204-263) and row alignment (decode.rs:122-134,158-159).
//
// The reference's picker is a sequential state machine over the correlation.  It is
// restated here in a form that parallelises (derivation in DESIGN.md "Peak picker"):
//
//   D   = min_distance = row*8/10                      (decode.rs:216)
//   root(p)      <=>  no corr[j] > corr[p] for j in (p, p+D]        (p "survives" the else-if at :250)
//   firstroot(s) =    smallest root >= s     == the peak the picker ends on when it starts at s
//   start s' after a peak p found from start s:  s' = max(p + D + 1, row*(s/row + 1))   (:241-246)
//   pushes at s': (s'/row - len) copies of s', the last of which is refined to firstroot(s')
//
// so the peak list is the orbit of  F(s) = max(firstroot(s) + D + 1, row*(s/row + 1)).
// k_roots finds every root with a van Herk / Gil-Werman sliding maximum (one CTA per block
// of D positions); the walk over the orbit touches only the root lists.
#pragma once

#include <cstdint>
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include "kernels_generic.cuh"
#include "launch.hpp"

namespace aptb200 {

constexpr u32 kNoSeed = 0xFFFFFFFFu;

__device__ __forceinline__ bool last_cta_arrives(u32 *ticket);
template <int THREADS>
__device__ void scan_root_counts(const u32 *root_count, u32 nblocks, u32 *block_off);

// ---------------------------------------------------------------------------------------------
// k_roots: block b owns positions [b*D, (b+1)*D).  For p in the block the window (p, p+D] splits
// into the rest of the block (suffix maximum) and a prefix of the next block (prefix maximum).
// Writes the block's roots, ascending, to root_list[b*D ...] and their count to root_count[b].
// Dynamic shared memory: 2*D floats.
// ---------------------------------------------------------------------------------------------
// Inclusive prefix scan over the CTA (one value per thread) with a binary op; warp shuffles + one smem hop.
template <int THREADS, typename T, typename Op>
__device__ __forceinline__ T block_scan_incl(T v, T identity, Op op, T *s_warp /* THREADS/32 entries */) {
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = op(v, t);
    }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        T w = lane < THREADS / 32 ? s_warp[lane] : identity;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w = op(w, t);
        }
        if (lane < THREADS / 32) s_warp[lane] = w;
    }
    __syncthreads();
    if (warp > 0) v = op(v, s_warp[warp - 1]);
    __syncthreads();
    return v;
}

// Inclusive SUFFIX scan over the CTA: thread t gets op over the values of threads t..THREADS-1.
template <int THREADS, typename T, typename Op>
__device__ __forceinline__ T block_scan_incl_rev(T v, T identity, Op op, T *s_warp /* THREADS/32 entries */) {
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr u32 NW = (THREADS + 31) / 32;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T t = __shfl_down_sync(0xffffffffu, v, o);
        if (lane + o < 32) v = op(v, t);
    }
    if (lane == 0) s_warp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        T w = lane < NW ? s_warp[lane] : identity;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T t = __shfl_down_sync(0xffffffffu, w, o);
            if (lane + o < 32) w = op(w, t);
        }
        if (lane < NW) s_warp[lane] = w;
    }
    __syncthreads();
    if (warp + 1 < NW) v = op(v, s_warp[warp + 1]);
    __syncthreads();
    return v;
}

template <int THREADS, int CHUNK>
__global__ void __launch_bounds__(THREADS, CHUNK <= 10 ? 4 : 2)
k_roots(const float *__restrict__ corr, u64 ncorr, u32 dist, u32 *__restrict__ root_list,
        u32 *__restrict__ root_count, SyncResult *__restrict__ result, u32 *__restrict__ block_off,
        u32 *__restrict__ ticket) {
    extern __shared__ float sm[];
    float *a = sm;             // a[0..D): this block, a[D..2D): next block
    __shared__ float s_wf[THREADS / 32];
    __shared__ u32 s_wu[THREADS / 32];
    __shared__ u32 s_seed;

    const float NEG = -INFINITY;
    const u32 tid = threadIdx.x;
    const u64 base = static_cast<u64>(blockIdx.x) * dist;

    if (tid == 0) s_seed = kNoSeed;
    // 16-byte loads where the block start allows it (corr is 16-byte aligned; base may not be)
    if ((dist & 3) == 0 && base + 2ull * dist <= ncorr) {
        const float4 *src = reinterpret_cast<const float4 *>(corr + base);
        for (u32 i = tid; i < dist / 2; i += THREADS) reinterpret_cast<float4 *>(a)[i] = __ldg(src + i);
    } else {
        for (u32 i = tid; i < 2 * dist; i += THREADS) {
            const u64 g = base + i;
            a[i] = g < ncorr ? __ldg(corr + g) : NEG;
        }
    }
    __syncthreads();

    // seed of the peak list: (0, 0.0) is replaced by the first corr[i] > 0.0 with i <= D
    // (decode.rs:208-209 with the else-if at :250 while i - 0 <= D).
    if (blockIdx.x == 0) {
        u32 first = kNoSeed;
        for (u32 i = tid; i <= dist && i < 2 * dist; i += THREADS)
            if (a[i] > 0.f) { first = i; break; }
        if (first != kNoSeed) atomicMin(&s_seed, first);
    }

    const u32 lo = tid * CHUNK;
    const u32 hi = min(lo + CHUNK, dist);   // chunk [lo, hi) of the block (may be empty)
    float va[CHUNK], vb[CHUNK];
    float cmax_a = NEG, cmax_b = NEG;
    if (CHUNK % 4 == 0 && (dist & 3) == 0 && lo + CHUNK <= dist) {
        // whole chunk inside the block and 16-byte aligned: vector loads, no bounds selects
#pragma unroll
        for (int c = 0; c < CHUNK; c += 4) {
            const float4 x = *reinterpret_cast<const float4 *>(a + lo + c), y = *reinterpret_cast<const float4 *>(a + dist + lo + c);
            va[c] = x.x; va[c + 1] = x.y; va[c + 2] = x.z; va[c + 3] = x.w;
            vb[c] = y.x; vb[c + 1] = y.y; vb[c + 2] = y.z; vb[c + 3] = y.w;
        }
    } else {
#pragma unroll
        for (int c = 0; c < CHUNK; ++c) {
            const u32 i = lo + c;
            va[c] = i < hi ? a[i] : NEG;
            vb[c] = i < hi ? a[dist + i] : NEG;
        }
    }
#pragma unroll
    for (int c = 0; c < CHUNK; ++c) {
        cmax_a = fmaxf(cmax_a, va[c]);
        cmax_b = fmaxf(cmax_b, vb[c]);
    }
    auto fmx = [](float x, float y) { return fmaxf(x, y); };
    // prefix maxima over the next block's chunks, suffix maxima over this block's chunks; each thread then needs the
    // neighbour's inclusive value (chunks < tid of the next block, chunks > tid of this block)
    const float pre_incl = block_scan_incl<THREADS>(cmax_b, NEG, fmx, s_wf);
    const float suf_incl = block_scan_incl_rev<THREADS>(cmax_a, NEG, fmx, s_wf);
    __syncthreads();                         // a[] is no longer needed (the chunks are in registers): reuse it
    float *s_pre = sm, *s_suf = sm + THREADS;
    s_pre[tid] = pre_incl;
    s_suf[tid] = suf_incl;
    __syncthreads();
    const float left_excl = tid > 0 ? s_pre[tid - 1] : NEG;
    const float right = tid + 1 < THREADS ? s_suf[tid + 1] : NEG;

    // prefix maxima inside the next block's chunk, then walk this block's chunk right-to-left
    float pm[CHUNK];
    {
        float run = left_excl;
#pragma unroll
        for (int c = 0; c < CHUNK; ++c) { run = fmaxf(run, vb[c]); pm[c] = run; }
    }
    u32 flags = 0;
    {
        float run = right;
#pragma unroll
        for (int c = CHUNK - 1; c >= 0; --c) {
            const u32 i = lo + c;
            if (i < hi) {
                const float wmax = fmaxf(run, pm[c]);       // max of corr over (p, p+D]
                if (base + i < ncorr && !(wmax > va[c])) flags |= 1u << c;
                run = fmaxf(run, va[c]);
            }
        }
    }
    const u32 cnt = __popc(flags);
    const u32 incl = block_scan_incl<THREADS>(cnt, 0u, [](u32 x, u32 y) { return x + y; }, s_wu);
    u32 w = incl - cnt;
    u32 *list = root_list + base;
#pragma unroll
    for (int c = 0; c < CHUNK; ++c)
        if (flags & (1u << c)) list[w++] = static_cast<u32>(base + lo + c);
    if (tid == THREADS - 1) root_count[blockIdx.x] = incl;
    if (blockIdx.x == 0 && tid == 0) result->seed_index = s_seed;
    // the last CTA to finish numbers the roots densely (exclusive scan of the per-block counts)
    if (ticket != nullptr && last_cta_arrives(ticket)) {
        scan_root_counts<THREADS>(root_count, gridDim.x, block_off);
        if (tid == 0) ticket[1] = 0;           // arrival counter of k_pick_links' grid barriers
    }
}

// Smallest root >= s.  Binary search in the block of s, then the first root of the following
// blocks (the last correlation index is always a root, so the search terminates).
__device__ __forceinline__ const u32 *ri_list(const RootIndex &ri, u32 b) {
    return ri.list + (ri.desc ? static_cast<u64>(ri.desc[b].off) : static_cast<u64>(b) * ri.block);
}

__device__ __forceinline__ u32 first_root(u32 s, const RootIndex &ri) {
    u32 b = s / ri.block;
    {
        const u32 *list = ri_list(ri, b);
        u32 lo = 0, hi = ri.count[b];
        while (lo < hi) {
            const u32 mid = (lo + hi) >> 1;
            if (list[mid] < s) lo = mid + 1; else hi = mid;
        }
        if (lo < ri.count[b]) return list[lo];
    }
    for (++b; b < ri.nblocks; ++b)
        if (ri.count[b] > 0) return ri_list(ri, b)[0];
    return 0xFFFFFFFFu;   // unreachable for s < ncorr
}

// ---------------------------------------------------------------------------------------------
// Sequential orbit walk by one thread: O(rows * log) dependent loads.  The always-correct
// fallback (pathological inputs with millions of roots, e.g. silence) and the v0 picker.
// ---------------------------------------------------------------------------------------------
__device__ void pick_sequential(u64 ncorr, u64 nwork, u32 row, u32 dist, const RootIndex &ri, u32 *__restrict__ positions,
                                u32 max_positions, SyncResult *__restrict__ result) {
    u32 len = 1;
    // peak #1: the seed (0, 0.0), refined if some corr[i] > 0 turns up within D of position 0
    const u32 seed = result->seed_index;
    u32 p = seed == kNoSeed ? 0u : first_root(seed, ri);
    positions[0] = p;
    u64 s = max(static_cast<u64>(p) + dist + 1, 2ull * row);
    while (s < ncorr) {
        const u32 target = static_cast<u32>(s / row);     // peaks.len() after the pushes at s
        for (; len + 1 < target && len < max_positions; ++len) positions[len] = static_cast<u32>(s);
        p = first_root(static_cast<u32>(s), ri);
        if (len < max_positions) positions[len] = p;
        ++len;
        s = max(static_cast<u64>(p) + dist + 1, static_cast<u64>(row) * (s / row + 1));
    }
    if (len > max_positions) len = max_positions;
    // rows: every peak but the last, as long as a whole row fits (decode.rs:125-127);
    // positions are non-decreasing so the passing ones are a prefix.
    u32 rows = 0;
    for (u32 i = 0; i + 1 < len; ++i)
        if (static_cast<u64>(positions[i]) + row < nwork) ++rows; else break;
    result->n_peaks = len;
    result->n_rows = rows;
    result->status = len < 5 ? 3u /* APT_ERR_FEW_SYNC_FRAMES */ : 0u;
}

__global__ void k_pick_sequential(u64 ncorr, u64 nwork, u32 row, u32 dist, const RootIndex ri, u32 *__restrict__ positions,
                                  u32 max_positions, SyncResult *__restrict__ result) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    if (result->status == kSyncRedo) return;
    pick_sequential(ncorr, nwork, row, dist, ri, positions, max_positions, result);
    u32 total = 0;
    for (u32 b = 0; b < ri.nblocks; ++b) total += ri.count[b];
    result->n_roots = total;
}

// ---------------------------------------------------------------------------------------------
// Parallel picker: the orbit of F by pointer doubling.
//
// Candidate starts: A_m = row*m (m < NR) and B_r = root_r + D + 1 (one per root, r in dense order) --
// F maps every start onto one of these, so F is a table J0 over NR + nroots nodes (+ END).
//   k_roots' last CTA     : exclusive scan of the per-block root counts -> dense root numbering
//   k_pick_links (grid)   : J0[c] = F(c), start position and peak of every candidate, one thread each
//   k_pick_links' last CTA: J_{k+1} = J_k o J_k in shared memory (global if it does not fit) while the
//                           orbit grows by orbit[n + 2^k] = J_k[orbit[n]]; then events -> positions.
// Falls back to the one-thread walk when the candidates exceed the scratch capacity.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 block_scan_inclusive_1024(u32 v, u32 *s_tmp) {
    // inclusive scan of one value per thread over a 1024-thread CTA
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    if (lane == 31) s_tmp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        u32 w = s_tmp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        s_tmp[lane] = w;
    }
    __syncthreads();
    if (warp > 0) v += s_tmp[warp - 1];
    __syncthreads();
    return v;
}

// True in exactly one CTA of the grid: the last one to arrive.  Resets the ticket for the next launch.
__device__ __forceinline__ bool last_cta_arrives(u32 *ticket) {
    __shared__ u32 s_is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const u32 t = atomicAdd(ticket, 1u);
        s_is_last = t == gridDim.x - 1;
        if (s_is_last) *ticket = 0;
    }
    __syncthreads();
    if (s_is_last) __threadfence();
    return s_is_last != 0;
}

// Exclusive scan of root_count[0..nblocks) into block_off[0..nblocks]; THREADS = blockDim.x.
template <int THREADS>
__device__ void scan_root_counts(const u32 *root_count, u32 nblocks, u32 *block_off) {
    __shared__ u32 s_tmp[32];
    const u32 T = THREADS;
    const u32 tid = threadIdx.x;
    const u32 per = (nblocks + T - 1) / T;
    const u32 b0 = min(tid * per, nblocks), b1 = min(b0 + per, nblocks);
    u32 local = 0;
    for (u32 b = b0; b < b1; ++b) local += __ldcg(root_count + b);
    const u32 incl = block_scan_incl<THREADS>(local, 0u, [](u32 x, u32 y) { return x + y; }, s_tmp);
    u32 run = incl - local;
    for (u32 b = b0; b < b1; ++b) { block_off[b] = run; run += __ldcg(root_count + b); }
    if (tid == T - 1) block_off[nblocks] = incl;
}

// smallest root >= s as (dense id, position); s < ncorr guarantees one exists
__device__ __forceinline__ void first_root_dense(u32 s, const RootIndex &ri, u32 &dense, u32 &pos) {
    const u32 nblocks = ri.nblocks;
    u32 b = s / ri.block;
    const u32 *list = ri_list(ri, b);
    const u32 cnt = ri.count[b];
    u32 lo = 0, hi = cnt;
    while (lo < hi) {
        const u32 mid = (lo + hi) >> 1;
        if (list[mid] < s) lo = mid + 1; else hi = mid;
    }
    if (lo < cnt) { dense = ri.base[b] + lo; pos = list[lo]; return; }
    // first root of the next non-empty block
    ++b;
    while (b < nblocks && ri.count[b] == 0) ++b;
    dense = b < nblocks ? ri.base[b] : 0u;
    pos = b < nblocks ? ri_list(ri, b)[0] : 0xFFFFFFFFu;
}

// position of the root with dense id r
__device__ __forceinline__ u32 root_by_id(u32 r, const RootIndex &ri) {
    if (ri.by_id) return ri.by_id[r];
    u32 lo = 0, hi = ri.nblocks;                  // largest b with base[b] <= r (base = exclusive scan of the counts)
    while (lo + 1 < hi) {
        const u32 mid = (lo + hi) >> 1;
        if (ri.base[mid] <= r) lo = mid; else hi = mid;
    }
    return ri_list(ri, lo)[r - ri.base[lo]];
}

// Grid-wide barrier for a cooperatively launched (co-resident) grid: monotonic arrival counter in global memory
// (zeroed by k_roots' last CTA before this kernel starts; never reset while CTAs may still be polling it).
__device__ __forceinline__ void grid_barrier(u32 *counter, u32 &target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        atomicAdd(counter, 1u);
        u32 seen;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
        } while (seen < target);
    }
    __syncthreads();
}

// Cooperative grid (all CTAs co-resident): J0 = F for every candidate, then pointer doubling with one grid
// barrier per level -- every level is a single pass of <= 1 element per thread, so the cost is the ~12 barriers.
__global__ void __launch_bounds__(1024)
k_pick_links(u64 ncorr, u64 nwork, u32 row, u32 dist, const RootIndex ri, u32 *__restrict__ positions, u32 max_positions,
             SyncResult *__restrict__ result, PickScratch sc) {
    __shared__ u32 s_tmp[32];
    __shared__ u32 s_misc[4];
    const u32 tid = threadIdx.x;
    constexpr u32 T = 1024;
    const u32 gtid = blockIdx.x * T + tid, gsize = gridDim.x * T;
    const u32 nblocks = ri.nblocks;
    if (result->status == kSyncRedo) return;          // the record pool overflowed: the host re-runs the sync stage
    const u32 nroots = __ldcg(ri.nroots);
    const u32 nr = static_cast<u32>((ncorr + row - 1) / row);      // A-type starts row*m < ncorr
    const u32 ncand = nr + nroots;
    const u32 END = ncand;
    u32 bar_target = 0;
    if (ncand + 1 > sc.cap || nr + 1 > max_positions) {
        // too many roots for the scratch (e.g. silence: every index is a root): correct-but-slow path
        if (blockIdx.x == 0 && tid == 0) {
            pick_sequential(ncorr, nwork, row, dist, ri, positions, max_positions, result);
            result->n_roots = nroots;
        }
        return;
    }

    // ---- J0 = F for every candidate (and END) ----
    for (u32 c = gtid; c <= ncand; c += gsize) {
        u32 nxt = END, s = 0xFFFFFFFFu, peak = 0;
        if (c < ncand) {
            u64 s64;
            if (c < nr) {
                s64 = static_cast<u64>(c) * row;
            } else {
                const u32 rp = root_by_id(c - nr, ri);
                s64 = static_cast<u64>(rp) + dist + 1;
            }
            if (s64 < ncorr) {
                s = static_cast<u32>(s64);
                u32 dense;
                first_root_dense(s, ri, dense, peak);
                const u64 sb = static_cast<u64>(peak) + dist + 1;
                const u64 sa = static_cast<u64>(row) * (s / row + 1);
                if (max(sa, sb) < ncorr) nxt = sb >= sa ? nr + dense : static_cast<u32>(sa / row);
            }
        }
        sc.cand_s[c] = s;
        sc.cand_peak[c] = peak;
        sc.ja[c] = nxt;
    }
    // ---- the first start, from the seed (decode.rs:208-209) ----
    if (gtid == 0) {
        const u32 seed = result->seed_index;
        u32 p1 = 0, start = END;
        u64 s2 = 2ull * row;
        if (seed != kNoSeed) {
            u32 dense;
            first_root_dense(seed, ri, dense, p1);
            const u64 sb = static_cast<u64>(p1) + dist + 1;
            if (sb >= s2) { s2 = sb; start = nr + dense; }
        }
        if (s2 < ncorr) { if (start == END) start = static_cast<u32>(s2 / row); } else start = END;
        positions[0] = p1;
        sc.orbit[0] = start;
    }
    grid_barrier(sc.ticket + 1, bar_target);

    // ---- doubling: orbit[n + 2^k] = J_k[orbit[n]];  J_{k+1} = J_k o J_k ----
    u32 *jc = sc.ja, *jn = sc.jb;
    const u32 max_events = min(nr + 1, max_positions);   // every event lands in a new row
    for (u32 span = 1; span < max_events; span <<= 1) {
        for (u32 n = gtid; n < span && n + span < max_events; n += gsize) sc.orbit[n + span] = __ldcg(jc + __ldcg(sc.orbit + n));
        if ((span << 1) < max_events)
            for (u32 c = gtid; c <= ncand; c += gsize) jn[c] = __ldcg(jc + __ldcg(jc + c));
        grid_barrier(sc.ticket + 1, bar_target);
        u32 *t = jc; jc = jn; jn = t;
    }

    // ---- events -> positions (decode.rs:241-253); END is absorbing so events are a prefix of orbit[] ----
    for (u32 n = gtid; n < max_events; n += gsize) {
        const u32 v = __ldcg(sc.orbit + n);
        if (v == END) continue;
        const u32 s = __ldcg(sc.cand_s + v);
        const u32 target = s / row;
        const u32 prev = n == 0 ? 1u : __ldcg(sc.cand_s + __ldcg(sc.orbit + n - 1)) / row;
        for (u32 j = prev; j + 1 < target; ++j) positions[j] = s;      // duplicates pushed by the `while`
        positions[target - 1] = __ldcg(sc.cand_peak + v);
    }
    grid_barrier(sc.ticket + 1, bar_target);
    if (blockIdx.x != 0) return;

    // ---- CTA 0: counts ----
    u32 my_events = 0;
    for (u32 n = tid; n < max_events; n += T) my_events += __ldcg(sc.orbit + n) != END;
    const u32 events = block_scan_inclusive_1024(my_events, s_tmp);
    if (tid == T - 1) s_misc[2] = events;
    __syncthreads();
    const u32 nev = s_misc[2];
    const u32 npeaks = nev == 0 ? 1u : __ldcg(sc.cand_s + __ldcg(sc.orbit + nev - 1)) / row;
    // rows that fit (decode.rs:125-127): positions are non-decreasing -> count of the passing prefix
    u32 cnt = 0;
    for (u32 i = tid; i + 1 < npeaks; i += T)
        if (static_cast<u64>(__ldcg(positions + i)) + row < nwork) ++cnt;
    const u32 total_rows = block_scan_inclusive_1024(cnt, s_tmp);
    if (tid == T - 1) {
        result->n_peaks = npeaks;
        result->n_rows = total_rows;
        result->status = npeaks < 5 ? 3u : 0u;
        result->n_roots = nroots;
    }
}

// ---------------------------------------------------------------------------------------------
// k_pick_cluster: the same orbit walk inside ONE thread-block cluster.  The jump tables live in the distributed
// shared memory of the cluster's CTAs (node c in CTA c / per), every level ends in a hardware cluster barrier
// instead of a global-memory grid barrier, and nothing but the root lists, the orbit and the positions touches
// global memory: ~11 levels of (one DSMEM gather per node + barrier.cluster) instead of 11 grid barriers at
// ~3.5 us each.  Recordings whose candidates do not fit the cluster's shared memory run the identical code on
// the global ping-pong tables (slower, still parallel); beyond the scratch capacity: the one-thread walk.
// ---------------------------------------------------------------------------------------------
constexpr u32 kPickClusterPer = 24576;       // nodes per CTA: 2 tables x 96 KB of dynamic shared memory

// F for one candidate start c (node numbering: A-type row*m for c < nr, then one B-type per root, END = nr + nroots):
// start position, the peak the picker ends on from there, and the node it continues from.
__device__ __forceinline__ void pick_node(u32 c, u32 nr, u32 ncand, u64 ncorr, u32 row, u32 dist, const RootIndex &ri,
                                          u32 &s, u32 &peak, u32 &nxt) {
    const u32 END = ncand;
    nxt = END;
    s = 0xFFFFFFFFu;
    peak = 0;
    if (c >= ncand) return;
    const u64 s64 = c < nr ? static_cast<u64>(c) * row : static_cast<u64>(root_by_id(c - nr, ri)) + dist + 1;
    if (s64 >= ncorr) return;
    s = static_cast<u32>(s64);
    u32 dense;
    first_root_dense(s, ri, dense, peak);
    const u64 sb = static_cast<u64>(peak) + dist + 1;
    const u64 sa = static_cast<u64>(row) * (s / row + 1);
    if (max(sa, sb) < ncorr) nxt = sb >= sa ? nr + dense : static_cast<u32>(sa / row);
}

// J0 for every node, one thread each over the WHOLE GPU (the chains of dependent loads behind F -- root list binary
// searches -- are latency-bound: 8 CTAs of a cluster would need several rounds of them, 148 SMs need one).
__global__ void __launch_bounds__(256)
k_pick_j0(u64 ncorr, u32 row, u32 dist, const RootIndex ri, u32 *__restrict__ positions, u32 max_positions,
          SyncResult *__restrict__ result, PickScratch sc) {
    if (result->status == kSyncRedo) return;
    const u32 nroots = __ldcg(ri.nroots);
    const u32 nr = static_cast<u32>((ncorr + row - 1) / row);
    const u32 ncand = nr + nroots;
    if (ncand + 1 > sc.cap || nr + 1 > max_positions) return;      // k_pick_cluster walks sequentially
    const u32 c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c <= ncand) {
        u32 s, peak, nxt;
        pick_node(c, nr, ncand, ncorr, row, dist, ri, s, peak, nxt);
        sc.cand_s[c] = s;
        sc.cand_peak[c] = peak;
        sc.ja[c] = nxt;
    }
    if (c == 0) {
        // the first start, from the seed (decode.rs:208-209)
        const u32 END = ncand;
        const u32 seed = result->seed_index;
        u32 p1 = 0, start = END;
        u64 s2 = 2ull * row;
        if (seed != kNoSeed) {
            u32 dense;
            first_root_dense(seed, ri, dense, p1);
            const u64 sb = static_cast<u64>(p1) + dist + 1;
            if (sb >= s2) { s2 = sb; start = nr + dense; }
        }
        if (s2 < ncorr) { if (start == END) start = static_cast<u32>(s2 / row); } else start = END;
        positions[0] = p1;
        sc.orbit[0] = start;
    }
}

__global__ void __launch_bounds__(1024, 1)
k_pick_cluster(u64 ncorr, u64 nwork, u32 row, u32 dist, const RootIndex ri, u32 *__restrict__ positions, u32 max_positions,
               SyncResult *__restrict__ result, PickScratch sc) {
    extern __shared__ u32 pc_tab[];             // [2][kPickClusterPer]
    __shared__ u32 s_tmp[32];
    __shared__ u32 s_misc[4];
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const u32 CS = cluster.num_blocks(), rank = cluster.block_rank();
    const u32 tid = threadIdx.x;
    constexpr u32 T = 1024;
    constexpr u32 per = kPickClusterPer;
    const u32 gtid = rank * T + tid, gsize = CS * T;
    if (result->status == kSyncRedo) return;          // the record pool overflowed: the host re-runs the sync stage
    const u32 nroots = __ldcg(ri.nroots);
    const u32 nr = static_cast<u32>((ncorr + row - 1) / row);      // A-type starts row*m < ncorr
    const u32 ncand = nr + nroots;
    const u32 END = ncand;
    if (ncand + 1 > sc.cap || nr + 1 > max_positions) {
        if (rank == 0 && tid == 0) {
            pick_sequential(ncorr, nwork, row, dist, ri, positions, max_positions, result);
            result->n_roots = nroots;
        }
        return;
    }
    const bool in_smem = ncand + 1 <= CS * per;
    u32 *gtab[2] = {sc.ja, sc.jb};
    auto tab_load = [&](u32 which, u32 c) -> u32 {
        if (in_smem) {
            const u32 r = c / per;
            return cluster.map_shared_rank(pc_tab + which * per, r)[c - r * per];
        }
        return __ldcg(gtab[which] + c);
    };
    // the nodes this thread owns
    const u32 c_first = in_smem ? rank * per + tid : gtid;
    const u32 c_limit = in_smem ? min(ncand + 1, (rank + 1) * per) : ncand + 1;
    const u32 c_step = in_smem ? T : gsize;

    // ---- J0 (k_pick_j0) into the cluster's shared memory ----
    if (in_smem) {
        for (u32 c = c_first; c < c_limit; c += c_step) pc_tab[c - rank * per] = __ldcg(sc.ja + c);
    }
    cluster.sync();

    // ---- doubling: orbit[n + 2^k] = J_k[orbit[n]];  J_{k+1} = J_k o J_k ----
    u32 cur = 0;
    const u32 max_events = min(nr + 1, max_positions);   // every event lands in a new row
    for (u32 span = 1; span < max_events; span <<= 1) {
        for (u32 n = gtid; n < span && n + span < max_events; n += gsize) sc.orbit[n + span] = tab_load(cur, __ldcg(sc.orbit + n));
        if ((span << 1) < max_events) {
            for (u32 c = c_first; c < c_limit; c += c_step) {
                const u32 mid = in_smem ? pc_tab[cur * per + (c - rank * per)] : __ldcg(gtab[cur] + c);
                const u32 v = tab_load(cur, mid);
                if (in_smem) pc_tab[(cur ^ 1) * per + (c - rank * per)] = v; else gtab[cur ^ 1][c] = v;
            }
        }
        cluster.sync();
        cur ^= 1;
    }

    // ---- events -> positions (decode.rs:241-253); END is absorbing so events are a prefix of orbit[] ----
    for (u32 n = gtid; n < max_events; n += gsize) {
        const u32 v = __ldcg(sc.orbit + n);
        if (v == END) continue;
        const u32 s = __ldcg(sc.cand_s + v);
        const u32 target = s / row;
        const u32 prev = n == 0 ? 1u : __ldcg(sc.cand_s + __ldcg(sc.orbit + n - 1)) / row;
        for (u32 j = prev; j + 1 < target; ++j) positions[j] = s;      // duplicates pushed by the `while`
        positions[target - 1] = __ldcg(sc.cand_peak + v);
    }
    cluster.sync();                                   // also keeps every CTA's tables alive until all remote reads are done
    if (rank != 0) return;

    // ---- CTA 0: counts ----
    u32 my_events = 0;
    for (u32 n = tid; n < max_events; n += T) my_events += __ldcg(sc.orbit + n) != END;
    const u32 events = block_scan_inclusive_1024(my_events, s_tmp);
    if (tid == T - 1) s_misc[2] = events;
    __syncthreads();
    const u32 nev = s_misc[2];
    const u32 npeaks = nev == 0 ? 1u : __ldcg(sc.cand_s + __ldcg(sc.orbit + nev - 1)) / row;
    u32 cnt = 0;
    for (u32 i = tid; i + 1 < npeaks; i += T)
        if (static_cast<u64>(__ldcg(positions + i)) + row < nwork) ++cnt;
    const u32 total_rows = block_scan_inclusive_1024(cnt, s_tmp);
    if (tid == T - 1) {
        result->n_peaks = npeaks;
        result->n_rows = total_rows;
        result->status = npeaks < 5 ? 3u : 0u;
        result->n_roots = nroots;
    }
}

// ---------------------------------------------------------------------------------------------
// k_gather_rows: aligned rows + final NoFilter/decimate stage fused (decode.rs:122-134, 158-159).
//   out[j*px + c] = f[pos[j] + c*dec]   for j < n_rows, c < px   (px = 2080, dec = work_rate/4160)
// Element 0 of the whole output is 0: dsp::filter with NoFilter never reads signal[0] (dsp.rs:399).
// positions == nullptr: the --no-sync branch, pos[j] = j*row (decode.rs:141-147).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_gather_rows(const float *__restrict__ f, const u32 *__restrict__ positions,
              const SyncResult *__restrict__ result, u32 fixed_rows, u32 row, u32 px, u32 dec,
              float *__restrict__ out) {
    const u32 n_rows = positions ? result->n_rows : fixed_rows;
    for (u32 j = blockIdx.x; j < n_rows; j += gridDim.x) {
        const u64 p = positions ? positions[j] : static_cast<u64>(j) * row;
        // 9 independent loads in flight per thread (px = 2080 = 8.1 x 256): the kernel is latency-bound otherwise
        constexpr u32 U = 9;
        for (u32 c0 = threadIdx.x; c0 < px; c0 += U * blockDim.x) {
            float v[U];
#pragma unroll
            for (u32 u = 0; u < U; ++u) {
                const u32 c = c0 + u * blockDim.x;
                v[u] = c < px ? __ldg(f + p + static_cast<u64>(c) * dec) : 0.f;
            }
#pragma unroll
            for (u32 u = 0; u < U; ++u) {
                const u32 c = c0 + u * blockDim.x;
                if (c < px) out[static_cast<u64>(j) * px + c] = (j == 0 && c == 0) ? 0.f : v[u];
            }
        }
    }
}

}  // namespace aptb200
