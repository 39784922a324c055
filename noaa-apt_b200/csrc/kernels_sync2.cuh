// Fused back half of decode(): demodulation low-pass + sync correlation + peak candidates without ever writing the
// low-passed signal or the correlation to HBM (dsp::filter dsp.rs:386-410 with the Lowpass of decode.rs:95-102, the
// correlation loop and the peak picker of find_sync decode.rs:204-263, row alignment + final decimation
// decode.rs:122-134,158-159).
//
//   k_lowpass_records : e -> (f, box sums, corr in registers / shared memory only) -> per tile of W positions: the tile
//                       maximum of corr, the tile's WEAK SUFFIX RECORDS (corr[p] >= everything later in the tile) and
//                       its STRICT PREFIX RECORDS (corr[p] > everything earlier in the tile), as (position, value) lists.
//   k_resolve_roots   : p is a ROOT (kernels_sync.cuh: no corr[j] > corr[p] for j in (p, p+D]) iff it is a suffix record
//                       of its tile, no tile strictly inside the window has a larger maximum, and the first prefix record
//                       of the window's last tile that exceeds corr[p] lies beyond p+D.  Roots per tile, ascending.
//   (k_pick_links / k_pick_cluster walk the orbit over the roots -- kernels_sync.cuh.)
//   k_gather_rows_lp  : out[j*2080 + c] = f[pos_j + dec*c] with f recomputed from e at just those positions (37 MACs per
//                       pixel), so f never exists in HBM at all.
//
// The kernels' corr values equal the reference's sequential sums to fp32 rounding (box-sum order, like
// kernels_lpsync.cuh); the picker's comparisons are exact on those values.  decode() needs the records of a tile to fit
// the shared pool; a recording that overflows it (silence, ramps: every index a record) reports kSyncRedo and the host
// re-runs the sync stage with the exact-order legacy kernels (k_lowpass_corr / k_corr_generic + k_roots).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_fast.cuh"
#include "kernels_lpsync.cuh"
#include "kernels_sync.cuh"
#include "launch.hpp"

namespace aptb200 {

constexpr int kRecTB = 64;                       // rows of 32 low-passed samples per tile (two rounds of a warp per phase)
constexpr int kRecRowPitch = 36;                 // floats per shared-memory row of 32 (+4: 16-byte accesses of 8
                                                 // consecutive rows hit 8 distinct bank groups)
constexpr int kRecShift = 3;                     // box-sum row r lives in physical row r + 3 (aliases dead e rows)
constexpr int kRecSmemFloats = (kRecTB + kRecShift) * kRecRowPitch;   // shared memory of one warp (9.4 KB)
// one warp per CTA, each waiting for its own tile's samples: the register file limits the warps per SM
__host__ __device__ constexpr int rec_ctas_per_sm(int nt) { return nt > 43 ? 12 : nt > 37 ? 16 : 20; }

__host__ __device__ constexpr int rec_tile_outputs(int pw) {   // W: correlation outputs per tile (multiple of 32)
    return (32 * kRecTB - 18 * 2 * pw - (2 * pw - 1)) / 32 * 32;
}

__device__ __forceinline__ float warp_max_all(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// max over the lanes below / above this one (-inf when there is none)
__device__ __forceinline__ float warp_excl_prefix_max(float v, u32 lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= static_cast<u32>(o)) v = fmaxf(v, t);
    }
    const float t = __shfl_up_sync(0xffffffffu, v, 1);
    return lane == 0 ? -INFINITY : t;
}
__device__ __forceinline__ float warp_excl_suffix_max(float v, u32 lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_down_sync(0xffffffffu, v, o);
        if (lane + o < 32) v = fmaxf(v, t);
    }
    const float t = __shfl_down_sync(0xffffffffu, v, 1);
    return lane == 31 ? -INFINITY : t;
}
__device__ __forceinline__ u32 warp_excl_sum(u32 v, u32 lane, u32 &total) {
    u32 x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= static_cast<u32>(o)) x += t;
    }
    total = __shfl_sync(0xffffffffu, x, 31);
    return x - v;
}

// ------------------------------------------------------------------------------------------------------------------
// k_lowpass_records.  One CTA = one warp = one tile at a time: positions [i0, i0 + W), i0 = tile * W.  Shared memory:
// (TB + 3) rows of 36 floats.
//   stage   : e[i0 - EOFF, i0 + 32*TB) -> rows (logical index m <-> e[i0 - EOFF + m]); samples with index < 1 or >= n
//             are zero (dsp.rs:399: signal[0] is never read)
//   phase 1 : lane = one row of 32 consecutive outputs f[i0 + 32r ..]: the 32+EOFF window in registers as packed pairs,
//             four passes (two parities x two halves) of 8 outputs x NPAIR FFMA2 with warp-uniform tap pairs (the
//             index algebra of kernels_lpsync.cuh); box sums B[n] = f[n] + ... + f[n+BOX-1] of the row straight from the
//             registers (the BOX-1 values of the next row come from the neighbouring lane by shuffle; rounds run from the
//             last row block to the first so that lane 31 gets them from the block done before) -> B rows
//   phase 3 : lane = 32 consecutive correlation outputs: streams its 32 + 18*BOX box sums (LDS.128, conflict-free) into
//             16 packed accumulators (19 signed box sums per output, decode.rs:188-198)
//   records : per-lane maxima -> warp scans -> flags; the tile's suffix and prefix records go to the pool in index order.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(float *dst, const float *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(Rec *dst, const Rec *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <int NT, int PW>
__global__ void __launch_bounds__(32, rec_ctas_per_sm(NT))
k_lowpass_records(const float *__restrict__ e, u64 n, u64 ncorr, const __grid_constant__ LpTaps taps, SyncCtl *__restrict__ ctl,
                  TileDesc *__restrict__ desc, Rec *__restrict__ pool, u32 pool_cap, u32 region, u32 ntiles) {
    constexpr int BOX = 2 * PW;
    constexpr int LOOK = 18 * BOX;
    constexpr int TB = kRecTB;
    constexpr int W = rec_tile_outputs(PW);
    constexpr int NI = W / 32;                              // correlation items (rows of 32 outputs) per tile
    constexpr int RD = (NI + 31) / 32;                      // rounds of the correlation phase
    static_assert(TB % 32 == 0 && NI >= 1 && RD <= 2, "one or two rounds of correlation items");
    static_assert(NT % 2 == 1, "odd tap counts only (Kaiser design, filters.rs:79)");
    constexpr int EOFF = (NT - 1 + 3) / 4 * 4;
    constexpr int NPAIR = (NT + 1) / 2;
    constexpr int WN = EOFF + 32;                           // window of one row, floats
    constexpr int LE = 32 * TB + EOFF;                      // staged e samples
    static_assert((LE + 31) / 32 <= TB + 2, "e rows");
    static_assert(EOFF - (NT - 1) >= 0 && EOFF + 31 + 1 < WN + 1, "window of a row");
    constexpr int PITCH = kRecRowPitch;

    extern __shared__ __align__(16) float rec_smem[];
    float *const s = rec_smem;
    const u32 lane = threadIdx.x & 31;

    // e[i0 - EOFF, i0 + 32*TB) -> rows of s (logical index m <-> e[i0 - EOFF + m]); samples with index < 1 or >= n are
    // zero (dsp.rs:399: signal[0] is never read).  Interior tiles: 16-byte cp.async, no registers, no waiting here.
    auto stage = [&](u32 tile) {
        const long long g0 = static_cast<long long>(tile) * W - EOFF;
        if (g0 >= 4 && static_cast<u64>(g0) + LE <= n) {
            const float *src = e + g0;
#pragma unroll 4
            for (u32 q4 = lane; q4 < LE / 4; q4 += 32) {
                const u32 m = 4 * q4;
                cp_async16(s + (m >> 5) * PITCH + (m & 31), src + m);
            }
        } else {
            for (u32 q4 = lane; q4 < LE / 4; q4 += 32) {
                const u32 m = 4 * q4;
                const long long g = g0 + m;
                float4 v;
                v.x = g >= 1 && static_cast<u64>(g) < n ? __ldg(e + g) : 0.f;
                v.y = g + 1 >= 1 && static_cast<u64>(g + 1) < n ? __ldg(e + g + 1) : 0.f;
                v.z = g + 2 >= 1 && static_cast<u64>(g + 2) < n ? __ldg(e + g + 2) : 0.f;
                v.w = g + 3 >= 1 && static_cast<u64>(g + 3) < n ? __ldg(e + g + 3) : 0.f;
                *reinterpret_cast<float4 *>(s + (m >> 5) * PITCH + (m & 31)) = v;
            }
        }
        cp_async_commit_group();
    };
    // Tiles are dealt out statically (every tile costs the same): CTA b takes the tiles b, b + gridDim.x, ...  No tickets:
    // two same-address atomics per tile (ticket + pool cursor, 11.7 k of them on one cache line) were what kept the first
    // version at ~52 us whatever the occupancy.
    u32 tile = blockIdx.x;
    if (tile < ntiles) stage(tile);
    for (u32 it = 0; tile < ntiles; ++it) {
        const u32 next = blockIdx.x + (it + 1) * gridDim.x;
        cp_async_wait_all();
        __syncwarp();
        const u64 i0 = static_cast<u64>(tile) * W;

        // ---- phase 1: low-pass + box sums, row blocks from the last to the first ----
        float carry[BOX - 1];
#pragma unroll
        for (int k = 0; k < BOX - 1; ++k) carry[k] = 0.f;
#pragma unroll 1
        for (int rb = TB / 32 - 1; rb >= 0; --rb) {
            const u32 r = 32 * rb + lane;
            const float *row = s + r * PITCH;
            // One window sample x the taps of two neighbouring outputs: FFMA2 R.F32 (broadcast) x UR.pair + R.pair, the form that
            // runs at 2.9 clk per sub-partition; the packed-window form (R.pair x UR.pair) used here before takes 5.0 clk
            // and made this phase the kernel's bound (profiles/r02_fma_rate_bench.txt).
            float w[WN];
#pragma unroll
            for (int k = 0; k < WN / 4; ++k) {
                const float4 q = *reinterpret_cast<const float4 *>(row + 4 * k + 4 * (k >> 3));
                w[4 * k] = q.x; w[4 * k + 1] = q.y; w[4 * k + 2] = q.z; w[4 * k + 3] = q.w;
            }
            float fr[32 + BOX];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                f32x2 acc[8];
#pragma unroll
                for (int v = 0; v < 8; ++v) acc[v] = 0ull;
#pragma unroll
                for (int j = -1; j < NT; ++j) {
                    const f32x2 t2 = pack2(taps.p[j + 1].x, taps.p[j + 1].y);   // (c[j], c[j+1]): outputs 2p and 2p+1 from sample EOFF+2p-j
#pragma unroll
                    for (int v = 0; v < 8; ++v) {
                        const float x = w[EOFF + 2 * (8 * h + v) - j];
                        acc[v] = fma2(pack2(x, x), t2, acc[v]);
                    }
                }
#pragma unroll
                for (int v = 0; v < 8; ++v) unpack2(acc[v], fr[16 * h + 2 * v], fr[16 * h + 2 * v + 1]);
            }
            // the first BOX-1 values of the next row: lane + 1, or (lane 31) the row block done before this one
#pragma unroll
            for (int k = 0; k < BOX - 1; ++k) {
                const float nb = __shfl_down_sync(0xffffffffu, fr[k], 1);
                fr[32 + k] = lane == 31 ? carry[k] : nb;
            }
            fr[32 + BOX - 1] = 0.f;
#pragma unroll
            for (int k = 0; k < BOX - 1; ++k) carry[k] = __shfl_sync(0xffffffffu, fr[k], 0);
            // box sums through pair sums P[k] = f[2k] + f[2k+1] (same order of additions as kernels_lpsync.cuh)
            float pr[(32 + BOX) / 2];
#pragma unroll
            for (int k = 0; k < (32 + BOX) / 2; ++k) pr[k] = fr[2 * k] + fr[2 * k + 1];
            float b[32];
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                float sm = pr[u + 1];
#pragma unroll
                for (int k = 2; k < PW; ++k) sm += pr[u + k];
                b[2 * u] = pr[u] + sm;
                b[2 * u + 1] = (fr[2 * u + 1] + sm) + fr[2 * u + BOX];
            }
            __syncwarp();                                   // every lane has read its window: the rows may be overwritten
            float *brow = s + (r + kRecShift) * PITCH;
#pragma unroll
            for (int k = 0; k < 8; ++k)
                *reinterpret_cast<float4 *>(brow + 4 * k) = make_float4(b[4 * k], b[4 * k + 1], b[4 * k + 2], b[4 * k + 3]);
        }
        __syncwarp();

        // ---- phase 3: correlation, RD rounds of 32 items ----
        float c[RD][32];
        float gm[RD][4];                                    // maxima of the lane's four groups of 8 outputs
        float mx[RD];
        u32 vmask[RD];
#pragma unroll
        for (int rd = 0; rd < RD; ++rd) {
            const u32 q = 32 * rd + lane;
            const u32 qa = q < NI ? q : NI - 1;             // idle lanes of the last round re-read the last item
            const float *brow = s + (qa + kRecShift) * PITCH;
            // Packed adds (FFMA2 with an immediate +-1: 5.0 clk per warp instruction for 64 adds; scalar FADD would be 1.16 clk
            // for 32) on purpose: the kernel is bound by instruction issue, not by the FMA pipe, and the scalar variant -- twice
            // the instructions -- measured 6 us slower (profiles/r02_fma_rate_bench.txt, DESIGN.md 3.2).
            const f32x2 plus1 = pack2(1.f, 1.f), minus1 = pack2(-1.f, -1.f);
            f32x2 acc[16];
#pragma unroll
            for (int v = 0; v < 16; ++v) acc[v] = 0ull;
#pragma unroll
            for (int k = 0; k < (32 + LOOK) / 4; ++k) {
                const float4 qv = *reinterpret_cast<const float4 *>(brow + 4 * k + 4 * (k >> 3));
                const f32x2 val[2] = {pack2(qv.x, qv.y), pack2(qv.z, qv.w)};
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int m = 4 * k + 2 * hh;           // box index relative to the item (compile time, even)
#pragma unroll
                    for (int bb = 0; bb < 19; ++bb) {
                        const int v = m - BOX * bb;         // first output of the pair run bb contributes to
                        if (v >= 0 && v < 32) {
                            // runs: bb = 0 '-', then (-,+) x 7 for bb = 1..14, then '-' x 4 (decode.rs:188-198)
                            const bool plus = bb >= 1 && bb <= 14 && (bb % 2 == 0);
                            acc[v / 2] = fma2(val[hh], plus ? plus1 : minus1, acc[v / 2]);
                        }
                    }
                }
            }
#pragma unroll
            for (int v = 0; v < 16; ++v) unpack2(acc[v], c[rd][2 * v], c[rd][2 * v + 1]);
            // outputs beyond the tile or beyond the correlation: -inf (only the last lanes of a tile / the last tile)
            const u64 gi = i0 + 32ull * q;
            const u32 nvalid = q < NI && gi < ncorr ? static_cast<u32>(ncorr - gi < 32 ? ncorr - gi : 32) : 0u;
            vmask[rd] = nvalid >= 32 ? 0xffffffffu : (1u << nvalid) - 1u;
            if (nvalid < 32) {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (static_cast<u32>(j) >= nvalid) c[rd][j] = -INFINITY;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float m8 = c[rd][8 * g];
#pragma unroll
                for (int j = 1; j < 8; ++j) m8 = fmaxf(m8, c[rd][8 * g + j]);
                gm[rd][g] = m8;
            }
            mx[rd] = fmaxf(fmaxf(gm[rd][0], gm[rd][1]), fmaxf(gm[rd][2], gm[rd][3]));
        }

        // ---- records: bounds from outside the lane by warp scans, then 8 independent chains of 8 per round ----
        float all[RD], pm[RD], sx[RD];
#pragma unroll
        for (int rd = 0; rd < RD; ++rd) all[rd] = warp_max_all(mx[rd]);
#pragma unroll
        for (int rd = 0; rd < RD; ++rd) {
            float before = -INFINITY, after = -INFINITY;
#pragma unroll
            for (int r2 = 0; r2 < RD; ++r2) {
                if (r2 < rd) before = fmaxf(before, all[r2]);
                if (r2 > rd) after = fmaxf(after, all[r2]);
            }
            pm[rd] = fmaxf(before, warp_excl_prefix_max(mx[rd], lane));
            sx[rd] = fmaxf(after, warp_excl_suffix_max(mx[rd], lane));
        }
        u32 ms[RD], mp[RD];
#pragma unroll
        for (int rd = 0; rd < RD; ++rd) {
            float sb[4], pb[4];
            sb[3] = sx[rd];
            sb[2] = fmaxf(sb[3], gm[rd][3]);
            sb[1] = fmaxf(sb[2], gm[rd][2]);
            sb[0] = fmaxf(sb[1], gm[rd][1]);
            pb[0] = pm[rd];
            pb[1] = fmaxf(pb[0], gm[rd][0]);
            pb[2] = fmaxf(pb[1], gm[rd][1]);
            pb[3] = fmaxf(pb[2], gm[rd][2]);
            u32 a = 0, p = 0;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float run = sb[g];
#pragma unroll
                for (int j = 8 * g + 7; j >= 8 * g; --j) {
                    if (!(run > c[rd][j])) a |= 1u << j;           // weak suffix record: nothing later is larger
                    run = fmaxf(run, c[rd][j]);
                }
                run = pb[g];
#pragma unroll
                for (int j = 8 * g; j < 8 * g + 8; ++j) {
                    if (c[rd][j] > run) p |= 1u << j;              // strict prefix record: larger than everything earlier
                    run = fmaxf(run, c[rd][j]);
                }
            }
            ms[rd] = a & vmask[rd];
            mp[rd] = p & vmask[rd];
        }
        u32 os[RD], op[RD], tot_s = 0, tot_p = 0;
#pragma unroll
        for (int rd = 0; rd < RD; ++rd) {
            u32 ts, tp;
            os[rd] = warp_excl_sum(__popc(ms[rd]), lane, ts) + tot_s;
            op[rd] = warp_excl_sum(__popc(mp[rd]), lane, tp) + tot_p;
            tot_s += ts;
            tot_p += tp;
        }
        // the tile's own region of the pool; only a tile with more than `region` records (long monotone stretches) takes its
        // space from the shared overflow area behind the regions (region == 0: everything comes from there)
        u32 base = tile * region;
        if (tot_s + tot_p > region) {                       // warp-uniform
            if (lane == 0) base = ntiles * region + atomicAdd(&ctl->pool_cursor, tot_s + tot_p);
            base = __shfl_sync(0xffffffffu, base, 0);
        }
        const bool fits = static_cast<u64>(base) + tot_s + tot_p <= pool_cap;
        if (fits) {
            // Every lane writes its own records straight from the registers that hold its 32 correlation values: one
            // predicated 8-byte store per (output, list), 128 per tile, all independent.  (The first version parked the values
            // in shared memory and ran a `while (mask)` loop per lane -- find-first-set, LDS, store, a dependent chain whose
            // trip count is the busiest lane's: a third of the kernel's time in the ncu source view.)
#pragma unroll
            for (int rd = 0; rd < RD; ++rd) {
                const u32 p0 = static_cast<u32>(i0) + 32 * (32 * rd + lane);
                u32 is = base + os[rd], ip = base + tot_s + op[rd];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (ms[rd] & (1u << j)) { pool[is] = Rec{p0 + j, c[rd][j]}; ++is; }
                    if (mp[rd] & (1u << j)) { pool[ip] = Rec{p0 + j, c[rd][j]}; ++ip; }
                }
            }
        }
        float tmax = all[0];
#pragma unroll
        for (int rd = 1; rd < RD; ++rd) tmax = fmaxf(tmax, all[rd]);
        if (lane == 0) {
            if (!fits) atomicExch(&ctl->overflow, 1u);
            desc[tile] = TileDesc{base, fits ? tot_s : 0u, fits ? tot_p : 0u, tmax};
        }
        __syncwarp();
        tile = next;
        if (tile < ntiles) stage(tile);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// k_resolve_roots: warp per tile.  The tile's suffix records and the prefix records of the two tiles a window can end in
// are staged in shared memory; surviving roots go to root_list (ascending, at the tile's pool offset) and get dense ids
// from an atomic cursor (ids are labels: any disjoint ranges do) -> tile_base[t], root position by id -> by_id.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kResolveThreads = 256;
constexpr int kResolveCache = 192;               // records of one list kept in shared memory (longer lists: global); 21 KB per CTA: 10 CTAs per SM

// first record of the ascending list L[0..np) whose value exceeds v; np if none
__device__ __forceinline__ u32 first_exceeding(const Rec *L, u32 np, float v) {
    u32 lo = 0, hi = np;
    while (lo < hi) {
        const u32 mid = (lo + hi) >> 1;
        if (L[mid].val > v) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__device__ __forceinline__ TileDesc shfl_desc(const TileDesc &d, u32 src) {
    TileDesc r;
    r.off = __shfl_sync(0xffffffffu, d.off, src);
    r.ns = __shfl_sync(0xffffffffu, d.ns, src);
    r.np = __shfl_sync(0xffffffffu, d.np, src);
    r.tmax = __shfl_sync(0xffffffffu, d.tmax, src);
    return r;
}

__global__ void __launch_bounds__(kResolveThreads)
k_resolve_roots(const TileDesc *__restrict__ desc, const Rec *__restrict__ pool, u32 ntiles, u32 tile_w, u32 dist, u64 ncorr,
                u32 *__restrict__ root_list, u32 *__restrict__ root_count, u32 *__restrict__ tile_base, u32 *__restrict__ by_id,
                SyncCtl *__restrict__ ctl, SyncResult *__restrict__ result) {
    __shared__ Rec s_p[kResolveThreads / 32][2][kResolveCache];
    __shared__ Rec s_s[kResolveThreads / 32][kResolveCache];
    __shared__ u32 s_r[kResolveThreads / 32][kResolveCache];
    if (*reinterpret_cast<volatile u32 *>(&ctl->overflow) != 0) {
        if (blockIdx.x == 0 && threadIdx.x == 0) result->status = kSyncRedo;
        return;
    }
    __shared__ u32 s_cnt[kResolveThreads / 32];
    __shared__ u32 s_base;
    const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const u32 t = blockIdx.x * (kResolveThreads / 32) + warp;
    u32 cnt = 0, list_off = 0;
    if (t < ntiles) {
        // one parallel load: the descriptors of tiles t .. tlo+1 (a window starting in tile t ends in tile tlo or tlo+1)
        const u32 tlo = t + dist / tile_w;                  // (t*W + D) / W
        const u32 span = min(tlo + 1 - t, 31u);
        TileDesc mine{0u, 0u, 0u, -INFINITY};
        if (lane <= span && t + lane < ntiles) mine = desc[t + lane];
        const TileDesc d = shfl_desc(mine, 0);
        const TileDesc dl[2] = {shfl_desc(mine, min(tlo - t, 31u)), shfl_desc(mine, min(tlo + 1 - t, 31u))};
        // between[k] = max of tmax over tiles t+1 .. t+k (inclusive prefix maximum over the lanes 1..k)
        float between = lane == 0 ? -INFINITY : mine.tmax;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(0xffffffffu, between, o);
            if (lane >= static_cast<u32>(o)) between = fmaxf(between, v);
        }
        // second parallel load: the tile's suffix records and the prefix records of the two end tiles
        const Rec *lst[2] = {nullptr, nullptr};
        u32 lnp[2] = {0, 0};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const u32 tt = tlo + k;
            if (tt < ntiles && tt > t && tt - t <= 31) {
                lnp[k] = dl[k].np;
                const Rec *src = pool + dl[k].off + dl[k].ns;
                if (dl[k].np <= kResolveCache) {
                    for (u32 i = lane; i < dl[k].np; i += 32) cp_async8(&s_p[warp][k][i], src + i);
                    lst[k] = s_p[warp][k];
                } else {
                    lst[k] = src;
                }
            }
        }
        const Rec *cand = pool + d.off;
        if (d.ns <= kResolveCache) {
            for (u32 i = lane; i < d.ns; i += 32) cp_async8(&s_s[warp][i], cand + i);
            cand = s_s[warp];
        }
        // all three lists are in flight together (a load-then-store loop pays one L2 round trip per 32 records)
        cp_async_commit_group();
        cp_async_wait_all();
        __syncwarp();
        list_off = d.off;
        const u32 tile_begin = t * tile_w;                  // correlation indices fit 32 bits (N_w < 2^32)
        const u32 last = static_cast<u32>(ncorr - 1);
        for (u32 c0 = 0; c0 < d.ns; c0 += 32) {
            const u32 ci = c0 + lane;
            bool root = false;
            u32 pos = 0, te = t, end = 0;
            float val = 0.f;
            if (ci < d.ns) {
                const Rec r = cand[ci];
                pos = r.pos;
                val = r.val;
                end = last - pos < dist ? last : pos + dist;          // last index of the window (p, p+D]
                root = true;
                te = t + (end - tile_begin) / tile_w;
            }
            // tiles strictly inside the window: t+1 .. te-1
            const u32 inner = te > t + 1 ? min(te - 1 - t, 31u) : 0u;
            const float bmax = __shfl_sync(0xffffffffu, between, inner);
            if (root && te > t) {
                if (inner > 0 && bmax > val) root = false;
                if (root) {
                    const Rec *L;
                    u32 np;
                    if (te == tlo && lst[0]) { L = lst[0]; np = lnp[0]; }
                    else if (te == tlo + 1 && lst[1]) { L = lst[1]; np = lnp[1]; }
                    else { const TileDesc dd = desc[te]; L = pool + dd.off + dd.ns; np = dd.np; }
                    const u32 k = first_exceeding(L, np, val);
                    if (k < np && L[k].pos <= end) root = false;
                }
            }
            const u32 bal = __ballot_sync(0xffffffffu, root);
            if (root) {
                const u32 k = cnt + __popc(bal & ((1u << lane) - 1));
                root_list[d.off + k] = pos;
                if (k < kResolveCache) s_r[warp][k] = pos;
            }
            cnt += __popc(bal);
        }
    }
    // dense ids: one atomic per CTA (its tiles take consecutive ranges) -- one per tile meant 5850 same-address atomics, all
    // issued within the same few microseconds of a kernel that runs as a single wave
    if (lane == 0) s_cnt[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 total = 0;
#pragma unroll
        for (int w = 0; w < kResolveThreads / 32; ++w) total += s_cnt[w];
        s_base = total ? atomicAdd(&ctl->root_cursor, total) : 0u;
    }
    __syncthreads();
    if (t < ntiles) {
        u32 base = s_base;
        for (u32 w = 0; w < warp; ++w) base += s_cnt[w];
        if (lane == 0) {
            root_count[t] = cnt;
            tile_base[t] = base;
        }
        for (u32 k = lane; k < cnt; k += 32) by_id[base + k] = k < kResolveCache ? s_r[warp][k] : root_list[list_off + k];
    }
    // seed of the peak list: first i <= D with corr[i] > 0.0 (decode.rs:208-209 + the else-if at :250) = the first
    // prefix record with a positive value
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        u32 seed = kNoSeed;
        for (u32 tt = 0; tt < ntiles && static_cast<u64>(tt) * tile_w <= dist && seed == kNoSeed; ++tt) {
            const TileDesc dd = desc[tt];
            const Rec *L = pool + dd.off + dd.ns;
            const u32 k = first_exceeding(L, dd.np, 0.f);
            if (k < dd.np && L[k].pos <= dist) seed = L[k].pos;
        }
        result->seed_index = seed;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// k_gather_rows_lp: aligned rows + final decimation, with the low-pass evaluated only where a pixel needs it:
//   out[j*px + c] = sum_{jj < NT} e[pos_j + DEC*c - jj] * lp[jj]      (samples with index < 1 contribute nothing)
// One CTA per half row: the e span of the half row sits in shared memory; a thread computes 4 consecutive pixels from
// a 16-byte aligned window of its own.  Element 0 of the whole output is 0 (NoFilter never reads signal[0], dsp.rs:399).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kGatherLpThreads = 288;            // 2080 / 2 = 1040 pixels = 260 quads per half row

__device__ __forceinline__ void cp_async4_zfill(float *dst, const float *src, bool valid) {
    const u32 bytes = valid ? 4u : 0u;            // src-size 0: nothing is read, the destination is zero-filled
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Four pixels of one thread: the window starts OFF samples into the 16-byte aligned floats at `src` (OFF = the row position's
// alignment, compile time: the register indices are fixed per variant).  One window sample x the taps it has in two
// neighbouring pixels (DEC samples apart): FFMA2 R.F32 (broadcast) x UR.pair + R.pair, NT + DEC of them per pixel pair --
// half the instructions of the scalar form and 2.9 clk each (the packed-window form R.pair x UR.pair takes 5.0;
// profiles/r02_fma_rate_bench.txt).
template <int NT, int DEC, int OFF>
__device__ __forceinline__ void gather_quad(const float *src, const LpTaps &lp, float (&acc)[4]) {
    constexpr int EOFF = (NT - 1 + 3) / 4 * 4;
    constexpr int WIN = (OFF + EOFF + 3 * DEC + 1 + 3) / 4 * 4;     // floats read for the 4 pixels
    static_assert(EOFF - (NT - 1) >= 0 && OFF + EOFF + 3 * DEC < WIN && NT + DEC <= 72, "window");
    float w[WIN];
#pragma unroll
    for (int k = 0; k < WIN / 4; ++k) {
        const float4 q = *reinterpret_cast<const float4 *>(src + 4 * k);
        w[4 * k] = q.x; w[4 * k + 1] = q.y; w[4 * k + 2] = q.z; w[4 * k + 3] = q.w;
    }
    f32x2 acc2[2] = {0ull, 0ull};
#pragma unroll
    for (int j = -DEC; j < NT; ++j) {
        const f32x2 t2 = pack2(lp.pd[j + DEC].x, lp.pd[j + DEC].y);   // (c[j], c[j+DEC])
#pragma unroll
        for (int pp = 0; pp < 2; ++pp) {
            const float x = w[OFF + EOFF + DEC * (2 * pp) - j];       // tap j of pixel 2pp, tap j+DEC of pixel 2pp+1
            acc2[pp] = fma2(pack2(x, x), t2, acc2[pp]);
        }
    }
    unpack2(acc2[0], acc[0], acc[1]);
    unpack2(acc2[1], acc[2], acc[3]);
}

// Persistent CTAs; the e span of the NEXT half row is copied into the other shared-memory buffer while the current one is
// computed.  A row starts at an arbitrary sample, so the span is staged from the 16-byte aligned address below it (16-byte
// cp.async: a quarter of the copy instructions of the first version, whose 4-byte copies kept the integer pipe busier than
// the FMA pipe) and the remainder (0..3 samples) selects one of four compute variants.
template <int NT, int DEC>
__global__ void __launch_bounds__(kGatherLpThreads)
k_gather_rows_lp(const float *__restrict__ e, u64 n, const u32 *__restrict__ positions, const SyncResult *__restrict__ result,
                 u32 fixed_rows, u32 row, u32 px, const __grid_constant__ LpTaps lp, float *__restrict__ out) {
    constexpr int EOFF = (NT - 1 + 3) / 4 * 4;
    constexpr int PARTS = 2;
    extern __shared__ __align__(16) float g_smem[];
    const u32 n_rows = positions ? (result->status == 0 ? result->n_rows : 0u) : fixed_rows;
    const u32 part_px = (px / PARTS + 3) / 4 * 4;              // pixels per part (multiple of 4)
    const u32 span = DEC * part_px + EOFF + 12;                 // staged samples per part (multiple of 4), incl. the alignment slack
    const u32 items = n_rows * PARTS;
    const bool out_aligned = (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    const bool e_aligned = (reinterpret_cast<uintptr_t>(e) & 15) == 0;
    // sample index of buf[0] of an item, and the offset of the row's window in it
    auto origin = [&](u32 item, long long &a0) -> u32 {
        const u32 j = item / PARTS, part = item % PARTS;
        const u64 p = positions ? positions[j] : static_cast<u64>(j) * row;
        const long long g0 = static_cast<long long>(p) + static_cast<long long>(DEC) * (part * part_px) - EOFF;
        a0 = g0 & ~3ll;                                            // floor to a multiple of 4 (also for negative g0)
        return static_cast<u32>(g0 - a0);
    };
    auto stage = [&](u32 item, float *buf) {
        long long a0;
        origin(item, a0);
        if (e_aligned && a0 >= 4 && static_cast<u64>(a0) + span <= n) {    // interior: no bounds to check (sample 0 is not inside)
            const float *src = e + a0;
            for (u32 i = 4 * threadIdx.x; i < span; i += 4 * blockDim.x) cp_async16(buf + i, src + i);
        } else {
            for (u32 i = threadIdx.x; i < span; i += blockDim.x) {
                const long long g = a0 + i;
                const bool ok = g >= 1 && static_cast<u64>(g) < n;    // dsp.rs:399: signal[0] is never read
                cp_async4_zfill(buf + i, ok ? e + g : e, ok);
            }
        }
    };
    u32 item = blockIdx.x;
    if (item < items) stage(item, g_smem);
    cp_async_commit();
    for (u32 it = 0; item < items; item += gridDim.x, ++it) {
        const float *cur = g_smem + (it & 1) * span;
        if (item + gridDim.x < items) stage(item + gridDim.x, g_smem + ((it + 1) & 1) * span);
        cp_async_commit();
        cp_async_wait<1>();                                     // this thread's copies of the current buffer have landed
        __syncthreads();                                        // ... and everybody else's
        const u32 j = item / PARTS, part = item % PARTS;
        long long a0;
        const u32 off = origin(item, a0);                       // CTA-uniform
        const u32 c_begin = part * part_px;
        const u32 c_end = min(px, c_begin + part_px);
        for (u32 c4 = 4 * threadIdx.x; c_begin + c4 < c_end; c4 += 4 * blockDim.x) {
            float acc[4];
            const float *src = cur + DEC * c4;                  // 16-byte aligned: DEC * c4 and span are multiples of 4
            switch (off) {
            case 0: gather_quad<NT, DEC, 0>(src, lp, acc); break;
            case 1: gather_quad<NT, DEC, 1>(src, lp, acc); break;
            case 2: gather_quad<NT, DEC, 2>(src, lp, acc); break;
            default: gather_quad<NT, DEC, 3>(src, lp, acc); break;
            }
            const u32 c = c_begin + c4;
            float *dst = out + static_cast<u64>(j) * px + c;
            if (j == 0 && c == 0) acc[0] = 0.f;
            if (out_aligned && c + 3 < c_end) {
                *reinterpret_cast<float4 *>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
            } else {
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (c + u < c_end) dst[u] = acc[u];
            }
        }
        __syncthreads();                                        // the buffer is free for the copy two items ahead
    }
}

}  // namespace aptb200
