// Tiled polyphase resampler fused with the envelope demodulator (fast_resampling dsp.rs:186-289 + demodulate
// dsp.rs:350-383), written for sm_100a.  It served L = 13 until kernels_ut.cuh replaced it there (92 -> 62 us) and
// still serves other small interpolation factors (L <= 13 groups, e.g. L = 26); the mbarrier / TMA / packed-fp32
// helpers below are shared by both.
//
// Formulation.  y[k] = sum_x h[x*L - k*M] * X[x].  Outputs k and k + P_out (P_out = lcm(8, L)) use the
// same taps on inputs shifted by P_in = P_out*M/L, so per "group" g (outputs 8g..8g+7 of a super-period)
//     acc[r][q] += T_g[u][r] * X[tile_x0 + q*P_in + w0_g + u]        r < 8, q < QT
// with w0_g the first input sample the group touches (rounded down to a multiple of 4 for 16-byte loads)
// and T_g the zero-padded slice of h its outputs see.  The group's two halves (outputs 0..3 / 4..7) have
// windows offset by `shift` samples, so the first shift/16 loop iterations skip half B and the last skip A.
//
// Structure.  One persistent, warp-specialised CTA per SM:
//   producer warp  : 1-D TMA bulk copies (cp.async.bulk -> UBLKCP) of the next tile's 32 input rows + one
//                    halo row into the free row stage (2 stages), completion on an mbarrier;
//   G compute warps: one per group.  A warp's 32 lanes are KS=4 interleaved slices of the sample axis x 8 row
//                    lanes; a thread owns 8 outputs x 4 rows as 16 packed fp32x2 accumulators.  Per loop
//                    iteration: 4 LDS.128 of samples (the 8 row lanes of a quarter-warp hit 8 distinct 16-byte
//                    bank groups because the row pitch/4 is odd), 8 warp-broadcast LDS.128 of taps (4 distinct
//                    addresses skewed across bank groups) and 64 FFMA2 (fma.rn.f32x2: tap pair x broadcast
//                    sample).  The four slices' partial sums go to shared-memory planes;
//   E epilogue warps: sum the planes, turn (r[k-1], r[k]) into the envelope (dsp.rs:373) and store float4 --
//                    while the compute warps are already on the next tile.  The resampled signal itself never
//                    reaches HBM.  r[K0-1] comes from the halo row (window of the last group of the previous
//                    super-period), computed by the last compute warp.
// Stages are handed over with full/empty mbarriers; the tap table is bulk-copied once per CTA.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_generic.cuh"
#include "launch.hpp"

namespace aptb200 {

// ---- mbarrier / TMA bulk-copy wrappers (PTX ISA: cp.async.bulk, mbarrier) -------------------------
__device__ __forceinline__ u32 smem_u32(const void *p) { return static_cast<u32>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(void *bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(void *bar, u32 parity) {
    u32 ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"   // suspend-time hint: sleep, don't spin
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(void *bar, u32 parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// global -> shared bulk copy, `bytes` a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, u32 bytes, void *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// warm L2 with a span of global memory (no shared-memory destination, no completion tracking)
__device__ __forceinline__ void tma_prefetch_l2(const void *src, u32 bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

constexpr int kTileR = 8, kTileH = 4, kTileQ = 4, kTileKS = 4;
constexpr int kTileRowLanes = 32 / kTileKS;           // 8
constexpr int kTileQT = kTileRowLanes * kTileQ;       // 32 rows per tile

// ---- packed fp32x2 helpers: one FFMA2 issue slot does two FMAs (each half rounded on its own) ----
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ float4 lds128(u32 addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

// One half (4 outputs, as two packed pairs) x 4 rows x the 4 consecutive samples of one 16-byte chunk.
// acc[p][j] packs outputs (2p, 2p+1) of row j; the tap pair comes straight out of the LDS.128 register quad,
// the sample is duplicated into both lanes of the packed operand.
__device__ __forceinline__ void half_fma2(f32x2 (&acc)[2][kTileQ], u32 tap_addr, const float4 (&s)[kTileQ]) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float4 tp = lds128(tap_addr + 16 * u);  // taps of outputs r = 0..3 for sample u of the chunk
        const f32x2 t01 = pack2(tp.x, tp.y), t23 = pack2(tp.z, tp.w);
#pragma unroll
        for (int j = 0; j < kTileQ; ++j) {
            const float sv = u == 0 ? s[j].x : u == 1 ? s[j].y : u == 2 ? s[j].z : s[j].w;
            const f32x2 sv2 = pack2(sv, sv);
            acc[0][j] = fma2(t01, sv2, acc[0][j]);
            acc[1][j] = fma2(t23, sv2, acc[1][j]);
        }
    }
}

__device__ __forceinline__ void mbar_arrive(void *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

constexpr int kWsEpilogueWarps = 6;

// group_xs[g] = w0_g, the (4-aligned) first input sample of group g relative to its row.
template <bool ENVELOPE>
__global__ void __launch_bounds__(32 * (13 + kWsEpilogueWarps + 1), 1)
k_polyphase_ws(const float *__restrict__ signal, u64 len, const float *__restrict__ tile_taps,
               const u32 *__restrict__ group_xs, TilePlan tp, u64 nout, u64 tile_begin, u64 ntiles, float cosphi2,
               float sinphi, float *__restrict__ out) {
    // tiles [tile_begin, ntiles) are computed; `signal` may be a biased pointer into a chunk buffer (signal + x is
    // valid for every sample x those tiles touch), `len` is always the length of the whole signal
    constexpr int Q = kTileQ, KS = kTileKS, QT = kTileQT, E = kWsEpilogueWarps;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // layout: [8 mbarriers + halo, 128 B][taps][stage 0: rows, halo row][stage 1][planes]
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(smem_raw);
    unsigned long long *bar_taps = bars + 0;
    unsigned long long *full_rows = bars + 1;     // [2] TMA -> compute
    unsigned long long *empty_rows = bars + 3;    // [2] compute -> producer
    unsigned long long *full_p = bars + 5;        // compute -> epilogue (planes + halo written)
    unsigned long long *empty_p = bars + 6;       // epilogue -> compute (planes consumed)
    float *s_halo = reinterpret_cast<float *>(bars + 8);
    float *s_taps = reinterpret_cast<float *>(smem_raw + 128);
    float *s_stage0 = s_taps + tp.groups * tp.group_stride;
    float *s_planes = s_stage0 + 2 * tp.stage_floats;

    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 G = tp.groups;
    const u32 tile_out = QT * tp.p_out;

    if (tid == 0) {
        mbar_init(bar_taps, 1);
        mbar_init(full_rows + 0, 1);
        mbar_init(full_rows + 1, 1);
        mbar_init(empty_rows + 0, G);
        mbar_init(empty_rows + 1, G);
        mbar_init(full_p, G);
        mbar_init(empty_p, E);
        fence_mbar_init();
    }
    __syncthreads();

    // Warp roles.  Warps are spread over the 4 SM sub-partitions round-robin (warp % 4); with 13 compute warps
    // sub-partition 0 gets four of them and the others three, so the producer (light) goes to sub-partition 0 and
    // the epilogue warps to the other three.
    const u32 prod_warp = (G + 3) / 4 * 4;                 // first warp index >= G on sub-partition 0
    const bool is_producer = warp == prod_warp;
    const bool is_compute = warp < G;
    if (is_producer) {
        // ======================================= producer =======================================
        const bool aligned16 = (reinterpret_cast<uintptr_t>(signal) & 15) == 0;
        const u32 w0_last = group_xs[G - 1];
        if (lane == 0) {
            fence_proxy_async();
            const u32 total = G * tp.group_stride * 4;
            mbar_expect_tx(bar_taps, total);
            for (u32 done = 0; done < total; done += 32768u)
                tma_bulk_g2s(reinterpret_cast<unsigned char *>(s_taps) + done,
                             reinterpret_cast<const unsigned char *>(tile_taps) + done, min(total - done, 32768u), bar_taps);
        }
        u32 n = 0;
        for (u64 tile = tile_begin + blockIdx.x; tile < ntiles; tile += gridDim.x, ++n) {
            const u32 st = n & 1;
            float *rows = s_stage0 + st * tp.stage_floats;
            float *vrow = rows + tp.rows_floats;
            const u64 x_base = tile * static_cast<u64>(QT) * tp.p_in;       // first input sample of row 0
            const u64 x_end = x_base + static_cast<u64>(QT - 1) * tp.p_in + tp.row_len;
            const bool want_halo = ENVELOPE && tile > 0;
            const u64 x_halo = x_base - tp.p_in + w0_last;                   // meaningful only when tile > 0
            mbar_wait(empty_rows + st, ((n >> 1) & 1) ^ 1);                 // stage free (first use passes)
            if (aligned16) {
                // One bulk copy per row pair (rows 2i, 2i+1 overlap in the signal).  The part of a pair that
                // exists (a multiple of 4 floats) comes by TMA; the rest -- the last <4 samples and everything
                // past the end of the signal, which reads as zero (signal.get(x) == None, dsp.rs:257) -- by this
                // warp's own stores.  Interior tiles are pure TMA.
                const u32 rpc = tp.rows_per_copy, ncopies = QT / rpc;
                const u32 pair_len = (rpc - 1) * tp.p_in + tp.row_len;
                const u64 halo_end = x_halo + tp.usteps;
                const bool edge = x_end > len || (want_halo && halo_end > len);
                auto valid_of = [&](u64 x0, u32 nfl) -> u32 {
                    return x0 >= len ? 0u : static_cast<u32>(min(static_cast<u64>(nfl), len - x0));
                };
                if (edge) {
                    for (u32 i = 0; i < ncopies; ++i) {
                        const u64 xr = x_base + static_cast<u64>(rpc * i) * tp.p_in;
                        const u32 valid = valid_of(xr, pair_len);
                        for (u32 c = (valid & ~3u) + lane; c < pair_len; c += 32)
                            rows[i * tp.pair_pitch + c] = c < valid ? __ldg(signal + xr + c) : 0.f;
                    }
                    if (want_halo) {
                        const u32 valid = valid_of(x_halo, tp.usteps);
                        for (u32 c = (valid & ~3u) + lane; c < tp.usteps; c += 32)
                            vrow[c] = c < valid ? __ldg(signal + x_halo + c) : 0.f;
                    }
                    __syncwarp();                 // the warp's stores are ordered before lane 0's release-arrive
                }
                if (lane == 0) {
                    fence_proxy_async();          // the stage was last read through the generic proxy
                    if (!edge) {
                        mbar_expect_tx(full_rows + st, (ncopies * pair_len + (want_halo ? tp.usteps : 0)) * 4);
                        for (u32 i = 0; i < ncopies; ++i)
                            tma_bulk_g2s(rows + i * tp.pair_pitch, signal + x_base + static_cast<u64>(rpc * i) * tp.p_in,
                                         pair_len * 4, full_rows + st);
                        if (want_halo) tma_bulk_g2s(vrow, signal + x_halo, tp.usteps * 4, full_rows + st);
                    } else {
                        u32 tx_floats = want_halo ? (valid_of(x_halo, tp.usteps) & ~3u) : 0u;
                        for (u32 i = 0; i < ncopies; ++i)
                            tx_floats += valid_of(x_base + static_cast<u64>(rpc * i) * tp.p_in, pair_len) & ~3u;
                        mbar_expect_tx(full_rows + st, tx_floats * 4);
                        for (u32 i = 0; i < ncopies; ++i) {
                            const u64 xr = x_base + static_cast<u64>(rpc * i) * tp.p_in;
                            const u32 nfl = valid_of(xr, pair_len) & ~3u;
                            if (nfl) tma_bulk_g2s(rows + i * tp.pair_pitch, signal + xr, nfl * 4, full_rows + st);
                        }
                        if (want_halo) {
                            const u32 nfl = valid_of(x_halo, tp.usteps) & ~3u;
                            if (nfl) tma_bulk_g2s(vrow, signal + x_halo, nfl * 4, full_rows + st);
                        }
                    }
                }
            } else {
                // unaligned signal pointer: the warp fills the whole stage itself (slow, correct)
                const u32 rpc = tp.rows_per_copy;
                const u32 pair_len = (rpc - 1) * tp.p_in + tp.row_len;
                for (u32 i = 0; i < QT / rpc; ++i)
                    for (u32 c = lane; c < pair_len; c += 32) {
                        const u64 x = x_base + static_cast<u64>(rpc * i) * tp.p_in + c;
                        rows[i * tp.pair_pitch + c] = x < len ? __ldg(signal + x) : 0.f;
                    }
                if (want_halo)
                    for (u32 i = lane; i < tp.usteps; i += 32) vrow[i] = x_halo + i < len ? __ldg(signal + x_halo + i) : 0.f;
                __syncwarp();
                if (lane == 0) mbar_arrive(full_rows + st);
            }
        }
    } else if (is_compute) {
        // ======================================= compute ========================================
        const u32 ks = lane >> 3, ql = lane & 7;
        const u32 w0 = group_xs[warp];
        const u32 it_a_end = tp.half_taps / 16;       // half A is active for iterations [0, it_a_end)
        const u32 it_b_begin = tp.halves == 2 ? tp.shift / 16 : tp.iters;   // half B for [it_b_begin, iters)
        const u32 rec_bytes = tp.halves * 64;         // one (iteration, slice lane) tap record
        const u32 R = 4 * tp.halves;
        const u32 tap_base = smem_u32(s_taps) + (warp * tp.group_stride + ks * tp.slice_stride) * 4;
        // row r lives at pair r/2, half r%2; this thread reads rows ql, ql+8, ql+16, ql+24
        const u32 row_off = (tp.rows_per_copy == 2 ? (ql >> 1) * tp.pair_pitch + (ql & 1) * tp.p_in : ql * tp.pair_pitch) * 4 +
                            (w0 + ks * 4) * 4;
        const u32 row_step8 = (8 / tp.rows_per_copy) * tp.pair_pitch * 4;
        const u32 plane_floats = QT * tp.plane_pitch;
        float *plane_dst = s_planes + ks * plane_floats + ql * tp.plane_pitch + warp * R;
        mbar_wait(bar_taps, 0);
        u32 n = 0;
        for (u64 tile = tile_begin + blockIdx.x; tile < ntiles; tile += gridDim.x, ++n) {
            const u32 st = n & 1;
            const float *rows = s_stage0 + st * tp.stage_floats;
            mbar_wait(full_rows + st, (n >> 1) & 1);
            f32x2 acc_a[2][Q], acc_b[2][Q];
#pragma unroll
            for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int j = 0; j < Q; ++j) acc_a[p][j] = acc_b[p][j] = 0ull;
            u32 tap_addr = tap_base;
            u32 row_addr = smem_u32(rows) + row_off;
            u32 it = 0;
            for (; it < it_b_begin; ++it) {                            // half A only
                float4 s[Q];
#pragma unroll
                for (int j = 0; j < Q; ++j) s[j] = lds128(row_addr + j * row_step8);
                half_fma2(acc_a, tap_addr, s);
                row_addr += KS * 16;
                tap_addr += rec_bytes;
            }
            for (; it < it_a_end; ++it) {                              // both halves
                float4 s[Q];
#pragma unroll
                for (int j = 0; j < Q; ++j) s[j] = lds128(row_addr + j * row_step8);
                half_fma2(acc_a, tap_addr, s);
                half_fma2(acc_b, tap_addr + 64, s);
                row_addr += KS * 16;
                tap_addr += rec_bytes;
            }
            for (; it < tp.iters; ++it) {                              // half B only
                float4 s[Q];
#pragma unroll
                for (int j = 0; j < Q; ++j) s[j] = lds128(row_addr + j * row_step8);
                half_fma2(acc_b, tap_addr + 64, s);
                row_addr += KS * 16;
                tap_addr += rec_bytes;
            }
            // r[K0 - 1]: the last output of the last group, applied to the halo row
            float halo = 0.f;
            if (ENVELOPE && warp == G - 1 && tile > 0) {
                const float *vrow = rows + tp.rows_floats;
                const float *tg = s_taps + static_cast<size_t>(G - 1) * tp.group_stride;
                // the group's last output: r = 3 of half B (two halves) or of half A (one)
                const u32 rec = 16 * tp.halves, off = tp.halves == 2 ? 16 + 3 : 3;
                const u32 ubeg = tp.halves == 2 ? tp.shift : 0, uend = tp.halves == 2 ? tp.usteps : tp.half_taps;
                for (u32 u = ubeg + lane; u < uend; u += 32) {
                    const u32 chunk = u >> 2, uu = u & 3;            // chunk = it*KS + ks
                    halo = fmaf(tg[(chunk & 3) * tp.slice_stride + (chunk >> 2) * rec + off + uu * 4], vrow[u], halo);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) halo += __shfl_xor_sync(0xffffffffu, halo, o);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty_rows + st);           // this warp is done with the stage
            // hand the partial sums to the epilogue warps
            mbar_wait(empty_p, (n & 1) ^ 1);
#pragma unroll
            for (int j = 0; j < Q; ++j) {
                float4 va, vb;
                unpack2(acc_a[0][j], va.x, va.y);
                unpack2(acc_a[1][j], va.z, va.w);
                unpack2(acc_b[0][j], vb.x, vb.y);
                unpack2(acc_b[1][j], vb.z, vb.w);
                float *dst = plane_dst + 8 * j * tp.plane_pitch;
                *reinterpret_cast<float4 *>(dst) = va;
                if (tp.halves == 2) *reinterpret_cast<float4 *>(dst + 4) = vb;
            }
            if (ENVELOPE && warp == G - 1 && lane == 0) *s_halo = halo;
            __syncwarp();
            if (lane == 0) mbar_arrive(full_p);
        }
    } else {
        // ======================================= epilogue =======================================
        const u32 e = warp - G - (warp > prod_warp ? 1 : 0);   // epilogue warps: every remaining warp, in order
        const u32 vec_per_row = tp.p_out / 4;
        const u32 nvec = QT * vec_per_row;
        const u32 plane_floats = QT * tp.plane_pitch;
        const float inv_sinphi = 1.f / sinphi;
        const bool out_aligned = (reinterpret_cast<uintptr_t>(out) & 15) == 0;
        u32 n = 0;
        for (u64 tile = tile_begin + blockIdx.x; tile < ntiles; tile += gridDim.x, ++n) {
            const u64 k_base = tile * tile_out;
            const bool full_tile = k_base + tile_out <= nout && out_aligned;
            float *out_tile = out + k_base;
            mbar_wait(full_p, n & 1);
            // two cells per lane and pass (independent chains -> ILP); cells are 4 consecutive outputs
            for (u32 v0 = e * 32 + lane; v0 < nvec; v0 += 2 * E * 32) {
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const u32 v = v0 + half * E * 32;
                    if (v >= nvec) break;
                    const u32 q = (v * tp.vec_magic) >> 16, c4 = v - q * vec_per_row;   // v / vec_per_row
                    const u32 kl = q * tp.p_out + 4 * c4;                    // output index inside the tile
                    const float *cell = s_planes + q * tp.plane_pitch + 4 * c4;
                    const float4 a = *reinterpret_cast<const float4 *>(cell);
                    const float4 b = *reinterpret_cast<const float4 *>(cell + plane_floats);
                    const float4 c = *reinterpret_cast<const float4 *>(cell + 2 * plane_floats);
                    const float4 d = *reinterpret_cast<const float4 *>(cell + 3 * plane_floats);
                    const float4 cur = make_float4((a.x + b.x) + (c.x + d.x), (a.y + b.y) + (c.y + d.y),
                                                   (a.z + b.z) + (c.z + d.z), (a.w + b.w) + (c.w + d.w));
                    float4 res = cur;
                    if (ENVELOPE) {
                        // previous output: left neighbour, last output of the previous row, or the halo for kl == 0
                        const float *pc = kl == 0 ? cell : c4 > 0 ? cell - 1 : cell - (tp.plane_pitch - tp.p_out) - 1;
                        float prev = (pc[0] + pc[plane_floats]) + (pc[2 * plane_floats] + pc[3 * plane_floats]);
                        if (kl == 0) prev = *s_halo;
                        res.x = envelope2_fast(prev, cur.x, cosphi2, inv_sinphi);
                        res.y = envelope2_fast(cur.x, cur.y, cosphi2, inv_sinphi);
                        res.z = envelope2_fast(cur.y, cur.z, cosphi2, inv_sinphi);
                        res.w = envelope2_fast(cur.z, cur.w, cosphi2, inv_sinphi);
                        if (kl == 0 && k_base == 0) res.x = 0.f;             // output[0] = 0 (dsp.rs:357)
                    }
                    if (full_tile) {
                        *reinterpret_cast<float4 *>(out_tile + kl) = res;
                    } else {
                        const u64 k = k_base + kl;
                        if (k < nout) out[k] = res.x;
                        if (k + 1 < nout) out[k + 1] = res.y;
                        if (k + 2 < nout) out[k + 2] = res.z;
                        if (k + 3 < nout) out[k + 3] = res.w;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty_p);
        }
    }
}

}  // namespace aptb200
