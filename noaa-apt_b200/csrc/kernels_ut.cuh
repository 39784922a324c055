// Polyphase resampler + envelope with the taps in the CONSTANT BANK (kernel parameter), read through the
// uniform datapath -- the hot kernel of the path for L = 13 (48/96/192 kHz -> 12 480 Hz).
// fast_resampling dsp.rs:186-289 + demodulate dsp.rs:350-383.
//
// Formulation.  Output k = L*q + r ("row" q, phase r < L) is
//     y[L*q + r] = sum_u h[u*L - r*M] * X[q*M + u]
// i.e. every row uses the SAME L tap sets T[u][r] = h[u*L - r*M] on a window that moves by M samples per row.
// A thread owns Q rows x the output PAIRS (2p, 2p+1) of its role (one packed fp32x2 accumulator per pair and row);
// the 32 lanes of a warp are 32 consecutive rows.  The tap pair (T[u][2p], T[u][2p+1]) is therefore warp-uniform:
// it is read with LDCU from the kernel-parameter constant bank into uniform registers and used directly as the
// packed operand of FFMA2 (`FFMA2 R, R.F32, UR.F32x2, R`); the only shared-memory traffic is the thread's own
// samples (one chunk of CH = 8 samples per row per loop iteration).  In isolation the form reaches 104-107 FMA/clk/SM,
// the FFMA2 pipe limit, against 70-84 for shared-memory tap operands (profiles/r01_microbench_uniform_taps.txt).
//
// Zero padding.  Pair p only sees samples fx(2p) .. lx(2p+1); the loop over 8-sample chunks is cut into
// segments with a fixed set of active pairs: ramp-up (pairs 0..a-1 for a = 1..NP-1), steady (all), ramp-down
// (pairs a..NP-1).  The tap stream in the parameter block is stored in exactly the order the loop consumes it.
//
// Pipeline.  One persistent CTA per SM owns a contiguous range of blocks (block = 32*Q rows = 32*Q*L outputs,
// whose input is ONE contiguous span of the signal: no duplication in shared memory).  A producer warp streams
// blocks into a ring of NSLOT shared-memory slots with one cp.async.bulk (TMA) per block, completion on a
// `full` mbarrier.  TWO compute warps share a block: role 0 owns the first half of the output pairs, role 1 the
// rest; warps draw (block, role) tickets from a shared-memory counter, so nothing couples the warps CTA-wide.
// After its FMA loop a warp publishes the one output its partner's envelope needs (role boundary / row boundary)
// in the words behind the slot, the pair meets on the `xch` mbarrier (nobody reads the samples any more), both
// compute their envelopes (dsp.rs:373), transpose them through the dead slot, meet on `staged`, store half of the
// block each as coalesced float4, and release the slot through the `empty` mbarrier (count 2).  r[k0-1] for the
// first output of a block is a dot product of role 1 split over its lanes (taps of output L-1 staged in shared memory).
#pragma once


#include <cstdint>
#include <utility>
#include <cuda_runtime.h>

#include "kernels_fast.cuh"
#include "launch.hpp"

namespace aptb200 {

constexpr int kUtMaxPairs = 8;

// Kernel-parameter block: everything in it is warp-uniform.  MAXV float4 = the tap stream.
template <int MAXV>
struct UtParams {
    float4 v[MAXV];
    u32 cs[kUtMaxPairs];      // first chunk of pair p
    u32 ce[kUtMaxPairs];      // one past its last chunk
};

struct UtGeom {
    u32 l, m;
    u32 back;                 // samples staged in front of the block's first row (halo window), multiple of 4
    u32 slot_floats;          // back + (rows-1)*m + 4*chunks, multiple of 4
    u32 nslot, warps;         // ring slots, compute warps
    u32 halo_u0, halo_n;      // output L-1: first sample (relative to its row) and number of taps
    u32 header_bytes;         // barriers + halo taps, multiple of 128
    u32 slot_stride;          // floats between slots: slot_floats + the 2*rows+4 exchange words behind each slot
    u32 stream_b;             // float4 index where the second role's tap stream starts
};

constexpr int CH = static_cast<int>(kUtChunk);   // samples per chunk (one loop iteration)

// the CH samples of one chunk of one row, with the widest load the row alignment allows
template <int VEC>
__device__ __forceinline__ void ut_load_chunk(const float *p, float (&s)[CH]) {
#pragma unroll
    for (int i = 0; i < CH; i += 4) {
        if (VEC == 4) {
            const float4 v = *reinterpret_cast<const float4 *>(p + i);
            s[i] = v.x; s[i + 1] = v.y; s[i + 2] = v.z; s[i + 3] = v.w;
        } else if (VEC == 2) {
            const float2 a = *reinterpret_cast<const float2 *>(p + i), b = *reinterpret_cast<const float2 *>(p + i + 2);
            s[i] = a.x; s[i + 1] = a.y; s[i + 2] = b.x; s[i + 3] = b.y;
        } else {
            s[i] = p[i]; s[i + 1] = p[i + 1]; s[i + 2] = p[i + 2]; s[i + 3] = p[i + 3];
        }
    }
}

// Chunks [cb, ce) with pairs [P0, P1) of a role active.  toff: running float4 index into the tap stream (uniform);
// per (chunk, pair) the stream holds CH/2 float4 = the tap pairs of the chunk's CH samples.
template <int P0, int P1, int NPR, int Q, int VEC, int MAXV>
__device__ __forceinline__ void ut_segment(const UtParams<MAXV> &prm, u32 cb, u32 ce, int &toff, const float *row0,
                                           u32 qstride, f32x2 (&acc)[Q][NPR]) {
#pragma unroll 1   // unrolled x2 the kernel is slower (code size, DESIGN.md §3.1)
    for (u32 c = cb; c < ce; ++c) {
        float s[Q][CH];
#pragma unroll
        for (int q = 0; q < Q; ++q) ut_load_chunk<VEC>(row0 + q * qstride + CH * c, s[q]);
#pragma unroll
        for (int p = P0; p < P1; ++p) {
#pragma unroll
            for (int i = 0; i < CH / 2; ++i) {
                const float4 t = prm.v[toff + (CH / 2) * (p - P0) + i];
                const f32x2 t0 = pack2(t.x, t.y), t1 = pack2(t.z, t.w);
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    acc[q][p] = fma2(t0, pack2(s[q][2 * i], s[q][2 * i]), acc[q][p]);
                    acc[q][p] = fma2(t1, pack2(s[q][2 * i + 1], s[q][2 * i + 1]), acc[q][p]);
                }
            }
        }
        toff += (CH / 2) * (P1 - P0);
    }
}

// One role = a contiguous range of pairs [PB, PB + NPR) of the row's outputs; its loop over chunks is cut into
// ramp-up (pairs PB..PB+a-1 active), steady (all) and ramp-down (pairs PB+a.. active) segments.
template <int PB, int NPR, int Q, int VEC, int MAXV, int... A>
__device__ __forceinline__ void ut_ramp_up(const UtParams<MAXV> &prm, int &toff, const float *row0, u32 qstride,
                                           f32x2 (&acc)[Q][NPR], std::integer_sequence<int, A...>) {
    (ut_segment<0, A + 1, NPR, Q, VEC, MAXV>(prm, prm.cs[PB + A], prm.cs[PB + A + 1], toff, row0, qstride, acc), ...);
}
template <int PB, int NPR, int Q, int VEC, int MAXV, int... A>
__device__ __forceinline__ void ut_ramp_down(const UtParams<MAXV> &prm, int &toff, const float *row0, u32 qstride,
                                             f32x2 (&acc)[Q][NPR], std::integer_sequence<int, A...>) {
    (ut_segment<A + 1, NPR, NPR, Q, VEC, MAXV>(prm, prm.ce[PB + A], prm.ce[PB + A + 1], toff, row0, qstride, acc), ...);
}

// Everything one warp does for one (block, role): FMA loop over the role's pairs, exchange of the boundary
// outputs with the partner warp, envelope, staging, its half of the coalesced stores.
template <int L, int PB, int NPR, bool LAST, int Q, int VEC, int MAXV, bool ENVELOPE>
__device__ __forceinline__ void ut_role(const UtParams<MAXV> &prm, const UtGeom &g, int toff, float *slot, u64 *xch_bar,
                                        u64 *staged_bar, u32 parity, u32 role, const float *halo_taps, u64 k0, u64 nout,
                                        float cosphi2, float inv_sinphi, float *__restrict__ out, u32 lane) {
    constexpr u32 RB = 32 * Q;
    constexpr int JB = 2 * PB;                                       // first output (phase) of this role
    constexpr int JN = (2 * NPR < L - JB) ? 2 * NPR : L - JB;        // number of real outputs
    const u32 m = g.m, qstride = 32 * m;
    f32x2 acc[Q][NPR];
#pragma unroll
    for (int q = 0; q < Q; ++q)
#pragma unroll
        for (int p = 0; p < NPR; ++p) acc[q][p] = 0ull;
    const float *row0 = slot + g.back + lane * m;
    ut_ramp_up<PB, NPR, Q, VEC, MAXV>(prm, toff, row0, qstride, acc, std::make_integer_sequence<int, NPR - 1>{});
    ut_segment<0, NPR, NPR, Q, VEC, MAXV>(prm, prm.cs[PB + NPR - 1], prm.ce[PB], toff, row0, qstride, acc);
    ut_ramp_down<PB, NPR, Q, VEC, MAXV>(prm, toff, row0, qstride, acc, std::make_integer_sequence<int, NPR - 1>{});
    // boundary outputs, exchanged through the words behind the slot's samples:
    //   xa[row]     = output JN-1 of the first role (needed by the second role's first output)
    //   xb[row + 1] = output L-1 of the row (needed by the next row's output 0); xb[0] = r[k0-1] (halo)
    float *xa = slot + g.slot_floats, *xb = xa + RB;
    if (ENVELOPE) {
        if (LAST) {
            // r[k0 - 1]: output L-1 of the row in front of the block, k-split over the lanes
            float halo = 0.f;
            if (k0 > 0) {
                const float *hw = slot + g.back - m;                   // that row's sample u sits at hw[u]
                for (u32 i = lane; i < g.halo_n; i += 32) halo = fmaf(halo_taps[i], hw[g.halo_u0 + i], halo);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) halo += __shfl_xor_sync(0xffffffffu, halo, o);
            }
            if (lane == 0) xb[0] = halo;
        }
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            float lo, hi;
            unpack2(acc[q][(JN - 1) / 2], lo, hi);
            const float last = (JN - 1) % 2 ? hi : lo;
            if (LAST) xb[q * 32 + lane + 1] = last;
            else xa[q * 32 + lane] = last;
        }
    }
    // both warps are past the FMA loop (nobody reads the samples any more) and have published
    __syncwarp();
    if (lane == 0) mbar_arrive(xch_bar);
    mbar_wait(xch_bar, parity);
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        float r[2 * NPR];
#pragma unroll
        for (int p = 0; p < NPR; ++p) unpack2(acc[q][p], r[2 * p], r[2 * p + 1]);
        const u32 row = q * 32 + lane;
        float *dst = slot + row * L + JB;
        if (ENVELOPE) {
            float prev = LAST ? xa[row] : xb[row];
#pragma unroll
            for (int j = 0; j < JN; ++j) {
                dst[j] = envelope2_fast(prev, r[j], cosphi2, inv_sinphi);
                prev = r[j];
            }
        } else {
#pragma unroll
            for (int j = 0; j < JN; ++j) dst[j] = r[j];
        }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(staged_bar);
    mbar_wait(staged_bar, parity);
    constexpr u32 nvec = RB * L / 4;                                   // RB*L is a multiple of 4
#pragma unroll
    for (u32 vi = 0; vi < (nvec + 63) / 64; ++vi) {
        const u32 v = lane + 32 * (2 * vi + role);
        const u64 k = k0 + 4 * v;
        if (v >= nvec || k >= nout) break;
        float4 val = *reinterpret_cast<const float4 *>(slot + 4 * v);
        if (ENVELOPE && k == 0) val.x = 0.f;                           // dsp.rs:364: the first sample has no predecessor
        if (k + 3 < nout) {
            *reinterpret_cast<float4 *>(out + k) = val;
        } else {
            out[k] = val.x;
            if (k + 1 < nout) out[k + 1] = val.y;
            if (k + 2 < nout) out[k + 2] = val.z;
        }
    }
}

template <int L, int Q, int VEC, int MAXV, bool ENVELOPE>
__global__ void __launch_bounds__(800, 1)
k_polyphase_ut(const __grid_constant__ UtParams<MAXV> prm, const float *__restrict__ signal, u64 len,
               const float *__restrict__ h, const UtGeom g, u64 nout, u64 blk_begin, u64 blk_end, float cosphi2,
               float inv_sinphi, float *__restrict__ out) {
    extern __shared__ __align__(128) unsigned char ut_smem[];
    u64 *full = reinterpret_cast<u64 *>(ut_smem);                 // [kUtMaxSlots] samples landed
    u64 *empty = full + kUtMaxSlots;                               // slot may be refilled (both warps done)
    u64 *xch = empty + kUtMaxSlots;                                // both warps past the FMA loop, boundary outputs published
    u64 *staged = xch + kUtMaxSlots;                               // both warps have staged their outputs
    u32 *ticket = reinterpret_cast<u32 *>(staged + kUtMaxSlots);   // next (block, role) sequence number
    float *halo_taps = reinterpret_cast<float *>(ut_smem + 1024);  // [halo_n] taps of output L-1 (for r[k0-1])
    float *slots = reinterpret_cast<float *>(ut_smem + g.header_bytes);

    constexpr u32 RB = 32 * Q;                                     // rows per block
    constexpr int NP = (L + 1) / 2;                                // pairs of outputs per row
    constexpr int NPA = (NP + 1) / 2, NPB = NP - NPA;              // role 0: pairs [0, NPA), role 1: [NPA, NP)
    const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const u32 m = g.m;
    // this CTA's contiguous range of blocks
    const u64 nb_all = blk_end - blk_begin;
    const u64 b0 = blk_begin + nb_all * blockIdx.x / gridDim.x;
    const u64 b1 = blk_begin + nb_all * (blockIdx.x + 1) / gridDim.x;
    const u32 nblk = static_cast<u32>(b1 - b0);

    if (threadIdx.x == 0) {
        for (u32 s = 0; s < g.nslot; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, 2);
            mbar_init(xch + s, 2);
            mbar_init(staged + s, 2);
        }
        *ticket = 0;
        fence_mbar_init();
    }
    if (ENVELOPE)
        for (u32 i = threadIdx.x; i < g.halo_n; i += blockDim.x)
            halo_taps[i] = __ldg(h + ((g.halo_u0 + i) * L - (L - 1) * g.m));
    __syncthreads();

    if (warp == g.warps) {
        // ===== producer warp =====
        for (u32 n = 0; n < nblk; ++n) {
            const u32 s = n % g.nslot;
            if (n >= g.nslot) mbar_wait(empty + s, ((n / g.nslot) - 1) & 1);
            float *dst = slots + static_cast<size_t>(s) * g.slot_stride;
            const long long x_lo = static_cast<long long>((b0 + n) * RB * m) - g.back;   // sample staged at dst[0]
            const long long x_hi = x_lo + g.slot_floats;
            if (x_lo >= 0 && static_cast<u64>(x_hi) <= len) {
                if (lane == 0) {
                    mbar_expect_tx(full + s, g.slot_floats * 4);
                    tma_bulk_g2s(dst, signal + x_lo, g.slot_floats * 4, full + s);
                }
            } else {
                // first / last blocks: bulk-copy the part that exists (16-byte granules), fill the rest
                const long long va = x_lo < 0 ? 0 : x_lo;                                 // x_lo is a multiple of 4
                long long vb = static_cast<long long>(len) < x_hi ? static_cast<long long>(len) : x_hi;
                if (vb < va) vb = va;
                const long long vb4 = va + ((vb - va) & ~3ll);
                for (long long x = x_lo + lane; x < x_hi; x += 32)
                    if (x < va || x >= vb4) dst[x - x_lo] = (x >= va && x < vb) ? __ldg(signal + x) : 0.f;
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    const u32 bytes = static_cast<u32>(vb4 - va) * 4;
                    if (bytes) {
                        mbar_expect_tx(full + s, bytes);
                        tma_bulk_g2s(dst + (va - x_lo), signal + va, bytes, full + s);
                    } else {
                        mbar_arrive(full + s);
                    }
                }
            }
        }
        return;
    }
    if (warp > g.warps) return;

    // ===== compute warps: tickets are (block, role) pairs; two warps share a block =====
    for (;;) {
        u32 t = 0;
        if (lane == 0) t = atomicAdd(ticket, 1u);
        t = __shfl_sync(0xffffffffu, t, 0);
        const u32 n = t >> 1, role = t & 1;
        if (n >= nblk) break;
        const u32 s = n % g.nslot, parity = (n / g.nslot) & 1;
        float *slot = slots + static_cast<size_t>(s) * g.slot_stride;
        mbar_wait(full + s, parity);
        const u64 k0 = (b0 + n) * RB * L;                          // first output of the block
        if (role == 0)
            ut_role<L, 0, NPA, false, Q, VEC, MAXV, ENVELOPE>(prm, g, 0, slot, xch + s, staged + s, parity, role, halo_taps, k0, nout,
                                                              cosphi2, inv_sinphi, out, lane);
        else
            ut_role<L, NPA, NPB, true, Q, VEC, MAXV, ENVELOPE>(prm, g, static_cast<int>(g.stream_b), slot, xch + s, staged + s, parity,
                                                               role, halo_taps, k0, nout, cosphi2, inv_sinphi, out, lane);
        fence_proxy_async();                                       // generic writes before the next bulk copy into the slot
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + s);
    }
}

}  // namespace aptb200
