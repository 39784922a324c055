// Kernel launchers: the only translation unit that instantiates the kernels.
#include "launch.hpp"

#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>

#include "aptb200.h"
#include "common.hpp"
#include "kernels_fast.cuh"
#include "kernels_generic.cuh"
#include "kernels_lpsync.cuh"
#include "kernels_ph.cuh"
#include "kernels_sync.cuh"
#include "kernels_sync2.cuh"
#include "kernels_post.cuh"
#include "kernels_ut.cuh"

namespace aptb200 {

namespace {

inline unsigned grid_for(u64 n, unsigned per_block, int sms) {
    const u64 blocks = (n + per_block - 1) / per_block;
    const u64 cap = static_cast<u64>(sms) * 16;
    return static_cast<unsigned>(std::max<u64>(1, std::min(blocks, cap)));
}

template <int CHUNK, int THREADS = 512>
int roots_with_chunk(const LaunchCtx &c, const float *corr, u64 ncorr, u32 dist, u32 nblocks, u32 *root_list,
                     u32 *root_count, SyncResult *result, const PickScratch *sc) {
    const size_t smem = 2ull * dist * sizeof(float);
    auto kern = k_roots<THREADS, CHUNK>;
    APT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kern<<<nblocks, THREADS, smem, c.stream>>>(corr, ncorr, dist, root_list, root_count, result,
                                            sc ? sc->block_off : nullptr, sc ? sc->ticket : nullptr);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

}  // namespace

int launch_polyphase(const LaunchCtx &c, const void *signal, int format, u64 len, const float *taps, u32 l, u32 m,
                     u64 off2, u64 k_begin, u64 nout, bool envelope, float cosphi2, float sinphi, float *out) {
    if (nout <= k_begin) return APT_OK;
    const unsigned grid = grid_for(nout - k_begin, 256, c.sm_count);
    if (format == APT_PCM16) {
        const int16_t *s = static_cast<const int16_t *>(signal);
        if (envelope) k_polyphase_generic<int16_t, true><<<grid, 256, 0, c.stream>>>(s, len, taps, l, m, off2, k_begin, nout, cosphi2, sinphi, out);
        else k_polyphase_generic<int16_t, false><<<grid, 256, 0, c.stream>>>(s, len, taps, l, m, off2, k_begin, nout, cosphi2, sinphi, out);
    } else {
        const float *s = static_cast<const float *>(signal);
        if (envelope) k_polyphase_generic<float, true><<<grid, 256, 0, c.stream>>>(s, len, taps, l, m, off2, k_begin, nout, cosphi2, sinphi, out);
        else k_polyphase_generic<float, false><<<grid, 256, 0, c.stream>>>(s, len, taps, l, m, off2, k_begin, nout, cosphi2, sinphi, out);
    }
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_polyphase_tiled(const LaunchCtx &c, const float *signal, u64 len, const float *tile_taps,
                           const u32 *group_xs, const TilePlan &tp, u64 nout, u64 tile_begin, u64 tile_end,
                           bool envelope, float cosphi2, float sinphi, float *out) {
    if (nout == 0) return APT_OK;
    const u64 tile_out = static_cast<u64>(tp.qt) * tp.p_out;
    u64 ntiles = (nout + tile_out - 1) / tile_out;
    if (tile_end != 0) ntiles = std::min(ntiles, tile_end);
    if (tile_begin >= ntiles) return APT_OK;
    const unsigned grid = static_cast<unsigned>(std::min<u64>(ntiles - tile_begin, static_cast<u64>(c.sm_count)));
    const unsigned block = 32 * (tp.groups + kWsEpilogueWarps + 1);   // compute + epilogue + producer warps
    if (envelope) {
        auto kern = k_polyphase_ws<true>;
        APT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tp.smem_bytes)));
        kern<<<grid, block, tp.smem_bytes, c.stream>>>(signal, len, tile_taps, group_xs, tp, nout, tile_begin, ntiles,
                                                        cosphi2, sinphi, out);
    } else {
        auto kern = k_polyphase_ws<false>;
        APT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tp.smem_bytes)));
        kern<<<grid, block, tp.smem_bytes, c.stream>>>(signal, len, tile_taps, group_xs, tp, nout, tile_begin, ntiles,
                                                        cosphi2, sinphi, out);
    }
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

namespace {
template <int Q, int VEC, int MAXV, bool ENV>
int launch_ut_inst(const LaunchCtx &c, const float *signal, u64 len, const float *h, const UtPlan &up,
                   const std::vector<float> &stream, u64 nout, u64 blk_begin, u64 blk_end, float cosphi2, float sinphi,
                   float *out) {
    static thread_local UtParams<MAXV> prm;                      // 6 / 30 KB: rebuilt per launch, passed by value
    memset(&prm, 0, sizeof(prm));
    memcpy(prm.v, stream.data(), stream.size() * sizeof(float));
    for (int p = 0; p < 8; ++p) {
        prm.cs[p] = up.cs[p];
        prm.ce[p] = up.ce[p];
    }
    const UtGeom g{up.l, up.m, up.back, up.slot_floats, up.nslot, up.warps, up.halo_u0, up.halo_n, up.header_bytes, up.slot_stride, up.stream_b};
    auto kern = k_polyphase_ut<static_cast<int>(kUtL), Q, VEC, MAXV, ENV>;
    APT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(up.smem_bytes)));
    const unsigned grid = static_cast<unsigned>(std::min<u64>(blk_end - blk_begin, static_cast<u64>(c.sm_count)));
    kern<<<grid, 32 * (up.warps + 1), up.smem_bytes, c.stream>>>(prm, signal, len, h, g, nout, blk_begin, blk_end, cosphi2,
                                                                 1.0f / sinphi, out);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}
template <int Q, int VEC, bool ENV>
int launch_ut_size(const LaunchCtx &c, const float *signal, u64 len, const float *h, const UtPlan &up,
                   const std::vector<float> &stream, u64 nout, u64 b0, u64 b1, float cosphi2, float sinphi, float *out) {
    if (up.nvec <= kUtMaxVecSmall)
        return launch_ut_inst<Q, VEC, static_cast<int>(kUtMaxVecSmall), ENV>(c, signal, len, h, up, stream, nout, b0, b1, cosphi2, sinphi, out);
    return launch_ut_inst<Q, VEC, static_cast<int>(kUtMaxVecLarge), ENV>(c, signal, len, h, up, stream, nout, b0, b1, cosphi2, sinphi, out);
}
template <int Q, bool ENV>
int launch_ut_vec(const LaunchCtx &c, const float *signal, u64 len, const float *h, const UtPlan &up,
                  const std::vector<float> &stream, u64 nout, u64 b0, u64 b1, float cosphi2, float sinphi, float *out) {
    switch (up.vec) {
    case 4: return launch_ut_size<Q, 4, ENV>(c, signal, len, h, up, stream, nout, b0, b1, cosphi2, sinphi, out);
    case 2: return launch_ut_size<Q, 2, ENV>(c, signal, len, h, up, stream, nout, b0, b1, cosphi2, sinphi, out);
    default: return launch_ut_size<Q, 1, ENV>(c, signal, len, h, up, stream, nout, b0, b1, cosphi2, sinphi, out);
    }
}
}  // namespace

int launch_polyphase_ut(const LaunchCtx &c, const float *signal, u64 len, const float *h, const UtPlan &up,
                        const std::vector<float> &stream, u64 nout, u64 blk_begin, u64 blk_end, bool envelope,
                        float cosphi2, float sinphi, float *out) {
    if (nout == 0) return APT_OK;
    const u64 blk_out = static_cast<u64>(up.rb) * up.l;
    u64 nblk = (nout + blk_out - 1) / blk_out;
    if (blk_end != 0) nblk = std::min(nblk, blk_end);
    if (blk_begin >= nblk) return APT_OK;
    if ((reinterpret_cast<uintptr_t>(signal) & 15) || (reinterpret_cast<uintptr_t>(out) & 15) || stream.size() != 4ull * up.nvec)
        return fail(APT_ERR_BAD_ARG, "uniform-tap resampler: misaligned buffers or inconsistent plan");
    if (up.q == 2)
        return envelope ? launch_ut_vec<2, true>(c, signal, len, h, up, stream, nout, blk_begin, nblk, cosphi2, sinphi, out)
                        : launch_ut_vec<2, false>(c, signal, len, h, up, stream, nout, blk_begin, nblk, cosphi2, sinphi, out);
    return envelope ? launch_ut_vec<1, true>(c, signal, len, h, up, stream, nout, blk_begin, nblk, cosphi2, sinphi, out)
                    : launch_ut_vec<1, false>(c, signal, len, h, up, stream, nout, blk_begin, nblk, cosphi2, sinphi, out);
}

int launch_polyphase_ph(const LaunchCtx &c, const void *signal, int format, u64 len, const float *table_dev,
                        const unsigned short *xs_dev, const PhPlan &pp, u64 nout, u64 tile_begin, u64 tile_end, bool envelope,
                        float cosphi2, float sinphi, float *out) {
    if (nout == 0) return APT_OK;
    const u64 tile_out = static_cast<u64>(kPhPeriods) * pp.l;
    u64 ntiles = (nout + tile_out - 1) / tile_out;
    if (tile_end != 0) ntiles = std::min(ntiles, tile_end);
    if (tile_begin >= ntiles) return APT_OK;
    const PhGeom g{pp.l, pp.m, pp.j, pp.pitch, pp.row_len, pp.smem_bytes};
    const unsigned grid = static_cast<unsigned>(std::min<u64>(ntiles - tile_begin, static_cast<u64>(c.sm_count)));
    auto launch = [&](auto kern, auto *sig) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pp.smem_bytes));
        kern<<<grid, 32 * kPhWarps, pp.smem_bytes, c.stream>>>(sig, len, table_dev, xs_dev, g, nout, tile_begin, ntiles, envelope ? 1 : 0,
                                                              cosphi2, 1.0f / sinphi, out);
    };
    const float *sf = static_cast<const float *>(signal);
    const int16_t *si = static_cast<const int16_t *>(signal);
    const bool pcm = format == APT_PCM16;
    switch (pp.jpad) {      // the shared window of a group of four phases
    case 24: if (pcm) launch(k_polyphase_ph<int16_t, 24>, si); else launch(k_polyphase_ph<float, 24>, sf); break;
    case 44: if (pcm) launch(k_polyphase_ph<int16_t, 44>, si); else launch(k_polyphase_ph<float, 44>, sf); break;
    case 84: if (pcm) launch(k_polyphase_ph<int16_t, 84>, si); else launch(k_polyphase_ph<float, 84>, sf); break;
    default: return fail(APT_ERR_BAD_ARG, "phase-major resampler: no instantiation for a window of %u samples", pp.jpad);
    }
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_fir_decimate(const LaunchCtx &c, const void *signal, int format, const float *coeff, u32 ntaps, u32 m,
                        u64 nout, float *out) {
    if (nout == 0) return APT_OK;
    const unsigned grid = grid_for(nout, 256, c.sm_count);
    if (format == APT_PCM16)
        k_fir_decimate_generic<int16_t><<<grid, 256, 0, c.stream>>>(static_cast<const int16_t *>(signal), coeff, ntaps, m, nout, out);
    else
        k_fir_decimate_generic<float><<<grid, 256, 0, c.stream>>>(static_cast<const float *>(signal), coeff, ntaps, m, nout, out);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_pcm16_to_f32(const LaunchCtx &c, const int16_t *in, u64 n, float *out) {
    if (n == 0) return APT_OK;
    k_pcm16_to_f32<<<grid_for(n / 8 + 1, 256, c.sm_count), 256, 0, c.stream>>>(in, n, out);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_envelope(const LaunchCtx &c, const float *x, u64 n, float cosphi2, float sinphi, float *out) {
    if (n == 0) return APT_OK;
    k_envelope<<<grid_for(n, 256, c.sm_count), 256, 0, c.stream>>>(x, n, cosphi2, sinphi, out);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_corr(const LaunchCtx &c, const float *f, u64 ncorr, const int8_t *guard, u32 glen, float *corr) {
    if (ncorr == 0) return APT_OK;
    k_corr_generic<<<grid_for(ncorr, 256, c.sm_count), 256, 0, c.stream>>>(f, ncorr, guard, glen, corr);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

static LpTaps make_lp_taps(const float *taps_host, u32 ntaps, int dec = 0) {
    LpTaps t{};
    auto tap = [&](long long j) { return j >= 0 && j < static_cast<long long>(ntaps) ? taps_host[j] : 0.f; };
    for (int i = 0; i < 32; ++i) {
        t.a_even[i] = make_float2(tap(2 * i), tap(2 * i - 1));
        t.a_odd[i] = make_float2(tap(2 * i + 1), tap(2 * i));
    }
    for (int j = -1; j < 63; ++j) t.p[j + 1] = make_float2(tap(j), tap(j + 1));
    for (int j = -dec; j < 72 - dec; ++j) t.pd[j + dec] = make_float2(tap(j), tap(j + dec));
    return t;
}

bool lowpass_corr_supported(u32 ntaps, u32 pw) {
    return (ntaps == 37 && pw == 3) || (ntaps == 43 && pw == 4) || (ntaps == 61 && pw == 5);
}

int launch_lowpass_corr(const LaunchCtx &c, const float *e, u64 n, const float *taps_host, u32 ntaps, u32 pw, float *f,
                        float *corr) {
    if (n == 0) return APT_OK;
    const LpTaps t = make_lp_taps(taps_host, ntaps);
    const u64 ncorr = n > 38ull * pw ? n - 38ull * pw : 0;
    const u64 ntiles = (n + kLpTile - 1) / kLpTile;
    // persistent: exactly the resident CTAs, each walks its tiles with the next tile's loads in flight
    auto launch = [&](auto kern) {
        static const int per_sm = [&] {          // per instantiation (generic lambda); the same on every B200
            int v = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kern, 256, 0) != cudaSuccess || v < 1) v = 2;
            return v;
        }();
        const unsigned grid = static_cast<unsigned>(std::min<u64>(ntiles, static_cast<u64>(c.sm_count) * per_sm));
        kern<<<grid, 256, 0, c.stream>>>(e, n, ncorr, t, f, corr);
    };
    if (ntaps == 37 && pw == 3) launch(k_lowpass_corr<37, 3>);
    else if (ntaps == 43 && pw == 4) launch(k_lowpass_corr<43, 4>);
    else if (ntaps == 61 && pw == 5) launch(k_lowpass_corr<61, 5>);
    else return fail(APT_ERR_BAD_ARG, "no fused low-pass/correlation kernel for %u taps, pixel width %u", ntaps, pw);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_roots(const LaunchCtx &c, const float *corr, u64 ncorr, u32 dist, u32 *root_list, u32 *root_count,
                 SyncResult *result, const PickScratch *sc) {
    const u32 nblocks = static_cast<u32>((ncorr + dist - 1) / dist);
    const u32 need = (dist + 511) / 512;
    if (need <= 10) return roots_with_chunk<10>(c, corr, ncorr, dist, nblocks, root_list, root_count, result, sc);
    if (need <= 13) return roots_with_chunk<13>(c, corr, ncorr, dist, nblocks, root_list, root_count, result, sc);
    if (need <= 17) return roots_with_chunk<17>(c, corr, ncorr, dist, nblocks, root_list, root_count, result, sc);
    if (need <= 32) return roots_with_chunk<32>(c, corr, ncorr, dist, nblocks, root_list, root_count, result, sc);
    return fail(APT_ERR_BAD_ARG, "work rate too high for the sync picker (min_distance %u)", dist);
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device; cache the outcome per device (0 unknown, 1 ok, -1 refused).
constexpr int kMaxDevices = 64;
template <typename K>
static bool smem_attr_once(std::atomic<signed char> *flags, K kern, size_t smem) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices)
        return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) == cudaSuccess;
    signed char v = flags[dev].load(std::memory_order_acquire);
    if (v == 0) {
        v = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) == cudaSuccess ? 1 : -1;
        if (v < 0) cudaGetLastError();
        flags[dev].store(v, std::memory_order_release);
    }
    return v > 0;
}

int launch_pick(const LaunchCtx &c, u64 ncorr, u64 nwork, u32 row, u32 dist, const RootIndex &ri_in, u32 *positions,
                u32 max_positions, SyncResult *result, const PickScratch *scratch, int *kernels_launched) {
    RootIndex ri = ri_in;
    int dummy = 0;
    int &nk = kernels_launched ? *kernels_launched : dummy;
    nk = 1;
    // Which parallel orbit walk: APTB200_PICK = cluster | grid forces one; by default the whole-GPU cooperative walk (39 us,
    // but it needs every SM) when the device is otherwise idle, the 8-CTA cluster walk (60 us on 8 SMs) when other
    // recordings are in flight on other streams (batch: 338 k vs 280 k Msamples/s at 64 streams).
    static const int forced = [] {
        const char *e = getenv("APTB200_PICK");
        if (!e) return -1;
        return !strcmp(e, "cluster") ? 1 : !strcmp(e, "grid") ? 2 : -1;
    }();
    const int mode = forced >= 0 ? forced : (c.busy ? 1 : 2);
    const u64 nr = (ncorr + row - 1) / row;
    if (scratch && mode == 1 && nr <= 20000) {
        // one 8-CTA cluster, jump tables in distributed shared memory (larger recordings: the whole-GPU cooperative grid)
        const size_t smem = 2ull * kPickClusterPer * sizeof(u32);
        static std::atomic<signed char> attr_cluster[kMaxDevices];
        if (smem_attr_once(attr_cluster, k_pick_cluster, smem)) {
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(8);
            cfg.blockDim = dim3(1024);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = c.stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = 8;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            PickScratch sc = *scratch;
            const unsigned j0_grid = (sc.cap + 1 + 255) / 256;      // one thread per possible node; the kernel knows how many exist
            k_pick_j0<<<j0_grid, 256, 0, c.stream>>>(ncorr, row, dist, ri, positions, max_positions, result, sc);
            APT_CUDA(cudaGetLastError());
            APT_CUDA(cudaLaunchKernelEx(&cfg, k_pick_cluster, ncorr, nwork, row, dist, ri, positions, max_positions, result, sc));
            nk = 2;
            return APT_OK;
        }
    }
    if (scratch) {
        // cooperative launch: the kernel's grid barriers need every CTA resident (1024 threads, no dynamic smem)
        int per_sm = 0;
        APT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pick_links, 1024, 0));
        const unsigned want = (scratch->cap + 1 + 1023) / 1024;
        const unsigned grid = std::max(1u, std::min(want, static_cast<unsigned>(std::max(per_sm, 1) * c.sm_count)));
        PickScratch sc = *scratch;
        void *args[] = {&ncorr, &nwork, &row, &dist, &ri, &positions, &max_positions, &result, &sc};
        APT_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void *>(k_pick_links), dim3(grid), dim3(1024), args, 0,
                                             c.stream));
    } else {
        k_pick_sequential<<<1, 32, 0, c.stream>>>(ncorr, nwork, row, dist, ri, positions, max_positions, result);
    }
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

u32 records_tile(u32 pw) { return static_cast<u32>(rec_tile_outputs(static_cast<int>(pw))); }

int launch_lowpass_records(const LaunchCtx &c, const float *e, u64 n, u64 ncorr, const float *taps_host, u32 ntaps, u32 pw,
                           SyncCtl *ctl, TileDesc *desc, Rec *pool, u32 pool_cap, u32 region, u32 ntiles) {
    if (ntiles == 0) return APT_OK;
    const LpTaps t = make_lp_taps(taps_host, ntaps);
    // one warp per CTA, as many CTAs as are resident; 9.4 KB of shared memory each needs no opt-in
    constexpr size_t smem = kRecSmemFloats * sizeof(float);
    static_assert(smem <= (48u << 10), "record kernel: dynamic shared memory above the default limit");
    auto launch = [&](auto kern) {
        static const int per_sm = [&] {
            int v = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kern, 32, smem) != cudaSuccess || v < 1) v = 1;
            return v;
        }();
        const unsigned grid = std::min<unsigned>(ntiles, static_cast<unsigned>(c.sm_count) * per_sm);
        kern<<<grid, 32, smem, c.stream>>>(e, n, ncorr, t, ctl, desc, pool, pool_cap, region, ntiles);
    };
    if (ntaps == 37 && pw == 3) launch(k_lowpass_records<37, 3>);
    else if (ntaps == 43 && pw == 4) launch(k_lowpass_records<43, 4>);
    else if (ntaps == 61 && pw == 5) launch(k_lowpass_records<61, 5>);
    else return fail(APT_ERR_BAD_ARG, "no fused low-pass/record kernel for %u taps, pixel width %u", ntaps, pw);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_resolve_roots(const LaunchCtx &c, const TileDesc *desc, const Rec *pool, u32 ntiles, u32 tile_w, u32 dist,
                         u64 ncorr, u32 *root_list, u32 *root_count, u32 *tile_base, u32 *by_id, SyncCtl *ctl,
                         SyncResult *result) {
    if (ntiles == 0) return APT_OK;
    const unsigned grid = (ntiles + kResolveThreads / 32 - 1) / (kResolveThreads / 32);
    k_resolve_roots<<<grid, kResolveThreads, 0, c.stream>>>(desc, pool, ntiles, tile_w, dist, ncorr, root_list, root_count, tile_base,
                                                            by_id, ctl, result);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_gather_lp(const LaunchCtx &c, const float *e, u64 n, const u32 *positions, const SyncResult *result,
                     u32 fixed_rows, u32 max_rows, u32 row, u32 px, u32 dec, const float *taps_host, u32 ntaps, float *out) {
    if (max_rows == 0) return APT_OK;
    const LpTaps lp = make_lp_taps(taps_host, ntaps, static_cast<int>(dec));
    const u32 part_px = (px / 2 + 3) / 4 * 4;
    const u32 eoff = (ntaps - 1 + 3) / 4 * 4;
    const size_t smem = 2 * (static_cast<size_t>(dec) * part_px + eoff + 12) * sizeof(float);  // double-buffered (the kernel's `span`)
    // persistent CTAs: exactly the resident ones (the register count decides: 3 per SM for 37 taps), and as many of those as
    // give every CTA the same number of half rows
    auto launch = [&](auto kern) {
        static const int per_sm = [&] {
            int v = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kern, kGatherLpThreads, smem) != cudaSuccess || v < 1) v = 1;
            return v;
        }();
        const u64 items = 2ull * max_rows;
        const u64 slots = static_cast<u64>(c.sm_count) * per_sm;
        const u64 rounds = (items + slots - 1) / slots;
        const unsigned grid = static_cast<unsigned>((items + rounds - 1) / rounds);
        kern<<<grid, kGatherLpThreads, smem, c.stream>>>(e, n, positions, result, fixed_rows, row, px, lp, out);
    };
    if (ntaps == 37 && dec == 3) launch(k_gather_rows_lp<37, 3>);
    else if (ntaps == 43 && dec == 4) launch(k_gather_rows_lp<43, 4>);
    else if (ntaps == 61 && dec == 5) launch(k_gather_rows_lp<61, 5>);
    else return fail(APT_ERR_BAD_ARG, "no fused gather kernel for %u taps, decimation %u", ntaps, dec);
    static_assert(kGatherLpThreads * 4 >= 1040, "one pass of a half row");
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_image_stage(const LaunchCtx &c, const float *rows, const SyncResult *result, u32 fixed_rows, u32 max_rows, u32 px,
                       int contrast, float percent, PostCtl *ctl, float *tel_a, float *tel_b, float *tel_v,
                       const float *bounds_dev, unsigned char *out, bool stats_only) {
    if (max_rows == 0) return APT_OK;
    const unsigned wide = static_cast<unsigned>(c.sm_count) * 8;
    if (!bounds_dev) {
        APT_CUDA(cudaMemsetAsync(ctl, 0, sizeof(PostCtl), c.stream));
        k_post_stats<<<std::min<unsigned>(max_rows, wide), 256, 0, c.stream>>>(rows, result, fixed_rows, px, ctl, tel_a, tel_b, tel_v);
        if (contrast == 1) k_post_histogram<<<wide / 2, 256, 0, c.stream>>>(rows, result, fixed_rows, px, ctl);
        k_post_bounds<<<1, 1024, 0, c.stream>>>(contrast, percent, result, fixed_rows, px, ctl, tel_a, tel_b, tel_v);
    }
    if (!stats_only) k_post_map_u8<<<wide, 256, 0, c.stream>>>(rows, result, fixed_rows, px, ctl, bounds_dev, out);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

int launch_quantize_i16(const LaunchCtx &c, const float *x, u64 n, PostCtl *ctl, short *out) {
    if (n == 0) return APT_OK;
    if (n >= (1ull << 32)) return fail(APT_ERR_BAD_ARG, "signal too long");
    APT_CUDA(cudaMemsetAsync(ctl, 0, sizeof(PostCtl), c.stream));
    const unsigned wide = static_cast<unsigned>(c.sm_count) * 8;
    // the signal as one "row" of n pixels: only the maximum is used
    k_post_stats<<<1, 256, 0, c.stream>>>(x, nullptr, 1, static_cast<u32>(n), ctl, nullptr, nullptr, nullptr);
    k_quantize_i16<<<wide, 256, 0, c.stream>>>(x, n, ctl, out);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

static size_t align_up(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

size_t pick_scratch_bytes(u32 max_blocks, u32 max_positions, u32 cap) {
    return align_up((static_cast<size_t>(max_blocks) + 1) * 4) + 4 * align_up((static_cast<size_t>(cap) + 1) * 4) +
           align_up((static_cast<size_t>(max_positions) + 1) * 4) + align_up(8);
}

PickScratch pick_scratch_carve(void *base, u32 max_blocks, u32 max_positions, u32 cap) {
    char *p = static_cast<char *>(base);
    auto take = [&](size_t count) {
        u32 *r = reinterpret_cast<u32 *>(p);
        p += align_up(count * 4);
        return r;
    };
    PickScratch s;
    s.block_off = take(static_cast<size_t>(max_blocks) + 1);
    s.cand_s = take(static_cast<size_t>(cap) + 1);
    s.cand_peak = take(static_cast<size_t>(cap) + 1);
    s.ja = take(static_cast<size_t>(cap) + 1);
    s.jb = take(static_cast<size_t>(cap) + 1);
    s.orbit = take(static_cast<size_t>(max_positions) + 1);
    s.ticket = take(2);
    s.cap = cap;
    return s;
}

int launch_gather(const LaunchCtx &c, const float *f, const u32 *positions, const SyncResult *result,
                  u32 fixed_rows, u32 max_rows, u32 row, u32 px, u32 dec, float *out) {
    if (max_rows == 0) return APT_OK;
    const unsigned grid = std::min<unsigned>(max_rows, static_cast<unsigned>(c.sm_count) * 16);
    k_gather_rows<<<grid, 256, 0, c.stream>>>(f, positions, result, fixed_rows, row, px, dec, out);
    APT_CUDA(cudaGetLastError());
    return APT_OK;
}

}  // namespace aptb200
