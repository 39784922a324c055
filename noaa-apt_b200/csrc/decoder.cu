// Decoder object and kernel sequence of decode::decode (decode.rs:43-162).
#include "decoder.hpp"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "common.hpp"
#include "launch.hpp"

namespace aptb200 {

std::string &last_error_slot() {
    static thread_local std::string slot;
    return slot;
}

int fail(int status, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error_slot() = buf;
    return status;
}

// ------------------------------------------------------------------------------------- plan

int make_plan(uint32_t input_rate, const apt_settings &s, Plan &p) {
    p = Plan{};
    p.input_rate = input_rate;
    p.st = s;
    if (s.work_rate > UINT32_MAX / kPxPerRow)   // PX_PER_ROW * work_rate overflows u32 (decode.rs:55)
        return fail(APT_ERR_BAD_ARG, "work_rate %u is too large", s.work_rate);

    // decode.rs:65-77 -> dsp::resample_with_filter (dsp.rs:62-98)
    int st = resample_ratio(input_rate, s.work_rate, p.first);
    if (st == APT_ERR_RESAMPLE_TO_ZERO) return fail(st, "Can't resample to 0Hz");
    if (st == APT_ERR_RATE_OVERFLOW)
        return fail(st, "Can't resample, looks like the sample rates do not have a big divisor in common. "
                        "input_rate: %u, output_rate: %u, l: %u, m: %u",
                    input_rate, s.work_rate, p.first.l, p.first.m);
    if (st != APT_OK) return fail(st, "invalid input rate %u", input_rate);
    p.first_polyphase = p.first.l > 1;

    apt_filter rf{APT_FILTER_LOWPASS_DC, Freq::hz(s.resample_cutout, input_rate).get_pi_rad(), s.resample_atten,
                  Freq::hz(s.resample_delta_freq, input_rate).get_pi_rad()};
    if (p.first_polyphase) resample_filter(rf, input_rate, input_rate * p.first.l);   // dsp.rs:93
    st = design(rf, p.h);
    if (st != APT_OK) return fail(st, "resampling filter cannot be designed (atten %g, delta_w %g)",
                                  (double)rf.atten, (double)rf.delta_w_pi);
    p.off2 = 2 * ((static_cast<uint64_t>(p.h.size()) - 1) / 2);
    p.tiled = p.first_polyphase && !getenv("APTB200_GENERIC_RESAMPLER") &&
              make_tile_plan(p.first.l, p.first.m, p.h, p.tile, p.tile_taps, p.tile_xs);
    p.ut = p.first_polyphase && !getenv("APTB200_GENERIC_RESAMPLER") &&
           make_ut_plan(p.first.l, p.first.m, p.h, p.utp, p.ut_stream);
    p.ph = p.first_polyphase && !p.ut && !p.tiled && !getenv("APTB200_GENERIC_RESAMPLER") &&
           make_ph_plan(p.first.l, p.first.m, p.h, p.php, p.ph_table, p.ph_xs);

    // decode.rs:95-100
    const float cut = static_cast<float>(kFinalRate) / static_cast<float>(s.work_rate);
    apt_filter lf{APT_FILTER_LOWPASS, cut, s.demodulation_atten, cut / 5.f};
    st = design(lf, p.lp);
    if (st != APT_OK) return fail(st, "demodulation filter cannot be designed (atten %g)", (double)lf.atten);

    // decode.rs:89 + dsp.rs:360-363
    const float phi = 2.f * Freq::hz(static_cast<float>(kCarrierHz), s.work_rate).get_rad();
    p.cosphi2 = std::cos(phi) * 2.f;
    p.sinphi = std::sin(phi);

    p.row = kPxPerRow * s.work_rate / kFinalRate;                       // decode.rs:55
    if (p.row == 0)   // work_rate < 2: the reference divides by zero (decode.rs:141); a status is the safe equivalent
        return fail(APT_ERR_BAD_ARG, "work_rate %u is too low: zero samples per image row", s.work_rate);
    p.dist = static_cast<uint32_t>(static_cast<uint64_t>(p.row) * 8 / 10);   // decode.rs:216
    p.work_multiple = s.work_rate % kFinalRate == 0;
    p.dec = s.work_rate / kFinalRate;
    if (p.work_multiple) sync_frame(s.work_rate, p.guard);
    // final stage ratio, decode.rs:158-159 (errors surface when the stage runs)
    p.last = Ratio{0, 0};
    resample_ratio(s.work_rate, kFinalRate, p.last);
    return APT_OK;
}

uint64_t plan_work_len(const Plan &p, uint64_t n) {
    if (p.first_polyphase) return polyphase_len(n, p.first.l, p.first.m, p.h.size());
    return n / p.first.m;   // decimate, dsp.rs:299-301
}

uint64_t plan_out_bound(const Plan &p, uint64_t n) {
    const uint64_t nw = plan_work_len(p, n);
    if (p.row == 0) return 0;
    const uint64_t rows = nw / p.row;
    if (p.work_multiple) return rows * kPxPerRow;
    return polyphase_len(rows * p.row, p.last.l, p.last.m, 1);
}

// ---------------------------------------------------------------------------------- helpers

namespace {

struct Prof {
    apt_decoder *d;
    int slot;
    Prof(apt_decoder *dec, const char *name) : d(dec), slot(-1) {
        d->launches++;
        if (!d->profiling) return;
        slot = d->ev_used++;
        if (slot >= static_cast<int>(d->ev_begin.size())) {
            cudaEvent_t a, b;
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            d->ev_begin.push_back(a);
            d->ev_end.push_back(b);
            d->kernel_names.emplace_back();
        }
        d->kernel_names[slot] = name;
        cudaEventRecord(d->ev_begin[slot], d->stream);
    }
    ~Prof() {
        if (slot >= 0) cudaEventRecord(d->ev_end[slot], d->stream);
    }
};

}  // namespace

// Cross-correlation + roots + orbit walk: decode::find_sync (decode.rs:204-263) on d_f[0..nwork).
int run_find_sync(apt_decoder *d, uint64_t nwork) {
    const Plan &p = d->plan;
    const LaunchCtx c{d->stream, d->sm_count};
    const uint32_t glen = static_cast<uint32_t>(p.guard.size());
    const uint64_t ncorr = nwork - glen;
    const uint32_t nblocks = static_cast<uint32_t>((ncorr + p.dist - 1) / p.dist);
    if (!d->job_corr_done) {
        Prof pr(d, "sync_correlation");
        APT_TRY(launch_corr(c, d->d_f, ncorr, d->d_guard, glen, d->d_corr));
    }
    {
        Prof pr(d, "sync_roots");
        APT_TRY(launch_roots(c, d->d_corr, ncorr, p.dist, d->d_root_list, d->d_root_count, d->d_res,
                             d->use_parallel_pick && d->d_pick ? &d->pick : nullptr));
    }
    {
        Prof pr(d, "sync_pick");
        const u32 *boff = d->d_pick ? d->pick.block_off : nullptr;
        const RootIndex ri{d->d_root_list, d->d_root_count, boff, nullptr, nullptr, boff ? boff + nblocks : nullptr, p.dist, nblocks};
        APT_TRY(launch_pick(c, ncorr, nwork, p.row, p.dist, ri, d->d_pos, d->max_positions, d->d_res,
                            d->use_parallel_pick && d->d_pick ? &d->pick : nullptr));
    }
    return APT_OK;
}

// Legacy / debug buffers (f, corr, per-block root lists): generic shapes, read_stage, and the redo after a record-pool
// overflow.  Allocated on first use.
int ensure_legacy_sync(apt_decoder *d) {
    const Plan &p = d->plan;
    APT_CUDA(cudaSetDevice(d->device));
    const size_t work_bytes = std::max<uint64_t>(d->max_work, 1) * sizeof(float);
    if (!d->d_f) APT_CUDA(cudaMalloc(&d->d_f, work_bytes));
    if (p.work_multiple && d->max_corr) {
        if (!d->d_corr) APT_CUDA(cudaMalloc(&d->d_corr, d->max_corr * sizeof(float)));
        if (!d->d_root_list) APT_CUDA(cudaMalloc(&d->d_root_list, static_cast<size_t>(d->max_blocks) * p.dist * sizeof(u32)));
    }
    return APT_OK;
}

// The back half with f and corr materialised in HBM: low-pass (+ correlation), roots, orbit walk, row gather.
static int enqueue_back_legacy(apt_decoder *d, uint64_t nwork, int sync, float *rows_out) {
    const Plan &p = d->plan;
    const LaunchCtx c{d->stream, d->sm_count};
    APT_TRY(ensure_legacy_sync(d));
    d->job_corr_done = false;
    const bool want_corr = sync && p.work_multiple && d->d_corr != nullptr;
    const u32 ntaps = static_cast<u32>(p.lp.size());
    if (d->use_fused_lowpass && lowpass_corr_supported(ntaps, p.dec) && p.work_multiple) {
        // low-pass and (when syncing) the sync cross-correlation in one pass over the envelope
        Prof pr(d, want_corr ? "lowpass_correlation" : "lowpass");
        APT_TRY(launch_lowpass_corr(c, d->d_e, nwork, p.lp.data(), ntaps, p.dec, d->d_f, want_corr ? d->d_corr : nullptr));
        d->job_corr_done = want_corr;
    } else {
        Prof pr(d, "lowpass");
        APT_TRY(launch_fir_decimate(c, d->d_e, APT_F32, d->d_lp, ntaps, 1, nwork, d->d_f));
    }
    if (sync) {
        APT_TRY(run_find_sync(d, nwork));
        Prof pr(d, "gather_rows");
        const u32 max_rows = static_cast<u32>(std::min<uint64_t>(nwork / p.row + 1, 1u << 30));
        APT_TRY(launch_gather(c, d->d_f, d->d_pos, d->d_res, 0, max_rows, p.row, kPxPerRow, p.dec, rows_out));
    }
    return APT_OK;
}

// Re-runs the sync stage of the job that just drained with the legacy kernels (record pool overflow); d_e is intact.
int redo_sync_legacy(apt_decoder *d) {
    APT_CUDA(cudaMemsetAsync(d->d_res, 0, sizeof(SyncResult), d->stream));
    return enqueue_back_legacy(d, d->job_work, 1, const_cast<float *>(d->job_rows_src));
}

// On-demand f / corr of the last job for read_stage after a fused run.
int materialise_stages(apt_decoder *d) {
    const Plan &p = d->plan;
    const LaunchCtx c{d->stream, d->sm_count};
    APT_TRY(ensure_legacy_sync(d));
    const u32 ntaps = static_cast<u32>(p.lp.size());
    APT_TRY(launch_lowpass_corr(c, d->d_e, d->last_work, p.lp.data(), ntaps, p.dec, d->d_f, d->d_corr));
    APT_CUDA(cudaStreamSynchronize(d->stream));
    d->last_fused = false;
    return APT_OK;
}

// one of the two TMA-staged resamplers serves this decoder's first stage (they take f32 samples only)
static bool fast_front(const apt_decoder *d) { return d->plan.ut || (d->plan.tiled && d->d_tile_taps); }
static bool ph_front(const apt_decoder *d) { return d->plan.ph && d->d_ph_table; }

// fast_resampling + demodulate of outputs produced from a device-resident (or staged) chunk.
// `in` is the address sample 0 of the recording would have (a biased pointer for chunk buffers).
static int launch_front_polyphase(apt_decoder *d, const void *in, int format, uint64_t n, uint64_t nwork,
                                  uint64_t tile_begin, uint64_t tile_end, uint64_t k_begin, uint64_t k_end,
                                  float *conv_base /* f32 view of a PCM16 chunk (already biased) or nullptr */) {
    const Plan &p = d->plan;
    const LaunchCtx c{d->stream, d->sm_count};
    if (p.ut && (format == APT_F32 || conv_base)) {
        const float *fin = format == APT_F32 ? static_cast<const float *>(in) : conv_base;
        if ((reinterpret_cast<uintptr_t>(fin) & 15) == 0)
            return launch_polyphase_ut(c, fin, n, d->d_h, p.utp, p.ut_stream, nwork, tile_begin, tile_end, true, p.cosphi2,
                                       p.sinphi, d->d_e);
    }
    if (p.tiled && d->d_tile_taps && (format == APT_F32 || conv_base)) {
        const float *fin = format == APT_F32 ? static_cast<const float *>(in) : conv_base;
        return launch_polyphase_tiled(c, fin, n, d->d_tile_taps, d->d_tile_xs, p.tile, nwork, tile_begin, tile_end, true,
                                      p.cosphi2, p.sinphi, d->d_e);
    }
    if (ph_front(d))   // large L: phase-major kernel, f32 or PCM16 samples (the cast is part of its row staging)
        return launch_polyphase_ph(c, in, format, n, d->d_ph_table, d->d_ph_xs, p.php, nwork, tile_begin, tile_end, true, p.cosphi2,
                                   p.sinphi, d->d_e);
    return launch_polyphase(c, in, format, n, d->d_h, p.first.l, p.first.m, p.off2, k_begin, k_end ? k_end : nwork, true,
                            p.cosphi2, p.sinphi, d->d_e);
}

// Long host recording: upload in chunks (with the filter-length overlap each chunk needs) on the copy stream while
// the previous chunk is resampled on the compute stream.  Only the polyphase first stage is chunked.
static int enqueue_front_chunked(apt_decoder *d, const void *host, int format, uint64_t n, uint64_t nwork) {
    const Plan &p = d->plan;
    const LaunchCtx c{d->stream, d->sm_count};
    const size_t sb = format == APT_PCM16 ? 2 : 4;
    const uint64_t cap = d->chunk_samples;
    const bool tiled = fast_front(d) || ph_front(d);
    const uint64_t l = p.first.l, m = p.first.m;
    uint64_t units, per_chunk;            // tiles / blocks or outputs
    // a unit (tile of the warp-specialised kernel, block of the uniform-tap kernel) reads unit_in new samples,
    // plus `before` samples in front of the first unit of a chunk and `after` beyond the start of the last one
    uint64_t unit_in = 0, unit_out = 0, before = 0, after = 0;
    if (p.ut) {
        unit_in = static_cast<uint64_t>(p.utp.rb) * m;
        unit_out = static_cast<uint64_t>(p.utp.rb) * l;
        before = p.utp.back;
        after = p.utp.slot_floats - p.utp.back;           // a block's span beyond its first row's first sample
    } else if (ph_front(d)) {
        unit_in = static_cast<uint64_t>(kPhTilePeriods) * m;              // a tile = 32 periods of m samples
        unit_out = static_cast<uint64_t>(kPhTilePeriods) * l;
        before = m + 4;                                                   // the period in front of the tile (+4 alignment)
        after = static_cast<uint64_t>(kPhTilePeriods - 1) * m + p.php.row_len;
    } else if (tiled) {
        unit_in = static_cast<uint64_t>(p.tile.qt) * p.tile.p_in;
        unit_out = static_cast<uint64_t>(p.tile.qt) * p.tile.p_out;
        before = p.tile.p_in - d->plan.tile_xs.back();    // halo row: window of the last group one super-period back
        after = static_cast<uint64_t>(p.tile.qt - 1) * p.tile.p_in + p.tile.row_len;
    }
    if (tiled) {
        units = (nwork + unit_out - 1) / unit_out;
        if (cap < before + after + unit_in + 64) return fail(APT_ERR_BAD_ARG, "chunk too small for one tile");
        per_chunk = (cap - before - after - 64) / unit_in + 1;
    } else {
        units = nwork;
        const uint64_t halo = p.off2 / l + 4;
        if (cap < 2 * halo + 1024) return fail(APT_ERR_BAD_ARG, "chunk too small for the filter");
        per_chunk = (cap - 2 * halo) * l / m;
    }
    if (per_chunk == 0) return fail(APT_ERR_BAD_ARG, "chunk too small");
    char *stage[2] = {static_cast<char *>(d->d_in), static_cast<char *>(d->d_in) + cap * 4};
    uint64_t chunk = 0;
    for (uint64_t u0 = 0; u0 < units; u0 += per_chunk, ++chunk) {
        const uint64_t u1 = std::min(units, u0 + per_chunk);
        const int b = static_cast<int>(chunk & 1);
        uint64_t xa, xb;
        if (tiled) {
            xa = u0 == 0 ? 0 : u0 * unit_in - before;
            xb = std::min<uint64_t>(n, (u1 - 1) * unit_in + after);
        } else {
            const uint64_t kfirst = u0 == 0 ? 0 : u0 - 1;                    // the envelope needs r[k0 - 1]
            xa = (kfirst * m + l - 1) / l;
            xa &= ~static_cast<uint64_t>(7);                                  // keep 16-byte alignment of PCM16 chunks
            xb = std::min<uint64_t>(n, ((u1 - 1) * m + p.off2) / l + 1);
        }
        if (xb <= xa || xb - xa > cap) return fail(APT_ERR_BAD_ARG, "internal: chunk geometry (%llu..%llu, cap %llu)",
                                                   (unsigned long long)xa, (unsigned long long)xb, (unsigned long long)cap);
        // copy stream: wait until the compute stream has finished with this buffer, then upload
        if (chunk >= 2) APT_CUDA(cudaStreamWaitEvent(d->copy_stream, d->ev_free[b], 0));
        if (d->job_in_pageable && d->stager)
            APT_CUDA(d->stager->upload(stage[b], static_cast<const char *>(host) + xa * sb, (xb - xa) * sb, d->copy_stream));
        else
            APT_CUDA(cudaMemcpyAsync(stage[b], static_cast<const char *>(host) + xa * sb, (xb - xa) * sb, cudaMemcpyHostToDevice,
                                     d->copy_stream));
        APT_CUDA(cudaEventRecord(d->ev_copied[b], d->copy_stream));
        APT_CUDA(cudaStreamWaitEvent(d->stream, d->ev_copied[b], 0));
        // compute stream: (cast,) resample + envelope of this chunk's outputs
        const void *in_biased = stage[b] - xa * sb;
        float *conv_biased = nullptr;
        if (format == APT_PCM16 && fast_front(d)) {
            APT_TRY(launch_pcm16_to_f32(c, reinterpret_cast<const int16_t *>(stage[b]), xb - xa, d->d_conv));
            d->launches++;
            conv_biased = d->d_conv - xa;
        }
        d->launches++;
        APT_TRY(launch_front_polyphase(d, in_biased, format, n, nwork, tiled ? u0 : 0, tiled ? u1 : 0, tiled ? 0 : u0,
                                       tiled ? 0 : u1, conv_biased));
        APT_CUDA(cudaEventRecord(d->ev_free[b], d->stream));
    }
    d->job_chunks = chunk;
    return APT_OK;
}

static int enqueue_front(apt_decoder *d, const void *in, int format, uint64_t n, uint64_t nwork, const void *host_chunked) {
    const Plan &p = d->plan;
    const LaunchCtx c{d->stream, d->sm_count};
    if (d->cb) {
        char msg[64];
        snprintf(msg, sizeof(msg), "Resampling to %u", p.st.work_rate);
        d->cb(0.1f, msg, d->cb_user);                                       // decode.rs:63
    }
    d->job_chunks = 0;
    if (p.first_polyphase) {
        // fast_resampling + demodulate fused: r is never written (decode.rs:77,89)
        Prof pr(d, "resample_envelope");
        if (host_chunked) {
            APT_TRY(enqueue_front_chunked(d, host_chunked, format, n, nwork));
        } else {
            float *conv = nullptr;
            if (format == APT_PCM16 && fast_front(d) && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
                // the WAV's int16 samples: `as f32` (wav.rs:37) on the device, then the same tiled kernel
                if (d->conv_cap < n) {
                    if (d->d_conv) APT_CUDA(cudaFree(d->d_conv));
                    d->d_conv = nullptr;
                    d->conv_cap = 0;
                    APT_CUDA(cudaMalloc(&d->d_conv, std::max<uint64_t>(d->max_samples, n) * sizeof(float)));
                    d->conv_cap = std::max<uint64_t>(d->max_samples, n);
                }
                APT_TRY(launch_pcm16_to_f32(c, static_cast<const int16_t *>(in), n, d->d_conv));
                d->launches++;
                conv = d->d_conv;
            }
            APT_TRY(launch_front_polyphase(d, in, format, n, nwork, 0, 0, 0, 0, conv));
        }
        if (d->cb) d->cb(0.4f, "Demodulating", d->cb_user);                 // decode.rs:87
    } else {
        {
            Prof pr(d, "filter_decimate");
            APT_TRY(launch_fir_decimate(c, in, format, d->d_h, static_cast<u32>(p.h.size()), p.first.m, nwork, d->d_r));
        }
        if (d->cb) d->cb(0.4f, "Demodulating", d->cb_user);
        Prof pr(d, "envelope");
        APT_TRY(launch_envelope(c, d->d_r, nwork, p.cosphi2, p.sinphi, d->d_e));
    }
    if (d->cb) d->cb(0.42f, "Filtering", d->cb_user);                       // decode.rs:93
    return APT_OK;
}

// Enqueues the whole of decode() on the decoder's stream.  `in` and `rows_out` are device pointers.
std::atomic<int> g_jobs_in_flight[64];      // per CUDA device: decodes submitted and not yet waited for

int decoder_enqueue(apt_decoder *d, const void *in, int format, uint64_t n, int sync, float *rows_out,
                    const void *host_chunked) {
    const Plan &p = d->plan;
    LaunchCtx c{d->stream, d->sm_count};
    c.busy = d->device >= 0 && d->device < 64 && g_jobs_in_flight[d->device].load(std::memory_order_relaxed) > 0 ? 1 : 0;
    const uint64_t nwork = plan_work_len(p, n);
    d->job_work = nwork;
    d->ev_used = 0;

    if (sync && d->use_records && d->d_ctl) APT_CUDA(cudaMemsetAsync(d->d_ctl, 0, sizeof(SyncCtl), d->stream));
    APT_TRY(enqueue_front(d, in, format, n, nwork, host_chunked));
    d->job_fused = false;
    const u32 ntaps = static_cast<u32>(p.lp.size());

    if (sync) {
        if (!p.work_multiple) {
            if (d->cb) d->cb(0.5f, "Syncing", d->cb_user);                  // decode.rs:107
            return fail(APT_ERR_WORK_RATE, "work_rate is not multiple of FINAL_RATE");   // decode.rs:172-176
        }
        d->job_fixed_out = 0;
        if (d->use_records && d->d_pool) {
            // fused stage: f and corr stay on chip; records -> roots -> orbit -> rows straight from the envelope
            const u64 ncorr = nwork - p.guard.size();
            const u32 ntiles = static_cast<u32>((ncorr + d->tile_w - 1) / d->tile_w);
            d->job_fused = true;
            {
                Prof pr(d, "lowpass_records");
                APT_TRY(launch_lowpass_records(c, d->d_e, nwork, ncorr, p.lp.data(), ntaps, p.dec, d->d_ctl, d->d_desc, d->d_pool,
                                               d->pool_cap, d->pool_region, ntiles));
            }
            if (d->cb) d->cb(0.5f, "Syncing", d->cb_user);
            {
                Prof pr(d, "resolve_roots");
                APT_TRY(launch_resolve_roots(c, d->d_desc, d->d_pool, ntiles, d->tile_w, p.dist, ncorr, d->d_roots2, d->d_root_count,
                                             d->d_tile_base, d->d_by_id, d->d_ctl, d->d_res));
            }
            {
                Prof pr(d, "sync_pick");
                const RootIndex ri{d->d_roots2, d->d_root_count, d->d_tile_base, d->d_desc, d->d_by_id, &d->d_ctl->root_cursor,
                                   d->tile_w, ntiles};
                int nk = 1;
                APT_TRY(launch_pick(c, ncorr, nwork, p.row, p.dist, ri, d->d_pos, d->max_positions, d->d_res,
                                    d->use_parallel_pick && d->d_pick ? &d->pick : nullptr, &nk));
                d->launches += static_cast<uint64_t>(nk - 1);               // Prof counted one
            }
            if (d->cb) d->cb(0.9f, "Resampling to 4160", d->cb_user);       // decode.rs:154
            Prof pr(d, "gather_rows");
            const u32 max_rows = static_cast<u32>(std::min<uint64_t>(nwork / p.row + 1, 1u << 30));
            APT_TRY(launch_gather_lp(c, d->d_e, nwork, d->d_pos, d->d_res, 0, max_rows, p.row, kPxPerRow, p.dec, p.lp.data(), ntaps,
                                     rows_out));
            return APT_OK;
        }
        if (d->cb) d->cb(0.5f, "Syncing", d->cb_user);
        APT_TRY(enqueue_back_legacy(d, nwork, 1, rows_out));
        if (d->cb) d->cb(0.9f, "Resampling to 4160", d->cb_user);
        return APT_OK;
    }

    if (d->cb) d->cb(0.5f, "Skipping Syncing", d->cb_user);                 // decode.rs:136
    const uint64_t rows = nwork / p.row;                                    // decode.rs:141-147
    if (d->cb) d->cb(0.9f, "Resampling to 4160", d->cb_user);
    if (p.work_multiple) {
        if (d->use_records) {
            d->job_fused = true;
            Prof pr(d, "gather_rows");
            APT_TRY(launch_gather_lp(c, d->d_e, nwork, nullptr, d->d_res, static_cast<u32>(rows), static_cast<u32>(rows), p.row,
                                     kPxPerRow, p.dec, p.lp.data(), ntaps, rows_out));
        } else {
            APT_TRY(enqueue_back_legacy(d, nwork, 0, rows_out));
            Prof pr(d, "gather_rows");
            APT_TRY(launch_gather(c, d->d_f, nullptr, d->d_res, static_cast<u32>(rows), static_cast<u32>(rows), p.row,
                                  kPxPerRow, p.dec, rows_out));
        }
        d->job_fixed_out = rows * kPxPerRow;
        return APT_OK;
    }
    APT_TRY(enqueue_back_legacy(d, nwork, 0, rows_out));
    // work_rate is not a multiple of 4160: the final stage is a real L/M resample with the one-tap
    // NoFilter (dsp.rs:79-98), i.e. zero-stuffing then keeping every M-th sample.
    if (p.last.l == 0) return fail(APT_ERR_RESAMPLE_TO_ZERO, "Can't resample to 0Hz");
    if (static_cast<uint64_t>(p.st.work_rate) * p.last.l > UINT32_MAX)
        return fail(APT_ERR_RATE_OVERFLOW, "Can't resample, looks like the sample rates do not have a big divisor "
                                           "in common. input_rate: %u, output_rate: %u", p.st.work_rate, kFinalRate);
    const uint64_t alen = rows * p.row;
    const uint64_t nout = polyphase_len(alen, p.last.l, p.last.m, 1);
    Prof pr(d, "final_resample");
    APT_TRY(launch_polyphase(c, d->d_f, APT_F32, alen, d->d_one, p.last.l, p.last.m, 0, 0, nout, false, 0.f, 1.f, rows_out));
    d->job_fixed_out = nout;
    return APT_OK;
}

}  // namespace aptb200
