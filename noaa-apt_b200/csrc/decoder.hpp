// The decoder object behind the C ABI: plan (filters, rates, sizes), device workspaces, one
// stream, and the kernel sequence of decode::decode (decode.rs:43-162).
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "aptb200.h"
#include <memory>

#include "filters_host.hpp"
#include "hostpool.hpp"
#include "launch.hpp"

namespace aptb200 {

// decode.rs:14-38
constexpr uint32_t kFinalRate = 4160;
constexpr uint32_t kPxPerRow = 2080;
constexpr uint32_t kCarrierHz = 2400;

// Everything decode() derives from (input_rate, settings) before touching a sample.
struct Plan {
    uint32_t input_rate = 0;
    apt_settings st{};
    Ratio first{};                 // input_rate -> work_rate (dsp.rs:73-75)
    bool first_polyphase = false;  // L > 1: fast_resampling; else filter + decimate
    std::vector<float> h;          // resampling filter taps (LowpassDcRemoval, decode.rs:65-76)
    uint64_t off2 = 0;             // 2 * ((N-1)/2): highest tap index fast_resampling touches
    std::vector<float> lp;         // demodulation low-pass taps (Lowpass, decode.rs:95-100)
    float cosphi2 = 0.f, sinphi = 1.f;   // dsp.rs:360-363
    uint32_t row = 0;              // samples_per_work_row (decode.rs:55)
    uint32_t dist = 0;             // min_distance (decode.rs:216)
    bool work_multiple = false;    // work_rate % 4160 == 0
    uint32_t dec = 0;              // work_rate / 4160 when work_multiple
    Ratio last{};                  // work_rate -> 4160 for the final NoFilter resample
    std::vector<int8_t> guard;     // sync template (empty unless work_multiple)
    bool tiled = false;            // the tiled sm_100a resampler fits this (L, M, taps)
    TilePlan tile{};
    std::vector<float> tile_taps;
    std::vector<u32> tile_xs;
    bool ph = false;               // the phase-major resampler (large L: 11025 / 22050 / 44100 Hz) fits
    PhPlan php{};
    std::vector<float> ph_table;
    std::vector<unsigned short> ph_xs;
    bool ut = false;               // the uniform-tap resampler (taps as a kernel parameter) fits: preferred
    UtPlan utp{};
    std::vector<float> ut_stream;
};

int make_plan(uint32_t input_rate, const apt_settings &s, Plan &plan);
// N_w for n input samples.
uint64_t plan_work_len(const Plan &p, uint64_t n);
// decode() output length for no-sync / upper bound for sync.
uint64_t plan_out_bound(const Plan &p, uint64_t n);

}  // namespace aptb200

struct apt_decoder {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    aptb200::Plan plan;

    uint64_t max_samples = 0, max_work = 0, max_corr = 0, max_out = 0;
    uint32_t max_blocks = 0, max_positions = 0;

    float *d_h = nullptr, *d_lp = nullptr, *d_one = nullptr;
    float *d_ph_table = nullptr;
    unsigned short *d_ph_xs = nullptr;
    float *d_tile_taps = nullptr;
    aptb200::u32 *d_tile_xs = nullptr;
    int8_t *d_guard = nullptr;
    void *d_in = nullptr;          // staging for submit_host (f32 sized)
    float *d_conv = nullptr;       // f32 copy of a PCM16 input for the tiled resampler (allocated on first use)
    // chunked upload of long host recordings (BASELINE configs[2]): two staging buffers of chunk_samples each,
    // a copy stream and events so that the H2D of chunk c+1 overlaps the resampling of chunk c
    uint64_t chunk_samples = 0;    // 0: the whole recording is staged at once
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    uint64_t job_chunks = 0;
    uint64_t conv_cap = 0;         // samples d_conv holds
    float *d_r = nullptr;          // resampled signal, only for the L == 1 first stage
    float *d_e = nullptr;          // envelope           ("demodulation_result")
    // fused sync stage (kernels_sync2.cuh): f and corr never reach HBM; per-tile records -> roots
    bool use_records = false;      // the fused stage serves this plan (standard / fast / slow profiles)
    aptb200::u32 tile_w = 0, max_tiles = 0, pool_cap = 0, pool_region = 0;   // pool_region: records of a tile's own pool region
    aptb200::SyncCtl *d_ctl = nullptr;
    aptb200::TileDesc *d_desc = nullptr;
    aptb200::Rec *d_pool = nullptr;
    aptb200::u32 *d_roots2 = nullptr;   // roots of tile t at d_roots2 + d_desc[t].off
    aptb200::u32 *d_tile_base = nullptr, *d_by_id = nullptr;   // dense root ids: first id of tile t, position by id
    bool job_fused = false;        // the current job ran the fused stage (f / corr were not materialised)
    bool last_fused = false;
    // legacy / debug buffers, allocated on first use (generic shapes, read_stage, pool overflow)
    float *d_f = nullptr;          // low-passed         ("filter_result")
    float *d_corr = nullptr;       // sync correlation   ("sync_correlation")
    float *d_aligned = nullptr;    // only when work_rate is not a multiple of 4160 (no-sync)
    aptb200::u32 *d_root_list = nullptr, *d_root_count = nullptr, *d_pos = nullptr;
    aptb200::SyncResult *d_res = nullptr;
    void *d_pick = nullptr;        // scratch of the parallel picker
    aptb200::PickScratch pick{};
    bool use_parallel_pick = true;
    bool use_fused_lowpass = true;
    bool job_corr_done = false;    // the correlation of the current job was produced by the fused low-pass kernel
    float *d_out = nullptr;        // rows for submit_host
    // pageable host buffers (what the reference-facing apt_decode receives) go through a pinned ring + copy threads
    aptb200::HostStager *stager = nullptr;                 // the one in use (own_stager, or the batch feeder's)
    std::unique_ptr<aptb200::HostStager> own_stager;
    float *h_out = nullptr;        // pinned landing buffer for the rows when the caller's buffer is pageable
    bool job_in_pageable = false, job_out_pageable = false;
    uint64_t job_d2h_floats = 0;   // rows copied back by the job (an upper bound when syncing: n_rows is not known yet)
    aptb200::SyncResult *h_res = nullptr;   // pinned

    // image mode (kernels_post.cuh): the job's output is the u8 image
    int image_contrast = -1;       // < 0: f32 rows
    float image_percent = 0.98f;
    aptb200::PostCtl *d_post = nullptr, *h_post = nullptr;   // device block; pinned copy of its head for the host
    float *d_tel = nullptr;        // 3 * max_rows floats: telemetry band means and variance per row
    unsigned char *d_out8 = nullptr;
    bool job_image = false;
    apt_image_info last_image{};

    // job in flight
    bool in_flight = false;
    bool job_host = false, job_sync = false;
    int job_status = APT_OK;
    uint64_t job_n = 0, job_work = 0, job_corr = 0, job_fixed_out = 0;
    const void *job_dev_in = nullptr;   // device address sample 0 would have (for a redo of the sync stage)
    float *job_out = nullptr;      // caller's buffer (host or device)
    uint64_t job_cap = 0;
    const float *job_rows_src = nullptr;
    uint64_t last_work = 0, last_rows = 0, last_peaks = 0, last_out = 0;

    // profiling
    bool profiling = false;
    std::vector<std::string> kernel_names;
    std::vector<cudaEvent_t> ev_begin, ev_end;
    std::vector<float> kernel_ms;
    int ev_used = 0;
    uint64_t launches = 0;

    apt_status_cb cb = nullptr;
    void *cb_user = nullptr;
};
