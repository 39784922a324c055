// Host-callable launchers of every kernel of the decode path (defined in launch.cu, the only
// translation unit that sees the kernels).  All pointers are device pointers.
#pragma once

#include <cstdint>
#include <vector>

#include <cuda_runtime.h>

namespace aptb200 {

typedef unsigned long long u64;
typedef unsigned int u32;

// Device-side summary of one decode (read back by the host after the stream drains).
struct SyncResult {
    u32 n_peaks;       // sync_pos.len()                       (decode.rs:110)
    u32 n_rows;        // rows that pass `pos + row < len`     (decode.rs:127)
    u32 status;        // APT_OK or APT_ERR_FEW_SYNC_FRAMES    (decode.rs:112-118)
    u32 seed_index;    // first i in [0, D] with corr[i] > 0, or 0xFFFFFFFF
    u32 n_roots;       // total number of roots (diagnostic)
    u32 pad[3];
};


// status code the device reports when the record pool of the fused sync stage overflowed: the host re-runs the stage with
// the legacy kernels (never leaves the library)
constexpr u32 kSyncRedo = 100;

// Control block of the fused sync stage (kernels_sync2.cuh); zeroed at the start of every job.
struct SyncCtl {
    u32 pad0;          // keeps the layout; pad[0] below is the picker's ticket
    u32 pool_cursor;   // record-pool entries handed out
    u32 overflow;      // the pool was exhausted
    u32 root_cursor;   // dense root ids handed out by k_resolve_roots (= number of roots when it is done)
    u32 pad[4];
};
struct TileDesc {      // one per tile of W correlation positions
    u32 off;           // first pool entry of the tile: ns suffix records, then np prefix records
    u32 ns, np;
    float tmax;        // maximum of the correlation over the tile
};
struct Rec {
    u32 pos;           // correlation index
    float val;
};
// Control / result block of the image stage (kernels_post.cuh); zeroed at the start of a job.
struct PostCtl {
    u32 nmin_key, max_key;   // ~key(min) and key(max) of the image under the monotone float -> u32 map
    u32 rows;                // image rows
    u32 status;              // 0 ok; 1 empty image; 2 percent: no low bucket; 3 too short for telemetry; 4 frame runs off the image
    float low, high;         // contrast bounds
    u32 telemetry_row, pad;
    float wedges_a[16], wedges_b[16];
    u32 buckets[1000];       // misc::percent histogram
};

// Where the picker finds the roots: per block of `block` positions an ascending list.
struct RootIndex {
    const u32 *list;
    const u32 *count;       // [nblocks] roots per block
    const u32 *base;        // [nblocks] dense id of the block's first root (may be nullptr for the sequential walk)
    const TileDesc *desc;   // list of block b starts at list + desc[b].off; nullptr: at list + b*block
    const u32 *by_id;       // root position by dense id; nullptr: `base` is an exclusive scan, found by binary search
    const u32 *nroots;      // total number of roots
    u32 block;
    u32 nblocks;
};

// Global scratch of the parallel peak picker (k_pick_parallel).
struct PickScratch {
    u32 *block_off;    // [nblocks + 1] exclusive scan of root_count (dense root numbering)
    u32 *cand_s;       // [cap + 1] start position of each candidate
    u32 *cand_peak;    // [cap + 1] firstroot(start)
    u32 *ja, *jb;      // [cap + 1] jump tables (J0, and the global ping-pong pair when smem is too small)
    u32 *orbit;        // [max_positions + 1]
    u32 *ticket;       // [2] last-CTA tickets of k_roots / k_pick_links (zero between launches)
    u32 cap;           // candidate capacity
};

// Geometry of the tiled kernel for one (L, M, taps) triple; built on the host (make_tile_plan).
struct TilePlan {
    u32 l, m;          // resampling ratio
    u32 halves;        // 2: groups of 8 outputs in two half windows; 1: groups of 4 outputs (one window)
    u32 groups;        // G = L / gcd(R, L), R = 4*halves (= compute warps per CTA); group g owns outputs R*g..R*g+R-1
    u32 p_out, p_in;   // outputs / inputs per super-period (p_out = 8G)
    u32 usteps;        // samples a group reads per row (= half_taps + shift), multiple of 16
    u32 half_taps;     // padded taps of one half (4 outputs), multiple of 16
    u32 shift;         // half B's window starts this many samples after half A's (multiple of 16)
    u32 iters;         // loop iterations = usteps / 16
    u32 row_len;       // samples of one row the kernel may touch (multiple of 4)
    u32 pair_pitch;    // floats between consecutive copies in shared memory
    u32 rows_per_copy; // 2: rows 2i, 2i+1 share one bulk copy (they overlap in the signal); 1: one copy per row
    u32 rows_floats;   // floats of the rows of one stage (qt * row_len)
    u32 plane_pitch;   // floats per row of a partial-sum plane (p_out + 4)
    u32 vec_magic;     // (v * vec_magic) >> 16 == v / (p_out/4) for every v < qt*p_out/4
    u32 qt;            // rows (super-periods) per tile
    u32 slice_stride;  // floats between the tap sub-tables of the 4 slice lanes (iters*32 + 8)
    u32 stage_floats;  // floats of one row stage (rows + halo row)
    u32 group_stride;  // floats of one group's tap table
    u32 smem_bytes;    // dynamic shared memory
    u32 ctas_per_sm;   // 2 when two CTAs fit an SM, else 1
    u64 off2;          // 2*((N-1)/2)
};

// Geometry of the uniform-tap kernel (kernels_ut.cuh) for one (L, M, taps) triple; built by make_ut_plan.
constexpr u32 kUtL = 13;               // the interpolation factor the kernel is instantiated for (48/96/192 kHz -> 12 480 Hz)
constexpr u32 kUtPairs = (kUtL + 1) / 2;   // packed accumulators per row
constexpr u32 kUtMaxVecSmall = 384;    // float4 entries of the tap stream: small / large parameter block
constexpr u32 kUtMaxVecLarge = 1900;
constexpr u32 kUtMaxSlots = 24;
constexpr u32 kUtChunk = 8;            // samples per loop iteration (chunk) of the kernel
struct UtPlan {
    u32 l, m;
    u32 np;            // pairs of outputs per row = ceil(L/2)
    u32 q;             // rows per thread: 2, or 1 when two rows do not fit shared memory (192 kHz input)
    u32 rb;            // rows per block = 32*q; a block = rb*L outputs from one contiguous span of the signal
    u32 vec;           // 4/2/1: widest aligned shared-memory load of a row's samples (M % 4 == 0 / M % 2 == 0 / odd)
    u32 back;          // samples staged in front of a block's first row (window of output k0-1), multiple of 4
    u32 chunks;        // a row touches samples [0, kUtChunk*chunks)
    u32 slot_floats;   // floats of one ring slot = back + (rb-1)*M + kUtChunk*chunks, rounded up to 4
    u32 slot_stride;   // floats between slots (slot_floats + 2*rb + 4 exchange words)
    u32 stream_b;      // float4 index of the second role's tap stream (roles: pairs [0, ceil(np/2)) and the rest)
    u32 nslot, warps;  // ring slots, compute warps
    u32 header_bytes;  // barriers, ticket and the halo output's taps in front of the slots (multiple of 128)
    u32 smem_bytes;
    u32 nvec;          // float4 entries of the tap stream
    u32 halo_u0, halo_n;   // output L-1: first sample relative to its row, number of taps
    u32 cs[8], ce[8];  // pair p is active in chunks [cs[p], ce[p])
    u64 off2;
};

// Geometry of the phase-major resampler (kernels_ph.cuh) for large interpolation factors; built by make_ph_plan.
constexpr u32 kPhTilePeriods = 32;   // periods (= l outputs each) per tile of the phase-major resampler
struct PhPlan {
    u32 l, m;
    u32 j, jpad;       // taps per output; jpad = WIN, the window four consecutive phases share (24 / 44 / 84 samples)
    u32 pitch;         // floats per shared-memory input row
    u32 row_len;       // samples staged per row
    u32 smem_bytes;
};

struct LaunchCtx {
    cudaStream_t stream;
    int sm_count;
    int busy = 0;      // other jobs are in flight on this device: prefer kernels with a small footprint (the 8-CTA cluster
                       // picker leaves 140 SMs to the other streams; alone, the whole-GPU cooperative walk is faster)
};

// fast_resampling (dsp.rs:186-289), optionally fused with demodulate (dsp.rs:350-383).
// format: APT_F32 / APT_PCM16 samples.
// Outputs [k_begin, k_end) only (k_end <= total outputs); `signal` is the address sample 0 would have.
int launch_polyphase(const LaunchCtx &c, const void *signal, int format, u64 len, const float *taps, u32 l, u32 m,
                     u64 off2, u64 k_begin, u64 k_end, bool envelope, float cosphi2, float sinphi, float *out);
// wav.rs:37: PCM16 -> f32 (both pointers 16-byte aligned).
int launch_pcm16_to_f32(const LaunchCtx &c, const int16_t *in, u64 n, float *out);
// dsp::filter + decimate (dsp.rs:396-404, 299-303).
int launch_fir_decimate(const LaunchCtx &c, const void *signal, int format, const float *coeff, u32 ntaps, u32 m,
                        u64 nout, float *out);
// dsp::demodulate (dsp.rs:350-383).
int launch_envelope(const LaunchCtx &c, const float *x, u64 n, float cosphi2, float sinphi, float *out);
// sync cross-correlation (decode.rs:225-233).
int launch_corr(const LaunchCtx &c, const float *f, u64 ncorr, const int8_t *guard, u32 glen, float *corr);
// Fused low-pass + sync correlation (kernels_lpsync.cuh).  Returns false when (ntaps, pixel width) has no
// instantiation -- the caller then uses launch_fir_decimate + launch_corr.  corr == nullptr: low-pass only.
bool lowpass_corr_supported(u32 ntaps, u32 pixel_width);
int launch_lowpass_corr(const LaunchCtx &c, const float *e, u64 n, const float *taps_host, u32 ntaps, u32 pixel_width,
                        float *f, float *corr);
// roots of the correlation (see kernels_sync.cuh).
int launch_roots(const LaunchCtx &c, const float *corr, u64 ncorr, u32 dist, u32 *root_list, u32 *root_count,
                 SyncResult *result, const PickScratch *scratch /* nullptr: no dense numbering */);
// orbit walk -> sync positions (decode.rs:241-253).
int launch_pick(const LaunchCtx &c, u64 ncorr, u64 nwork, u32 row, u32 dist, const RootIndex &ri, u32 *positions,
                u32 max_positions, SyncResult *result, const PickScratch *scratch /* nullptr: sequential walk */,
                int *kernels_launched = nullptr);
// Fused sync stage (kernels_sync2.cuh): low-pass + correlation + per-tile records, then the roots; f and corr never reach HBM.
u32 records_tile(u32 pixel_width);   // correlation positions per tile
int launch_lowpass_records(const LaunchCtx &c, const float *e, u64 n, u64 ncorr, const float *taps_host, u32 ntaps,
                           u32 pixel_width, SyncCtl *ctl, TileDesc *desc, Rec *pool, u32 pool_cap, u32 region, u32 ntiles);
int launch_resolve_roots(const LaunchCtx &c, const TileDesc *desc, const Rec *pool, u32 ntiles, u32 tile_w, u32 dist,
                         u64 ncorr, u32 *root_list, u32 *root_count, u32 *tile_base, u32 *by_id, SyncCtl *ctl,
                         SyncResult *result);
// aligned rows + final decimation with the low-pass evaluated per pixel from the envelope (f never exists in HBM).
int launch_gather_lp(const LaunchCtx &c, const float *e, u64 n, const u32 *positions, const SyncResult *result,
                     u32 fixed_rows, u32 max_rows, u32 row, u32 px, u32 dec, const float *taps_host, u32 ntaps, float *out);
// Bytes of scratch k_pick_parallel needs, and carving of one allocation into a PickScratch.
size_t pick_scratch_bytes(u32 max_blocks, u32 max_positions, u32 cap);
PickScratch pick_scratch_carve(void *base, u32 max_blocks, u32 max_positions, u32 cap);
// aligned rows + final decimation (decode.rs:122-134, 158-159).  positions == nullptr: no-sync rows.
int launch_gather(const LaunchCtx &c, const float *f, const u32 *positions, const SyncResult *result,
                  u32 fixed_rows, u32 max_rows, u32 row, u32 px, u32 dec, float *out);

// Image stage (SURVEY.md §8 f3): contrast bounds + telemetry statistics + u8 map of `rows` (f32, device), rows counted by
// `result` (sync decode) or fixed_rows.  contrast: 0 min/max, 1 percent, 2 telemetry (aptb200.h apt_contrast); bounds_dev !=
// nullptr: map with the two floats there instead (stage entry point).  tel_* are per-row scratch (max_rows floats each).
int launch_image_stage(const LaunchCtx &c, const float *rows, const SyncResult *result, u32 fixed_rows, u32 max_rows, u32 px,
                       int contrast, float percent, PostCtl *ctl, float *tel_a, float *tel_b, float *tel_v,
                       const float *bounds_dev, unsigned char *out, bool stats_only);

// wav.rs:71-85: normalise by the maximum and quantise to i16 (x, out: device; ctl: scratch control block).
int launch_quantize_i16(const LaunchCtx &c, const float *x, u64 n, PostCtl *ctl, short *out);

// Builds the geometry and the zero-padded per-group tap table of the tiled polyphase kernel for
// (l, m, taps).  Returns false when the shape does not fit the kernel (the generic kernel is used then).
bool make_tile_plan(u32 l, u32 m, const std::vector<float> &taps, TilePlan &tp, std::vector<float> &tile_taps,
                    std::vector<u32> &group_xs);
// Tiled fast_resampling (+ envelope).  f32 samples only.
// Tiles [tile_begin, tile_end) (tile_end == 0: all); `signal` is the address sample 0 would have.
int launch_polyphase_tiled(const LaunchCtx &c, const float *signal, u64 len, const float *tile_taps,
                           const u32 *group_xs, const TilePlan &tp, u64 nout, u64 tile_begin, u64 tile_end,
                           bool envelope, float cosphi2, float sinphi, float *out);

// Phase-major resampler (+ envelope) for large L (11025 / 22050 / 44100 Hz input).  make_ph_plan returns false when the
// shape does not fit (then the generic kernel serves it); table = [l/4][jpad][4] taps laid out against the groups' windows,
// xs = [l/4] window starts (row index), both go to HBM.
bool make_ph_plan(u32 l, u32 m, const std::vector<float> &taps, PhPlan &pp, std::vector<float> &table,
                  std::vector<unsigned short> &xs);
// Tiles of 32 periods (32*l outputs) [tile_begin, tile_end) (tile_end == 0: all); `signal` is the address sample 0 would have.
int launch_polyphase_ph(const LaunchCtx &c, const void *signal, int format, u64 len, const float *table_dev,
                        const unsigned short *xs_dev, const PhPlan &pp, u64 nout, u64 tile_begin, u64 tile_end, bool envelope,
                        float cosphi2, float sinphi, float *out);

// Uniform-tap resampler (+ envelope): taps travel as a kernel parameter.  Returns false from make_ut_plan when
// (l, m, taps) does not fit (L other than 13/14, tap stream too long, rows too long for shared memory).
bool make_ut_plan(u32 l, u32 m, const std::vector<float> &taps, UtPlan &up, std::vector<float> &stream);
// Blocks [blk_begin, blk_end) (blk_end == 0: all); `signal` is the 16-byte-aligned address sample 0 would have;
// `h` the filter taps in device memory (for the one halo output per block).
int launch_polyphase_ut(const LaunchCtx &c, const float *signal, u64 len, const float *h, const UtPlan &up,
                        const std::vector<float> &stream, u64 nout, u64 blk_begin, u64 blk_end, bool envelope,
                        float cosphi2, float sinphi, float *out);

}  // namespace aptb200
