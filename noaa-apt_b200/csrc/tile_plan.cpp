// Host-side geometry of the tiled polyphase kernel (kernels_fast.cuh).
#include <algorithm>
#include <numeric>

#include "launch.hpp"

namespace aptb200 {

namespace {
constexpr u32 kH = 4, kQ = 4, kKS = 4, kQT = (32 / kKS) * kQ;
constexpr u32 kMaxGroups = 13;                 // warps per CTA the kernel is compiled for (416 threads)
constexpr u32 kSmemTwoCtas = (233472 - 2 * 1024) / 2 - 512;   // dynamic bytes that still let two CTAs share an SM
constexpr u32 kSmemOneCta = 227 * 1024;
constexpr u32 kIterSamples = 4 * kKS;          // samples consumed per loop iteration (one 16-byte chunk per slice lane)
}  // namespace

// One attempt with R = 4*halves outputs per group (halves = 2: two half windows per group; 1: a single one).
static bool try_tile_plan(u32 halves, u32 l, u32 m, const std::vector<float> &taps, TilePlan &tp,
                          std::vector<float> &tile_taps, std::vector<u32> &group_xs) {
    const u32 kR = kH * halves;
    if (l < 2 || m == 0 || taps.empty()) return false;
    const u64 off2 = 2 * ((static_cast<u64>(taps.size()) - 1) / 2);
    const u32 groups = l / std::gcd(kR, l);
    if (groups > kMaxGroups) return false;
    const u64 p_out = static_cast<u64>(kR) * groups;
    const u64 p_in = p_out * m / l;            // exact: p_out is a multiple of l
    if (p_in % 4 != 0 || p_in > (1u << 20)) return false;

    // Per group: outputs k0..k0+3 (half A) and k0+4..k0+7 (half B).  Half B's window starts `shift`
    // samples after half A's, so the first shift/16 loop iterations touch only A and the last only B.
    auto first_x = [&](u64 k) { return (k * m + l - 1) / l; };          // first sample output k touches
    auto last_x = [&](u64 k) { return (k * m + off2) / l; };            // last one
    u64 d_min = ~0ull, d_max = 0;
    for (u32 g = 0; g < groups && halves == 2; ++g) {
        const u64 k0 = static_cast<u64>(kR) * g;
        const u64 d = first_x(k0 + kH) - first_x(k0);
        d_min = std::min(d_min, d);
        d_max = std::max(d_max, d);
    }
    if (halves == 1) d_min = d_max = 0;
    // Candidate shifts (multiples of one loop iteration).  A larger shift than the smallest spacing is fine
    // as long as every group's window start is pulled back far enough for half B to still see its first tap.
    u64 shift = 0, ua = 0, max_w0 = 0;
    bool have = false;
    const u64 cands[3] = {0, d_min / kIterSamples * kIterSamples, (d_max + kIterSamples - 1) / kIterSamples * kIterSamples};
    for (u64 cand : cands) {
        std::vector<u32> xs(groups);
        u64 need = 0, mw = 0;
        bool ok = true;
        for (u32 g = 0; g < groups && ok; ++g) {
            const u64 k0 = static_cast<u64>(kR) * g;
            if (halves == 2 && first_x(k0 + kH) < cand) { ok = false; break; }
            const u64 w0 = (halves == 2 ? std::min(first_x(k0), first_x(k0 + kH) - cand) : first_x(k0)) &
                           ~static_cast<u64>(3);                                // 16-byte aligned
            xs[g] = static_cast<u32>(w0);
            need = std::max(need, last_x(k0 + kH - 1) - w0 + 1);               // half A relative to w0
            if (halves == 2) need = std::max(need, last_x(k0 + kR - 1) - (w0 + cand) + 1);   // half B relative to w0 + shift
            mw = std::max(mw, w0);
        }
        if (!ok) continue;
        const u64 cand_ua = (need + kIterSamples - 1) / kIterSamples * kIterSamples;   // taps per half, padded
        if (!have || cand_ua < ua || (cand_ua == ua && cand_ua + cand < ua + shift)) {
            have = true;
            shift = cand;
            ua = cand_ua;
            max_w0 = mw;
            group_xs = xs;
        }
    }
    if (!have) return false;
    const u64 span = ua + shift;                                              // samples a group reads per row
    const u64 iters = span / kIterSamples;
    // Rows are staged in pairs: one bulk copy brings rows 2i and 2i+1 (they are p_in apart in the signal and
    // overlap), pairs are pair_pitch floats apart.  pair_pitch is padded until the 8 row lanes of a quarter-warp
    // (rows r = 0..7: pair r/2, half r%2) start in 8 different 16-byte bank groups -> conflict-free LDS.128.
    const u64 row_len = (max_w0 + span + 3) / 4 * 4;     // samples of one row the kernel may touch
    u64 pair_pitch = p_in + row_len;
    u32 rows_per_copy = 2;
    for (;; pair_pitch += 4) {
        u32 seen = 0;
        for (u32 r = 0; r < 8; ++r) seen |= 1u << (((r >> 1) * (pair_pitch / 4) + (r & 1) * (p_in / 4)) % 8);
        if (seen == 0xFF) break;
        if (pair_pitch > p_in + row_len + 64) {
            // no skew separates the 8 row lanes for this p_in: one bulk copy per row, odd pitch in 16-byte units
            rows_per_copy = 1;
            pair_pitch = row_len;
            if ((pair_pitch / 4) % 2 == 0) pair_pitch += 4;
            break;
        }
    }

    // Tap table [group][slice lane][iteration][32]: 16 floats for half A (4 samples x 4 outputs), 16 for half B.
    // Each slice lane's sub-table is followed by 8 floats of padding, which skews the four slice lanes of a
    // warp onto different 16-byte bank groups (sub-table stride/4 = 2 mod 8).
    const u64 rec = halves * 4 * kH;                     // 16 floats per half per (iteration, slice lane)
    u64 lane_stride = iters * rec + 8;                   // floats between the sub-tables of one group
    for (;; lane_stride += 4) {                          // the 4 slice lanes must start in 4 different bank groups
        u32 seen = 0;
        for (u32 ks = 0; ks < kKS; ++ks) seen |= 1u << ((ks * (lane_stride / 4)) % 8);
        if (__builtin_popcount(seen) == static_cast<int>(kKS)) break;
    }
    const u64 group_stride = kKS * lane_stride;
    u64 plane_pitch = p_out + 4;                         // partial-sum planes [slice][row][plane_pitch]
    if ((plane_pitch / 4) % 2 == 0) plane_pitch += 4;    // odd in 16-byte units: conflict-free float4 stores
    const u64 rows_floats = static_cast<u64>(kQT / rows_per_copy) * pair_pitch;
    // warp-specialised kernel: barriers + taps + 2 row stages (each with its halo row) + partial-sum planes
    const u64 stage_floats = rows_floats + span;
    const u64 planes_floats = kKS * static_cast<u64>(kQT) * plane_pitch;
    const u64 smem = 128 + (groups * group_stride + 2 * stage_floats + planes_floats) * 4;
    if (smem > kSmemOneCta) return false;

    tile_taps.assign(groups * group_stride, 0.f);
    auto tap_at = [&](long long idx) -> float {
        return idx >= 0 && static_cast<u64>(idx) <= off2 ? taps[static_cast<size_t>(idx)] : 0.f;
    };
    for (u32 g = 0; g < groups; ++g) {
        const u64 k0 = static_cast<u64>(kR) * g;
        for (u64 it = 0; it < iters; ++it) {
            for (u32 ks = 0; ks < kKS; ++ks) {
                float *dst = &tile_taps[g * group_stride + ks * lane_stride + it * rec];
                for (u32 uu = 0; uu < 4; ++uu) {
                    const u64 u = (it * kKS + ks) * 4 + uu;             // sample index relative to w0
                    const long long x = static_cast<long long>(group_xs[g] + u);
                    for (u32 r = 0; r < kH; ++r) {
                        // half A sees sample u as its tap u; half B (window starts `shift` later) likewise
                        dst[uu * kH + r] = u < ua ? tap_at(x * l - static_cast<long long>((k0 + r) * m)) : 0.f;
                        if (halves == 2)
                            dst[16 + uu * kH + r] =
                                u >= shift ? tap_at(x * l - static_cast<long long>((k0 + kH + r) * m)) : 0.f;
                    }
                }
            }
        }
    }
    tp.l = l;
    tp.m = m;
    tp.groups = groups;
    tp.p_out = static_cast<u32>(p_out);
    tp.p_in = static_cast<u32>(p_in);
    tp.usteps = static_cast<u32>(span);
    tp.half_taps = static_cast<u32>(ua);
    tp.shift = static_cast<u32>(shift);
    tp.iters = static_cast<u32>(iters);
    tp.row_len = static_cast<u32>(row_len);
    tp.pair_pitch = static_cast<u32>(pair_pitch);
    tp.rows_per_copy = rows_per_copy;
    tp.rows_floats = static_cast<u32>(rows_floats);
    tp.plane_pitch = static_cast<u32>(plane_pitch);
    tp.halves = halves;
    tp.qt = kQT;
    {
        const u32 vpr = static_cast<u32>(p_out / 4), nvec = kQT * vpr;
        tp.vec_magic = (65536u + vpr - 1) / vpr;
        for (u32 v = 0; v < nvec; ++v)
            if (((v * tp.vec_magic) >> 16) != v / vpr) return false;   // cannot happen for vpr <= 26, checked anyway
    }
    tp.slice_stride = static_cast<u32>(lane_stride);
    tp.group_stride = static_cast<u32>(group_stride);
    tp.smem_bytes = static_cast<u32>(smem);
    tp.ctas_per_sm = 1;
    tp.stage_floats = static_cast<u32>(stage_floats);
    tp.off2 = off2;
    return true;
}

bool make_tile_plan(u32 l, u32 m, const std::vector<float> &taps, TilePlan &tp, std::vector<float> &tile_taps,
                    std::vector<u32> &group_xs) {
    // 8 outputs per group when it fits shared memory, else 4 (96 kHz input, the slow profile)
    if (try_tile_plan(2, l, m, taps, tp, tile_taps, group_xs)) return true;
    return try_tile_plan(1, l, m, taps, tp, tile_taps, group_xs);
}

}  // namespace aptb200
