// Host-side geometry and tap stream of the uniform-tap polyphase kernel (kernels_ut.cuh).
#include <algorithm>
#include <cstdlib>

#include "launch.hpp"

namespace aptb200 {

namespace {
constexpr u32 kSmemBudget = 227 * 1024;
constexpr u32 kInflightBytes = 40 * 1024;   // keep about this much of the signal in flight per SM (latency x HBM share)
}  // namespace

bool make_ut_plan(u32 l, u32 m, const std::vector<float> &taps, UtPlan &up, std::vector<float> &stream) {
    if (l < 2 || m == 0 || taps.empty() || getenv("APTB200_NO_UNIFORM_TAPS")) return false;
    const u32 np = (l + 1) / 2;
    if (l != kUtL) return false;                            // the kernel is instantiated for L = 13
    const u64 off2 = 2 * ((static_cast<u64>(taps.size()) - 1) / 2);
    auto fx = [&](u64 r) { return (r * m + l - 1) / l; };   // first / last sample (relative to the row) output r touches
    auto lx = [&](u64 r) { return (r * m + off2) / l; };
    u32 cs[8] = {0}, ce[8] = {0};
    for (u32 p = 0; p < np; ++p) {
        const u64 hi = 2 * p + 1 < l ? std::max(lx(2 * p), lx(2 * p + 1)) : lx(2 * p);
        cs[p] = static_cast<u32>(fx(2 * p) / kUtChunk);
        ce[p] = static_cast<u32>(hi / kUtChunk + 1);
        if (p && (cs[p] < cs[p - 1] || ce[p] < ce[p - 1])) return false;
    }
    // two roles share a block: pairs [0, npa) and [npa, np); within a role every pair must have started before
    // the role's first pair ends (ramp-up / steady / ramp-down structure of the kernel's loop)
    const u32 npa = (np + 1) / 2, npb = np - npa;
    if (cs[0] != 0 || npb == 0 || cs[npa - 1] > ce[0] || cs[np - 1] > ce[npa]) return false;
    const u32 chunks = ce[np - 1];
    if (chunks > 4096) return false;

    // tap stream in consumption order, role by role: ramp-up segments, steady, ramp-down; per (chunk, active
    // pair) 2*CH floats {T[CH*c][2p], T[CH*c][2p+1], T[CH*c+1][2p], ... T[CH*c+CH-1][2p+1]},  T[u][r] = h[u*l - r*m]
    auto tap = [&](u64 u, u32 r) -> float {
        if (r >= l) return 0.f;
        const long long idx = static_cast<long long>(u * l) - static_cast<long long>(static_cast<u64>(r) * m);
        return idx >= 0 && static_cast<u64>(idx) <= off2 ? taps[static_cast<size_t>(idx)] : 0.f;
    };
    stream.clear();
    auto emit = [&](u32 c0, u32 c1, u32 p0, u32 p1) {
        for (u32 c = c0; c < c1; ++c)
            for (u32 p = p0; p < p1; ++p)
                for (u32 uu = 0; uu < kUtChunk; ++uu) {
                    stream.push_back(tap(static_cast<u64>(kUtChunk) * c + uu, 2 * p));
                    stream.push_back(tap(static_cast<u64>(kUtChunk) * c + uu, 2 * p + 1));
                }
    };
    auto emit_role = [&](u32 pb, u32 npr) {
        for (u32 a = 1; a < npr; ++a) emit(cs[pb + a - 1], cs[pb + a], pb, pb + a);
        emit(cs[pb + npr - 1], ce[pb], pb, pb + npr);
        for (u32 a = 1; a < npr; ++a) emit(ce[pb + a - 1], ce[pb + a], pb + a, pb + npr);
    };
    emit_role(0, npa);
    const u32 stream_b = static_cast<u32>(stream.size() / 4);
    emit_role(npa, npb);
    const u32 nvec = static_cast<u32>(stream.size() / 4);
    if (nvec > kUtMaxVecLarge) return false;

    const u32 halo_u0 = static_cast<u32>(fx(l - 1));
    const u32 halo_n = static_cast<u32>(lx(l - 1) - fx(l - 1) + 1);
    const u32 back = (m > halo_u0 ? (m - halo_u0 + 3) / 4 * 4 : 0);
    const u32 header = (1024 + halo_n * 4 + 127) / 128 * 128;
    if (header > 16 * 1024) return false;
    bool ok = false;
    // rows per thread: 2 measured best (48 kHz: 71 us against 76 for q = 4, which leaves room for only 12 warps;
    // 96 kHz: 142 us against 181 for q = 1, whose one uniform load per FFMA2 saturates the uniform-load port);
    // q = 1 only when two rows per thread do not fit shared memory (192 kHz)
    for (u32 q : {2u, 1u}) {
        const u32 rb = 32 * q;
        const u64 slot_floats = (static_cast<u64>(back) + static_cast<u64>(rb - 1) * m + static_cast<u64>(kUtChunk) * chunks + 3) / 4 * 4;
        const u64 slot_stride = slot_floats + 2 * rb + 4;          // + the exchange words of the two roles
        const u64 slot_bytes = slot_stride * 4;
        if (static_cast<u64>(rb) * l > slot_floats) continue;      // the block's outputs are transposed through its slot
        const u32 nslot = static_cast<u32>(std::min<u64>(kUtMaxSlots, (kSmemBudget - header) / slot_bytes));
        const u32 spare = static_cast<u32>(std::max<u64>(2, (kInflightBytes + slot_bytes - 1) / slot_bytes));
        if (nslot < spare + 3) continue;                           // at least 3 blocks (6 warps) in compute
        const u32 warps = std::min<u32>(24, 2 * (nslot - spare));   // two warps per block in compute
        up.q = q;
        up.rb = rb;
        up.slot_floats = static_cast<u32>(slot_floats);
        up.warps = warps;
        up.nslot = std::min(nslot, warps / 2 + spare + 1);
        up.slot_stride = static_cast<u32>(slot_stride);
        up.header_bytes = header;
        up.smem_bytes = header + up.nslot * static_cast<u32>(slot_bytes);
        ok = true;
        break;
    }
    if (!ok) return false;
    up.l = l;
    up.m = m;
    up.np = np;
    up.vec = m % 4 == 0 ? 4 : m % 2 == 0 ? 2 : 1;
    up.back = back;
    up.chunks = chunks;
    up.nvec = nvec;
    up.stream_b = stream_b;
    up.halo_u0 = halo_u0;
    up.halo_n = halo_n;
    up.off2 = off2;
    for (u32 p = 0; p < 8; ++p) {
        up.cs[p] = cs[p];
        up.ce[p] = ce[p];
    }
    return true;
}

}  // namespace aptb200
