// rtfs_snapshot.cu — the device side of saving a progressive frame and resuming it (rt_frame_save, rt_frame_resume,
// rt_multi_frame_resume; the entry points are in rtfs_frame.cu, the format in include/rtfs_b200.h).
// Save: snapshot_pack_kernel reads the frame's totals on the first device and writes the pixel sections in file order into
// a staging buffer, the flags packed 32 to a word with __ballot_sync, summing the checksum terms of what it wrote.
// Resume: snapshot_unpack_kernel writes the sections back into the first part's sums and Q and the frame's flags, checks
// every pixel against the frame's rules, and recomputes the checksum and the frame's counts for the host to compare with
// the header.  The checksum is a sum of per-word terms, so integer atomics give one fixed value whatever the order.
#include "rtfs_device.h"

#include <cstring>

namespace rtfs {
namespace {

constexpr int kSnapshotThreads = 256; // eight warps: eight groups of 64 pixels a block

__device__ __forceinline__ void tally_add(unsigned long long *slot, unsigned long long v) {
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(slot, v);
}

// Warp g packs pixels [64 g, 64 g + 64): lane l the pixels 64 g + l and 64 g + 32 + l (their sums and Q), and the two
// ballots are flag word g.
__global__ void __launch_bounds__(kSnapshotThreads) snapshot_pack_kernel(const int4 *stats, const unsigned long long *sq, const uint8_t *flags,
                                                                         const SnapshotSections s, unsigned long long *checksum) {
    const size_t group = (size_t(blockIdx.x) * kSnapshotThreads + threadIdx.x) / 32;
    const unsigned lane = threadIdx.x & 31;
    if (group >= snapshot_flag_words(s.n_pixels)) return; // (whole warps)
    const size_t w_sq = 2 * s.n_pixels, w_flags = w_sq + (s.noise ? s.n_pixels : 0);
    unsigned long long sum = 0;
    uint32_t half[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const size_t p = 64 * group + 32 * h + lane;
        bool on = false;
        if (p < s.n_pixels) {
            const ulonglong2 v = reinterpret_cast<const ulonglong2 *>(stats)[p];
            reinterpret_cast<ulonglong2 *>(s.words)[p] = v;
            sum += snapshot_mix(s.first_word + 2 * p, v.x) + snapshot_mix(s.first_word + 2 * p + 1, v.y);
            if (s.noise) {
                const unsigned long long q = sq[p];
                s.words[w_sq + p] = q;
                sum += snapshot_mix(s.first_word + w_sq + p, q);
            }
            on = flags[p] != 0;
        }
        half[h] = __ballot_sync(0xffffffffu, on);
    }
    if (lane == 0) {
        const unsigned long long w = (unsigned long long)half[0] | ((unsigned long long)half[1] << 32);
        s.words[w_flags + group] = w;
        sum += snapshot_mix(s.first_word + w_flags + group, w);
    }
    tally_add(checksum, sum);
}

// The inverse of snapshot_pack_kernel, with the checks: a pixel breaks a rule if a channel sum lies outside [0, 255 n], Q
// outside [0, 3 255^2 n], or its count n is not samples_done (still sampled) or n_probe or a checkpoint <= samples_done
// (stopped); a flag past the last pixel breaks one too.
__global__ void __launch_bounds__(kSnapshotThreads) snapshot_unpack_kernel(const SnapshotSections s, const SnapshotRules r, int4 *stats,
                                                                           unsigned long long *sq, uint8_t *flags, SnapshotTally *tally) {
    const size_t group = (size_t(blockIdx.x) * kSnapshotThreads + threadIdx.x) / 32;
    const unsigned lane = threadIdx.x & 31;
    if (group >= snapshot_flag_words(s.n_pixels)) return;
    const size_t w_sq = 2 * s.n_pixels, w_flags = w_sq + (s.noise ? s.n_pixels : 0);
    const unsigned long long fw = s.words[w_flags + group];
    unsigned long long sum = lane == 0 ? snapshot_mix(s.first_word + w_flags + group, fw) : 0ull;
    unsigned long long counts = 0, active = 0, flagged = 0, bad = ~0ull;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const size_t p = 64 * group + 32 * h + lane;
        const bool on = (fw >> (32 * h + lane)) & 1ull;
        if (p >= s.n_pixels) {
            if (on) bad = min(bad, (unsigned long long)p);
            continue;
        }
        const ulonglong2 v = reinterpret_cast<const ulonglong2 *>(s.words)[p];
        sum += snapshot_mix(s.first_word + 2 * p, v.x) + snapshot_mix(s.first_word + 2 * p + 1, v.y);
        int4 px;
        std::memcpy(&px, &v, sizeof px);
        const long long n = px.w, top = 255ll * n;
        bool ok = n >= 0 && px.x >= 0 && px.y >= 0 && px.z >= 0 && px.x <= top && px.y <= top && px.z <= top;
        if (on) ok = ok && n == r.samples_done;
        else
            ok = ok && (n == r.n_probe || (r.conv_interval > 0 && n >= r.conv_min && n <= r.samples_done && (n - r.conv_min) % r.conv_interval == 0));
        if (s.noise) {
            const unsigned long long q = s.words[w_sq + p];
            sum += snapshot_mix(s.first_word + w_sq + p, q);
            ok = ok && n >= 0 && q <= 3ull * 255ull * 255ull * (unsigned long long)n;
            sq[p] = q;
        }
        stats[p] = px;
        flags[p] = on ? 1 : 0;
        counts += (unsigned long long)(unsigned)px.w;
        active += on ? 1 : 0;
        flagged += (on || n > r.n_probe) ? 1 : 0;
        if (!ok) bad = min(bad, (unsigned long long)p);
    }
    tally_add(&tally->checksum, sum);
    tally_add(&tally->counts, counts);
    tally_add(&tally->active, active);
    tally_add(&tally->flagged, flagged);
    for (int off = 16; off > 0; off >>= 1) bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, off));
    if (lane == 0 && bad != ~0ull) atomicMin(&tally->first_bad, bad);
}

unsigned snapshot_blocks(size_t n_pixels) { return unsigned((snapshot_flag_words(n_pixels) + kSnapshotThreads / 32 - 1) / (kSnapshotThreads / 32)); }

// the fingerprint's accumulator: every value is one 64-bit word, folded in order
struct Fingerprint {
    uint64_t h = 0x5254465346505254ull, i = 0;
    void word(uint64_t w) { h = snapshot_mix(i++, h ^ w); }
    void f64(double d) {
        uint64_t w;
        std::memcpy(&w, &d, sizeof w);
        word(w);
    }
    void bytes(const uint8_t *b, size_t n) {
        for (size_t k = 0; k < n; k += 8) {
            uint64_t w = 0;
            std::memcpy(&w, b + k, std::min<size_t>(8, n - k));
            word(w);
        }
    }
};

} // namespace

uint64_t snapshot_checksum(const void *bytes, size_t n, uint64_t first_word) {
    const auto *b = static_cast<const uint8_t *>(bytes);
    uint64_t sum = 0;
    for (size_t k = 0; k < n / 8; ++k) {
        uint64_t w;
        std::memcpy(&w, b + 8 * k, sizeof w);
        sum += snapshot_mix(first_word + k, w);
    }
    return sum;
}

uint64_t scene_fingerprint(const RtScene *scene) {
    Fingerprint f;
    f.word(scene->objects.size());
    for (const RtHittable &o : scene->objects) {
        f.word(uint64_t(uint32_t(o.shape)) | uint64_t(uint32_t(o.style)) << 32);
        for (double v : o.p) f.f64(v);
        for (double v : o.n) f.f64(v);
        for (double v : {o.radius, o.albedo, o.fuzz, o.ior, o.prob}) f.f64(v);
        f.word(uint64_t(uint32_t(o.texture)) | uint64_t(o.colour[0]) << 32 | uint64_t(o.colour[1]) << 40 | uint64_t(o.colour[2]) << 48);
    }
    f.word(scene->textures.size());
    for (size_t t = 0; t < scene->textures.size(); ++t) {
        const RtTexture &x = scene->textures[t];
        f.word(uint64_t(uint32_t(x.kind)) | uint64_t(x.colour[0]) << 32 | uint64_t(x.colour[1]) << 40 | uint64_t(x.colour[2]) << 48);
        f.word(uint64_t(uint32_t(x.width)) | uint64_t(uint32_t(x.height)) << 32);
        f.word(uint64_t(uint32_t(x.even)) | uint64_t(uint32_t(x.odd)) << 32);
        for (double v : {x.grid_size, x.map_centre[0], x.map_centre[1], x.map_centre[2], x.map_radius}) f.f64(v);
        if (x.kind == RT_TEX_IMAGE) f.bytes(scene->texture_pixels[t].data(), scene->texture_pixels[t].size());
    }
    return f.h;
}

int launch_snapshot_pack(const int32_t *stats, const unsigned long long *sq, const uint8_t *flags, const SnapshotSections &s,
                         unsigned long long *checksum, cudaStream_t st) {
    if (!s.n_pixels) return RT_OK;
    snapshot_pack_kernel<<<snapshot_blocks(s.n_pixels), kSnapshotThreads, 0, st>>>(reinterpret_cast<const int4 *>(stats), sq, flags, s, checksum);
    RT_CUDA(cudaGetLastError());
    return RT_OK;
}

int launch_snapshot_unpack(const SnapshotSections &s, const SnapshotRules &rules, int32_t *stats, unsigned long long *sq, uint8_t *flags,
                           SnapshotTally *tally, cudaStream_t st) {
    if (!s.n_pixels) return RT_OK;
    snapshot_unpack_kernel<<<snapshot_blocks(s.n_pixels), kSnapshotThreads, 0, st>>>(s, rules, reinterpret_cast<int4 *>(stats), sq, flags, tally);
    RT_CUDA(cudaGetLastError());
    return RT_OK;
}

} // namespace rtfs
