// ck_monomerize.cuh -- `monomerize` on the device (SURVEY 8f row 4): for every record the end index of its last monomer.
//
// What it replaces in the reference (per record):
//   Monomerizer::first_monomer_end_index            lib/src/monomerize.rs:50-99
//   Monomerizer::last_monomer_end_index             lib/src/monomerize.rs:100-125
//   Monomerizer::last_monomer_end_index_sensitive   lib/src/monomerize.rs:127-141
//
// One warp per record, bytes as they are (library semantics).  first(): the seed is the last seed_len bytes; the 32 lanes
// test 128 candidate start positions of the text seq[.. n - seed_len] at a time (four per lane) (bio's ShiftAnd::find_all reports every
// occurrence, overlapping ones included, by increasing start), the occurrences of a round are taken in position order and
// the Hamming distance of prefix seq[.. occ + seed_len] against the suffix of the same length is counted by the whole
// warp (four bytes per lane and step); the first occurrence within the allowed distance ends the search.  The sensitive pass runs the same code over a
// view that reads the monomer backwards through bio's complement table (no reverse complement is materialised).
#pragma once
#include "ck_device.cuh"
#include "ck_kernels.cuh"

namespace ck {

#ifndef CK_MONO_NONE
#define CK_MONO_NONE 0xffffffffu
#endif

struct MonoArgs {
    const u8 *bytes; const u64 *offsets; const u32 *lens; u32 n_records;   // lens: optional normalised lengths (ck_dev_normalize)
    u32 seed_len;          // 1 .. 63
    u32 use_identity;      // 1: max distance = len - floor(len * identity) (f64, as the reference computes it)
    u64 overlap_dist;      // 0: otherwise
    double identity;
    u32 flags;             // bit0: sensitive (reverse-complement pass), bit1: first_monomer_end_index only
    u32 *out_end;          // CK_MONO_NONE = None
};

template <bool RC> struct MonoView {
    const u8 *s; u32 n;    // RC: position j reads comp[s[n - 1 - j]]
    __device__ __forceinline__ u32 at(u32 j) const { return RC ? (u32)s_tab.comp[s[n - 1u - j]] : (u32)s[j]; }
};

template <bool RC> __device__ u32 mono_first(const MonoArgs &a, MonoView<RC> v)
{
    const u32 s = a.seed_len, n = v.n, lane = lane_id();
    if (n <= s || n < 2 * s) return CK_MONO_NONE;          // no room for an occurrence in seq[.. n - s]
    const u32 limit = n - 2 * s + 1;                        // candidate starts 0 .. n - 2 s
    // the first K = min(seed_len, 4) bytes of the seed as one word: a candidate start must match it before the rest of the
    // seed is looked at (1 in 256 random positions passes instead of 1 in 4, so the divergent tail below is rare)
    const u32 K = min(s, 4u);
    const u32 kmask = K == 4 ? 0xffffffffu : (1u << (8 * K)) - 1u;
    u32 seedw = 0;
    for (u32 k = 0; k < K; k++) seedw |= v.at(n - s + k) << (8 * k);
    // 128 candidate starts per round, four consecutive ones per lane (seven independent byte loads)
    for (u32 base = 0; base < limit; base += 128) {
        const u32 p0 = base + 4 * lane;
        u32 hit = 0;
        if (p0 < limit) {
            u32 b[7];
#pragma unroll
            for (u32 k = 0; k < 7; k++) b[k] = p0 + k < n ? v.at(p0 + k) : 0u;
#pragma unroll
            for (u32 q = 0; q < 4; q++) {
                const u32 w = (b[q] | (b[q + 1] << 8) | (b[q + 2] << 16) | (b[q + 3] << 24)) & kmask;
                if (p0 + q < limit && w == seedw) hit |= 1u << q;
            }
        }
        for (u32 h = hit; h; h &= h - 1) {                  // the rest of the seed for the positions that passed
            const u32 q = (u32)__ffs(h) - 1u, p = p0 + q;
            bool match = true;
            for (u32 k = K; match && k < s; k++) match = v.at(p + k) == v.at(n - s + k);
            if (!match) hit &= ~(1u << q);
        }
        u32 lanes = __ballot_sync(CK_FULL, hit != 0);
        while (lanes) {                                     // occurrences in position order: by lane, then inside the lane
            const u32 l = (u32)__ffs(lanes) - 1u;
            lanes &= lanes - 1u;
            u32 hq = __shfl_sync(CK_FULL, hit, l);
            while (hq) {
                const u32 occ = base + 4 * l + (u32)__ffs(hq) - 1u;
                hq &= hq - 1u;
                const u32 m = occ + s;                      // overlap length
                u32 cnt = 0;
                for (u32 t = 4 * lane; t < m; t += 128) {   // four bytes per lane and step
#pragma unroll
                    for (u32 u = 0; u < 4; u++)
                        if (t + u < m) cnt += v.at(n - m + t + u) != v.at(t + u);
                }
                const u64 dist = __reduce_add_sync(CK_FULL, cnt);
                const u64 maxd = a.use_identity ? (u64)m - (u64)floor((double)m * a.identity) : a.overlap_dist;
                if (dist <= maxd) return n - m;
            }
        }
    }
    return CK_MONO_NONE;
}

__global__ void __launch_bounds__(256) k_monomerize(MonoArgs a)
{
    stab_load();
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (u32 rec = gw; rec < a.n_records; rec += nw) {
        const u64 off = a.offsets[rec];
        const u32 n = a.lens ? a.lens[rec] : (u32)(a.offsets[rec + 1] - off);
        const u8 *seq = a.bytes + off;
        u32 idx = mono_first<false>(a, MonoView<false>{seq, n});
        if (!(a.flags & 2u)) {
            while (idx != CK_MONO_NONE) {                   // lib/src/monomerize.rs:103-114
                const u32 nxt = mono_first<false>(a, MonoView<false>{seq, idx});
                if (nxt == CK_MONO_NONE) break;
                idx = nxt;
            }
            if (a.flags & 1u) {                             // lib/src/monomerize.rs:127-141: Some(k) -> M - (M - k) = k
                const u32 M = idx == CK_MONO_NONE ? n : idx;
                const u32 k = mono_first<true>(a, MonoView<true>{seq, M});
                if (k != CK_MONO_NONE) idx = k;
            }
        }
        if (lane_id() == 0) a.out_end[rec] = idx;
    }
}

// ---------------------------------------------------------------------------------------------
// The consumer closure of `circkit monomerize` (src/monomerize.rs:102-143) on the device, for the batch API
// (ck_mono_submit): k_mono_select decides per record what is written and how long it is, the compaction of ck_lib.cu
// (the one uniq's survivors use) lays the written records out, k_mono_gather writes full_seq[.. monomer_len] of each.
//
// full_seq (seq_io 0.3.2 Record::full_seq) is the record without its '\n's and without a '\r' that ends a line or the
// record.  k_monomerize's index counts normalised symbols but is applied to full_seq, which keeps the ' ' / '\t' that
// normalisation drops: that is what the reference does.
struct MonoSelectArgs {
    const u8 *raw; const u64 *offsets; const u32 *lens;   // lens: normalised lengths (CK_F_NORMALIZE), else nullptr
    u32 n_records; u32 normalize; u32 keep_all; u32 seed_len;
    u64 min_length, max_length, min_overlap;                // max_length: ~0 = unset; min_overlap: 0 = unset
    double min_overlap_percent;                             // NaN = unset
    u32 *end;              // in: k_monomerize's answer; out: the worker's result (CK_MONO_NONE = None)
    u32 *full_len, *monomer_len; u8 *written;
};

// the 16 record bytes src[p .. p + 16) (bytes at or past len read as anything) from aligned 16-byte words
__device__ __forceinline__ uint4 mono_load16(const u8 *src, u32 p, u32 len)
{
    const u8 *b = src + p;
    const u32 sh = (u32)((size_t)b & 15u);
    return prep_load16(reinterpret_cast<const uint4 *>(b - sh), sh, sh != 0 && p + 16u - sh < len, p < len);
}
__device__ __forceinline__ u32 mono_mask4(u32 w, u32 c)    // bit k: byte k of w equals c
{
    return (((__vcmpeq4(w, c) & 0x01010101u) * 0x01020408u) >> 24) & 15u;
}
// bit k: byte p + k exists and is not part of full_seq.  Every lane of the warp calls it (lane l + 1 holds the byte after
// lane l's sixteen; lane 31 reads it).
__device__ __forceinline__ u32 mono_fullseq_drop(uint4 q, const u8 *src, u32 p, u32 len)
{
    const u32 valid = p >= len ? 0u : len - p >= 16 ? 0xffffu : (1u << (len - p)) - 1u;
    const u32 nl = (mono_mask4(q.x, 0x0a0a0a0au) | mono_mask4(q.y, 0x0a0a0a0au) << 4 | mono_mask4(q.z, 0x0a0a0a0au) << 8
                    | mono_mask4(q.w, 0x0a0a0a0au) << 12) & valid;
    const u32 cr = (mono_mask4(q.x, 0x0d0d0d0du) | mono_mask4(q.y, 0x0d0d0d0du) << 4 | mono_mask4(q.z, 0x0d0d0d0du) << 8
                    | mono_mask4(q.w, 0x0d0d0d0du) << 12) & valid;
    u32 nxt = __shfl_down_sync(CK_FULL, nl & 1u, 1);
    if (lane_id() == 31) nxt = p + 16 < len && src[p + 16] == '\n';
    const u32 last = p < len && len - p <= 16 ? 1u << (len - p - 1) : 0u;
    return nl | (cr & ((nl >> 1) | (nxt << 15) | last));
}

__global__ void __launch_bounds__(256) k_mono_select(MonoSelectArgs a)
{
    const u32 lane = lane_id();
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (u32 rec = gw; rec < a.n_records; rec += nw) {
        const u64 off = a.offsets[rec];
        const u32 rawlen = (u32)(a.offsets[rec + 1] - off);
        u32 full = rawlen;                                  // library semantics: the bytes as they are
        if (a.normalize) {
            const u8 *src = a.raw + off;
            u32 drop = 0;
            for (u32 base = 0; base < rawlen; base += 512) {
                const u32 p = base + 16 * lane;
                drop += __popc(mono_fullseq_drop(mono_load16(src, p, rawlen), src, p, rawlen));
            }
            full = rawlen - __reduce_add_sync(CK_FULL, drop);
        }
        if (lane == 0) {
            const u32 n = a.lens ? a.lens[rec] : rawlen;
            u32 idx = a.end[rec];
            if (n < a.seed_len || n < a.min_length) idx = CK_MONO_NONE;     // worker closure, src/monomerize.rs:92-96
            bool ok = idx != CK_MONO_NONE;
            if (ok) {                                       // consumer closure, :107-135
                const long long diff = (long long)full - (long long)idx;
                if (idx < a.min_length || idx > a.max_length) ok = false;
                if (a.min_overlap && (diff < 0 || (u64)diff < a.min_overlap)) ok = false;
                if (__ddiv_rn((double)diff, (double)idx) < a.min_overlap_percent) ok = false;   // NaN: false
            }
            a.end[rec] = idx;
            a.full_len[rec] = full;
            a.monomer_len[rec] = ok ? min(idx, full) : full;
            a.written[rec] = ok || a.keep_all;
        }
    }
}

#define CK_MONO_STAGE 544u     // 15 carried bytes + 512 + the rounding of the last store, per warp

// One warp per written record k: full_seq[.. monomer_len] (CK_F_NORMALIZE; else the raw bytes) to compact + compact_off[k].
// The warp reads 512 raw bytes per step (16 per lane), packs the kept ones into a per-warp stage through a warp prefix sum
// and stores the stage as whole 16-byte vectors (compact_off is 16-byte aligned; the last vector may run into the record's
// 16-byte rounding); it stops reading once monomer_len bytes are out.
__global__ void __launch_bounds__(256) k_mono_gather(const u8 *raw, const u64 *offsets, const u32 *sel, const u32 *n_sel,
                                                     const u32 *monomer_len, const u64 *compact_off, u32 normalize, u8 *compact)
{
    __shared__ __align__(16) u8 stage_all[8][CK_MONO_STAGE];
    u8 *stage = stage_all[threadIdx.x >> 5];
    const u32 lane = lane_id();
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const u32 ns = *n_sel;
    for (u32 k = gw; k < ns; k += nw) {
        const u32 rec = sel[k], want = monomer_len[rec];
        const u64 off = offsets[rec];
        const u32 rawlen = (u32)(offsets[rec + 1] - off);
        const u8 *src = raw + off;
        u8 *dst = compact + compact_off[k];
        u32 done = 0, carry = 0;                            // bytes staged so far / of them still in the stage
        for (u32 base = 0; done < want && base < rawlen; base += 512) {
            const u32 p = base + 16 * lane;
            const uint4 q = mono_load16(src, p, rawlen);
            u32 keep = p >= rawlen ? 0u : rawlen - p >= 16 ? 0xffffu : (1u << (rawlen - p)) - 1u;
            if (normalize) keep &= ~mono_fullseq_drop(q, src, p, rawlen);
            const u32 cnt = __popc(keep);
            u32 incl = cnt;
#pragma unroll
            for (u32 d = 1; d < 32; d <<= 1) {
                const u32 t = __shfl_up_sync(CK_FULL, incl, d);
                if (lane >= d) incl += t;
            }
            const u32 tot = __shfl_sync(CK_FULL, incl, 31);
            const u32 room = want - done;
            u32 j = incl - cnt;
            for (u32 m = keep; m && j < room; m &= m - 1u) stage[carry + j++] = (u8)prep_byte(q, __ffs(m) - 1);
            const u32 got = min(tot, room);
            __syncwarp();
            const u32 fill = carry + got;
            const bool last = done + got >= want;
            const u32 vecs = last ? (fill + 15) / 16 : fill / 16;
            u8 *out = dst + (done - carry);                 // done - carry: bytes stored so far, a multiple of 16
            for (u32 c = lane; c < vecs; c += 32) reinterpret_cast<uint4 *>(out)[c] = reinterpret_cast<const uint4 *>(stage)[c];
            __syncwarp();
            const u32 rest = last ? 0u : fill - 16 * vecs;
            if (lane < rest) stage[lane] = stage[16 * vecs + lane];
            __syncwarp();
            carry = rest;
            done += got;
        }
    }
}

}  // namespace ck
