// ck_fasta.cuh -- FASTA text batches on the device (ck_fasta_submit / ck_fasta_wait): the record split of seq_io 0.3.2's
// fasta::Reader and the output framing of the CLI ('>' head '\n' body '\n', src/canonicalize.rs:33-37, src/uniq.rs:50-61,
// src/monomerize.rs:137-140), so that the host hands over the decompressed text and writes what comes back.
//
// Split (in stream order):
//   k_fasta_count   one CTA per 4 KB tile of the text: how many records start in it (a '>' at 0 or after a '\n')
//   (exclusive scan of the tile counts: where each tile's starts go; the last entry is the record count)
//   k_fasta_starts  the start positions, in order; none is written at or past `cap` (max_batch_records)
//   k_fasta_ranges  one warp per record: head and seq ranges with one trailing '\r' trimmed each, seq lengths, the longest
//   (exclusive scan of the seq lengths = offsets of the record arena)
//   k_fasta_gather  one warp per record: the seq bytes into the arena the batch pipelines take (d_raw / d_off)
// Framing, once a pipeline has run:
//   k_fasta_frame_lens  framed length of every written record (head + body + 3); an exclusive scan places them
//   k_fasta_frame       one warp per written record: '>' head '\n' body '\n'
// Every position into the text is 64-bit.
#pragma once
#include "ck_device.cuh"
#include "ck_kernels.cuh"
#include "ck_monomerize.cuh"

namespace ck {

#define CK_FASTA_TILE 4096u     // text bytes per CTA of k_fasta_count / k_fasta_starts (256 threads x 16 bytes)

// bit k: byte p + k of the text starts a record.  p is a multiple of 16 and the buffer holds 16 readable bytes past nbytes.
__device__ __forceinline__ u32 fasta_start_mask(const u8 *text, u64 nbytes, u64 p)
{
    if (p >= nbytes) return 0;
    const uint4 q = *reinterpret_cast<const uint4 *>(text + p);
    const u32 gt = mono_mask4(q.x, 0x3e3e3e3eu) | mono_mask4(q.y, 0x3e3e3e3eu) << 4 | mono_mask4(q.z, 0x3e3e3e3eu) << 8
                   | mono_mask4(q.w, 0x3e3e3e3eu) << 12;
    const u32 nl = mono_mask4(q.x, 0x0a0a0a0au) | mono_mask4(q.y, 0x0a0a0a0au) << 4 | mono_mask4(q.z, 0x0a0a0a0au) << 8
                   | mono_mask4(q.w, 0x0a0a0a0au) << 12;
    const u32 prev = p == 0 ? 1u : (text[p - 1] == '\n' ? 1u : 0u);
    const u32 valid = nbytes - p >= 16 ? 0xffffu : (1u << (nbytes - p)) - 1u;
    return gt & ((nl << 1) | prev) & valid;
}

__global__ void __launch_bounds__(256) k_fasta_count(const u8 *text, u64 nbytes, u32 *tile_count)
{
    __shared__ u32 part[8];
    const u64 p = (u64)blockIdx.x * CK_FASTA_TILE + 16u * threadIdx.x;
    const u32 w = __reduce_add_sync(CK_FULL, (u32)__popc(fasta_start_mask(text, nbytes, p)));
    if (lane_id() == 0) part[threadIdx.x >> 5] = w;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 t = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) t += part[i];
        tile_count[blockIdx.x] = t;
    }
}

// tile_off: exclusive scan of k_fasta_count's counts.  Starts at ranks >= cap are counted but not stored.
__global__ void __launch_bounds__(256) k_fasta_starts(const u8 *text, u64 nbytes, const u32 *tile_off, u32 cap, u64 *starts)
{
    __shared__ u32 wsum[8];
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    const u64 p = (u64)blockIdx.x * CK_FASTA_TILE + 16u * threadIdx.x;
    const u32 m = fasta_start_mask(text, nbytes, p), c = (u32)__popc(m);
    u32 incl = c;
#pragma unroll
    for (u32 d = 1; d < 32; d <<= 1) {
        const u32 t = __shfl_up_sync(CK_FULL, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    u32 pos = tile_off[blockIdx.x] + incl - c;
    for (u32 k = 0; k < warp; k++) pos += wsum[k];
    for (u32 mm = m; mm; mm &= mm - 1u, pos++)
        if (pos < cap) starts[pos] = p + (u32)(__ffs(mm) - 1);
}

struct FastaRangeArgs {
    const u8 *text; u64 nbytes;
    const u64 *starts; const u32 *n_found; u32 cap;    // records found (may exceed cap: the submit then refuses the batch)
    u64 *head, *seq;        // 2 per record: [lo, hi) in the text
    u64 *seq_len;           // seq_hi - seq_lo
    u64 *longest;           // max of seq_len (zeroed by the caller)
};

// cli.Records' rules: record i spans starts[i] .. the '\n' before starts[i + 1] (the last one: the text's end, without one
// final '\n'); head = after '>' up to the first '\n' of the span (or the span's end), seq = the rest; one trailing '\r' of
// each is trimmed.
__global__ void __launch_bounds__(256) k_fasta_ranges(FastaRangeArgs a)
{
    const u32 lane = lane_id();
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const u32 nf = *a.n_found, n = min(nf, a.cap);
    const u64 last_end = a.text[a.nbytes - 1] == '\n' ? a.nbytes - 1 : a.nbytes;
    u64 longest = 0;
    for (u32 rec = gw; rec < n; rec += nw) {
        const u64 s = a.starts[rec];
        const u64 e = rec + 1 < n ? a.starts[rec + 1] - 1 : last_end;
        u64 first = e;                                      // the header's '\n'; e: none inside the span
        for (u64 b = s; b < e; b += 32) {
            const u64 p = b + lane;
            const u32 hit = __ballot_sync(CK_FULL, p < e && a.text[p] == '\n');
            if (hit) { first = b + (u32)(__ffs(hit) - 1); break; }
        }
        const bool has_seq = first < e;
        const u64 hlo = s + 1;
        u64 hhi = max(has_seq ? first : e, hlo);
        if (hhi > hlo && a.text[hhi - 1] == '\r') hhi--;
        const u64 slo = has_seq ? first + 1 : e;
        u64 shi = max(e, slo);
        if (shi > slo && a.text[shi - 1] == '\r') shi--;
        if (lane == 0) {
            a.head[2 * (u64)rec] = hlo; a.head[2 * (u64)rec + 1] = hhi;
            a.seq[2 * (u64)rec] = slo; a.seq[2 * (u64)rec + 1] = shi;
            a.seq_len[rec] = shi - slo;
        }
        longest = max(longest, shi - slo);
    }
    if (lane == 0 && longest) atomicMax(a.longest, longest);
}

// dst[0 .. len) = src[0 .. len) by one warp: single bytes up to dst's next 16-byte boundary, then aligned 16-byte stores of
// 16 source bytes each (two aligned loads and a funnel shift when the source is not aligned alike), then the tail.  The
// source buffer must hold 16 readable bytes past src + len.
__device__ __forceinline__ void warp_copy(u8 *dst, const u8 *src, u64 len)
{
    const u32 lane = lane_id();
    const u64 head = min(len, (u64)((16u - (u32)((size_t)dst & 15u)) & 15u));
    for (u64 b = lane; b < head; b += 32) dst[b] = src[b];
    const u8 *s2 = src + head;
    uint4 *d2 = reinterpret_cast<uint4 *>(dst + head);
    const u64 vecs = (len - head) >> 4;
    const u32 sh = (u32)((size_t)s2 & 15u);
    const uint4 *w = reinterpret_cast<const uint4 *>(s2 - sh);
    for (u64 c = lane; c < vecs; c += 32) d2[c] = prep_load16(w + c, sh, sh != 0);
    for (u64 b = head + (vecs << 4) + lane; b < len; b += 32) dst[b] = src[b];
}

__global__ void __launch_bounds__(256) k_fasta_gather(const u8 *text, const u64 *seq, const u64 *off, u32 n, u8 *raw)
{
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (u32 rec = gw; rec < n; rec += nw) {
        const u64 lo = seq[2 * (u64)rec], hi = seq[2 * (u64)rec + 1];
        warp_copy(raw + off[rec], text + lo, hi - lo);
    }
}

#define CK_FRAME_CANON 0u       // canonical bytes: the CK_F_ALIGNED_OUT arena, record i at out_byte(off[i], i), lens[i] bytes
#define CK_FRAME_RAW 1u         // record.seq(): the seq range of the text
#define CK_FRAME_COMPACT 2u     // monomers: written record k at arena + coff[k], lens[i] bytes

struct FastaFrameArgs {
    const u8 *text; const u64 *head; const u64 *seq;
    const u32 *sel; const u32 *n_sel; u32 n;            // the written records (increasing) and their number
    u32 body;                                           // CK_FRAME_*
    const u8 *arena; const u64 *off; const u32 *lens; const u64 *coff;
    u64 *flen; const u64 *fofs; u8 *frame;              // framed lengths (n + 1 entries), their exclusive scan, the output
};

__device__ __forceinline__ u64 frame_body(const FastaFrameArgs &a, u32 k, u32 rec, const u8 *&src)
{
    if (a.body == CK_FRAME_RAW) {
        src = a.text + a.seq[2 * (u64)rec];
        return a.seq[2 * (u64)rec + 1] - a.seq[2 * (u64)rec];
    }
    src = a.arena + (a.body == CK_FRAME_CANON ? out_byte(a.off[rec], rec) : a.coff[k]);
    return a.lens[rec];
}

__global__ void __launch_bounds__(256) k_fasta_frame_lens(FastaFrameArgs a)
{
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > a.n) return;
    u64 len = 0;
    if (k < *a.n_sel) {
        const u32 rec = a.sel[k];
        const u8 *src;
        len = a.head[2 * (u64)rec + 1] - a.head[2 * (u64)rec] + frame_body(a, k, rec, src) + 3;
    }
    a.flen[k] = len;
}

__global__ void __launch_bounds__(256) k_fasta_frame(FastaFrameArgs a)
{
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const u32 ns = *a.n_sel;
    for (u32 k = gw; k < ns; k += nw) {
        const u32 rec = a.sel[k];
        const u64 hlo = a.head[2 * (u64)rec], hl = a.head[2 * (u64)rec + 1] - hlo;
        const u8 *src;
        const u64 bl = frame_body(a, k, rec, src);
        u8 *dst = a.frame + a.fofs[k];
        if (lane_id() == 0) { dst[0] = '>'; dst[1 + hl] = '\n'; dst[2 + hl + bl] = '\n'; }
        warp_copy(dst + 1, a.text + hlo, hl);
        warp_copy(dst + 2 + hl, src, bl);
    }
}

}  // namespace ck
