// ck_deflate.cuh -- raw DEFLATE (RFC 1951) on the device for ck_deflate_submit / ck_deflate_wait: the `.gz` output of the CLI.
//
// One call compresses up to CK_DEFLATE_MAX_BYTES of input, optionally preceded by a dictionary (the <= 32 KiB that came
// before it), into non-final blocks that end byte-aligned with an empty stored block (00 00 ff ff, zlib's Z_SYNC_FLUSH), so
// that consecutive calls concatenate into one deflate stream.  The input is cut into segments of CKZ_SEG bytes; every
// segment becomes one block (dynamic Huffman, fixed Huffman or stored, whichever is smallest) that starts on a byte
// boundary, so the segments are coded independently and placed by a scan of their byte sizes.  Matches may reach 32 KiB
// back into earlier segments or the dictionary (the whole input is resident), so the ratio is that of one stream.
//
// In stream order, over buf = dict || input (N = dict + n positions, 64 zero bytes past the end):
//   k_defl_keys   hash of the 8 (then 4) bytes at every position; (CUB radix sort of (hash, position): stable, so equal
//                 hashes come out in position order)
//   k_defl_links  prev[p] = the previous position with the same hash (a hash chain per key, nearest first)
//   k_defl_match  one CTA per segment: byte histogram -> literal cost estimate; CRC-32 of the segment; for every position
//                 the longest match (3..258, never past the segment's end, nearest on ties) over <= CKZ_C8 candidates of the
//                 8-byte chain and, when that finds less than 8 bytes, <= CKZ_C4 of the 4-byte chain; a match is kept only
//                 when its estimated code length is below that of the literals it replaces (DNA literals cost ~2 bits, so
//                 the short, far matches a 3-byte hash finds in random sequence are dropped)
//   k_defl_parse  one CTA per segment, one lane parsing: greedy with zlib's one-step lazy evaluation over the match table
//                 (staged through shared memory); tokens and symbol frequencies
//   k_defl_huff   one CTA per segment: length-limited Huffman codes (15 bits; 7 for the code-length code), the dynamic
//                 block header, the exact byte size of each block type and the choice
//   k_defl_place  one CTA: exclusive scan of the segment sizes -> byte offsets and the total; CRC-32 of the whole input
//                 from the segments' CRCs by GF(2) shifts, continued from crc_in
//   k_defl_pack   one CTA per segment: a scan of the tokens' bit lengths, then every lane writes its run of tokens with
//                 funnel shifts; words wholly inside a lane's bit range are stored, shared edge words are OR-ed atomically
//                 into the zeroed output
#pragma once
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "ck_device.cuh"

namespace ck {

#define CKZ_SEG 65536u            // input bytes per segment (one block, one CTA)
#define CKZ_MAX_SEGS 1024u        // CK_DEFLATE_MAX_BYTES / CKZ_SEG
#define CKZ_WIN 32768u            // DEFLATE's window
#define CKZ_HBITS 24              // bits of the chain hashes (the radix sort sorts these only)
#define CKZ_C8 16u                // candidates walked on the 8-byte chain
#define CKZ_C4 4u                 // candidates walked on the 4-byte chain
#define CKZ_LAZY 32u              // matches shorter than this are checked against the next position's (zlib's lazy rule)
#define CKZ_NONE 0xffffffffu
#define CKZ_LL 288                // literal/length alphabet as the fixed code numbers it (286, 287 never occur)
#define CKZ_SYMS (CKZ_LL + 30)    // + the distance alphabet
#define CKZ_HDR_WORDS 160u        // a dynamic header is at most 3 + 14 + 57 + 316 * 14 bits
#define CKZ_PARSE_CHUNK 4096u
#define CKZ_STORED 0u
#define CKZ_FIXED 1u
#define CKZ_DYNAMIC 2u

struct DeflateArgs {
    const u8 *buf;                // dict || input, 64 zero bytes past the end
    u32 dict, n, nseg;
    const u32 *prev8, *prev4;     // hash chains over buf
    u32 *match;                   // n: len | dist << 16 (0: literal)
    u32 *tok;                     // n: segment s's tokens from s * CKZ_SEG; literal = byte << 16, match as `match`
    u32 *ntok;                    // nseg
    u32 *freq;                    // nseg * CKZ_SYMS
    u32 *seg_crc;                 // nseg: CRC register of the segment from 0 (no pre / post inversion)
    u32 *table;                   // nseg * CKZ_SYMS: reversed code | length << 16 of the chosen code
    u32 *hdr;                     // nseg * CKZ_HDR_WORDS: the block header's bits
    u32 *meta;                    // nseg * 4: header bits, block type, byte size
    u64 *off;                     // nseg: byte offset of the segment's output
    u32 *out;                     // zeroed, ck_deflate_bound(n) bytes rounded up to words
    u32 *result;                  // [0..1] output bytes, [2] CRC-32
    u32 crc_in;
};

// ---- CRC-32 (reflected 0xedb88320) in GF(2): register shifts by multiplication with x^(8 len) mod P ----------------------
__device__ __forceinline__ u32 crc_multmodp(u32 a, u32 b)     // a * b mod P, a != 0
{
    u32 m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}

// x^(8 nbytes) mod P: the operator that runs a CRC register over nbytes zero bytes
__device__ __forceinline__ u32 crc_x8n(u64 nbytes)
{
    u32 p = 1u << 31, sq = 1u << 30;                  // x^0, x^1
    for (int k = 0; k < 3; k++) sq = crc_multmodp(sq, sq);   // x^8
    while (nbytes) {
        if (nbytes & 1) p = crc_multmodp(sq, p);
        nbytes >>= 1;
        if (nbytes) sq = crc_multmodp(sq, sq);
    }
    return p;
}

// ---- symbols of lengths and distances (RFC 1951 3.2.5) ----------------------------------------------------------------
__device__ __forceinline__ u32 defl_lsym(u32 len, u32 &nb, u32 &extra)   // len 3..258 -> 257..285
{
    if (len == 258) { nb = 0; extra = 0; return 285; }
    const u32 v = len - 3;
    if (v < 8) { nb = 0; extra = 0; return 257 + v; }
    nb = 29 - __clz(v);                               // floor(log2 v) - 2
    extra = v & ((1u << nb) - 1);
    return 257 + 4 * nb + (v >> nb);                  // 265 + 4 (nb - 1) + ((v >> nb) - 4)
}

__device__ __forceinline__ u32 defl_dsym(u32 dist, u32 &nb, u32 &extra)  // dist 1..32768 -> 0..29
{
    const u32 v = dist - 1;
    if (v < 4) { nb = 0; extra = 0; return v; }
    const u32 lg = 31 - __clz(v);
    nb = lg - 1;
    extra = v & ((1u << nb) - 1);
    return 2 * lg + ((v >> nb) & 1);
}

__device__ __forceinline__ u32 defl_lext(u32 sym) { return sym >= 265 && sym < 285 ? (sym - 261) >> 2 : 0; }
__device__ __forceinline__ u32 defl_dext(u32 code) { return code >= 4 ? (code >> 1) - 1 : 0; }

// ---- k_defl_keys / k_defl_links: hash chains -----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_defl_keys(const u8 *buf, u32 total, u32 width, u32 *keys, u32 *vals)
{
    const u32 i = blockIdx.x * 256u + threadIdx.x;
    if (i >= total) return;
    u64 v = 0;
    for (u32 k = 0; k < width; k++) v |= (u64)buf[i + k] << (8 * k);
    const u64 mul = width == 8 ? 0x9e3779b97f4a7c15ull : 0xff51afd7ed558ccdull;
    keys[i] = (u32)((v * mul) >> (64 - CKZ_HBITS));
    vals[i] = i;
}

__global__ void __launch_bounds__(256) k_defl_links(const u32 *skeys, const u32 *svals, u32 total, u32 *prev)
{
    const u32 k = blockIdx.x * 256u + threadIdx.x;
    if (k >= total) return;
    prev[svals[k]] = k > 0 && skeys[k - 1] == skeys[k] ? svals[k - 1] : CKZ_NONE;
}

// ---- k_defl_match ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 defl_match_len(const u8 *buf, u32 c, u32 p, u32 maxlen, u32 best)
{
    if (best && best < maxlen && buf[c + best] != buf[p + best]) return 0;   // cannot beat `best`
    u32 k = 0;
    while (k < maxlen && buf[c + k] == buf[p + k]) k++;
    return k;
}

__global__ void __launch_bounds__(256) k_defl_match(DeflateArgs a)
{
    __shared__ u32 hist[256], tab[256];
    __shared__ float cost[256];
    typedef cub::BlockReduce<u32, 256> Reduce;
    __shared__ typename Reduce::TempStorage red;
    const u32 seg = blockIdx.x, t = threadIdx.x;
    const u32 lo = seg * CKZ_SEG, hi = min(lo + CKZ_SEG, a.n), len = hi - lo;
    const u8 *in = a.buf + a.dict;
    hist[t] = 0;
    {
        u32 c = t;
        for (int k = 0; k < 8; k++) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
        tab[t] = c;
    }
    __syncthreads();
    for (u32 p = lo + t; p < hi; p += 256) atomicAdd(&hist[in[p]], 1u);
    // CRC of this lane's run of the segment, shifted over the bytes that follow it in the segment
    const u32 run = (len + 255) / 256, ra = min(lo + t * run, hi), rb = min(ra + run, hi);
    u32 c = 0;
    for (u32 p = ra; p < rb; p++) c = tab[(c ^ in[p]) & 255] ^ (c >> 8);
    if (rb > ra && hi > rb) c = crc_multmodp(crc_x8n(hi - rb), c);
    const u32 x = Reduce(red).Reduce(c, [](u32 u, u32 v) { return u ^ v; });
    if (t == 0) a.seg_crc[seg] = x;
    __syncthreads();
    cost[t] = hist[t] ? fmaxf(__log2f((float)len / (float)hist[t]), 1.f) : 16.f;   // a Huffman code has >= 1 bit
    __syncthreads();
    for (u32 p = lo + t; p < hi; p += 256) {
        const u32 P = a.dict + p, maxlen = min(258u, hi - p), lim = P > CKZ_WIN ? P - CKZ_WIN : 0;
        u32 best = 0, bd = 0;
        if (maxlen >= 4) {
            u32 cand = a.prev8[P];
            for (u32 k = 0; k < CKZ_C8 && cand != CKZ_NONE && cand >= lim; k++) {
                const u32 l = defl_match_len(a.buf, cand, P, maxlen, best);
                if (l > best) { best = l; bd = P - cand; if (l == maxlen) break; }
                cand = a.prev8[cand];
            }
            if (best < 8) {
                cand = a.prev4[P];
                for (u32 k = 0; k < CKZ_C4 && cand != CKZ_NONE && cand >= lim; k++) {
                    const u32 l = defl_match_len(a.buf, cand, P, maxlen, best);
                    if (l > best) { best = l; bd = P - cand; if (l == maxlen) break; }
                    cand = a.prev4[cand];
                }
            }
        }
        u32 m = 0;
        if (best >= 3) {
            float lit = 0.f;
            for (u32 k = 0; k < best; k++) lit += cost[a.buf[P + k]];
            u32 lnb, ldx, dnb, ddx;
            defl_lsym(best, lnb, ldx);
            defl_dsym(bd, dnb, ddx);
            if (lit > (float)(13 + lnb + dnb)) m = best | bd << 16;   // ~7-bit length and ~6-bit distance symbols
        }
        a.match[p] = m;
    }
}

// ---- k_defl_parse ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_defl_parse(DeflateArgs a)
{
    __shared__ u32 sm[CKZ_PARSE_CHUNK + 1];
    __shared__ u8 sb[CKZ_PARSE_CHUNK];
    __shared__ u32 fq[CKZ_SYMS];
    __shared__ u32 s_p, s_nt;
    const u32 seg = blockIdx.x, t = threadIdx.x;
    const u32 lo = seg * CKZ_SEG, hi = min(lo + CKZ_SEG, a.n);
    const u8 *in = a.buf + a.dict;
    u32 *tok = a.tok + lo;
    for (u32 i = t; i < CKZ_SYMS; i += 128) fq[i] = 0;
    if (t == 0) { s_p = lo; s_nt = 0; }
    __syncthreads();
    for (;;) {
        const u32 base = s_p;
        if (base >= hi) break;
        const u32 cnt = min(CKZ_PARSE_CHUNK + 1, hi - base);
        for (u32 i = t; i < cnt; i += 128) {
            sm[i] = a.match[base + i];
            if (i < CKZ_PARSE_CHUNK) sb[i] = in[base + i];
        }
        __syncthreads();
        if (t == 0) {
            u32 p = base, nt = s_nt;
            const u32 end = min(base + CKZ_PARSE_CHUNK, hi);
            while (p < end) {
                const u32 m = sm[p - base], L = m & 0x1ff;
                if (L && !(L < CKZ_LAZY && p + 1 < hi && (sm[p + 1 - base] & 0x1ff) > L)) {
                    u32 nb, ex;
                    fq[defl_lsym(L, nb, ex)]++;
                    fq[CKZ_LL + defl_dsym(m >> 16, nb, ex)]++;
                    tok[nt++] = m;
                    p += L;
                } else {
                    const u32 b = sb[p - base];
                    fq[b]++;
                    tok[nt++] = b << 16;
                    p++;
                }
            }
            s_p = p; s_nt = nt;
        }
        __syncthreads();
    }
    if (t == 0) { a.ntok[seg] = s_nt; fq[256] = 1; }
    __syncthreads();
    for (u32 i = t; i < CKZ_SYMS; i += 128) a.freq[(u64)seg * CKZ_SYMS + i] = fq[i];
}

// ---- k_defl_huff ----------------------------------------------------------------------------------------------------------
struct HuffScratch {
    u32 sym[CKZ_LL], w[CKZ_LL], num[16], next[16], m;
};

// Code lengths <= maxbits of the n symbols with frequencies f (all threads call it).  Symbols are ranked by (frequency,
// index) in parallel; one lane builds the Huffman depths in place (Moffat and Katajainen), clamps them to maxbits and
// repairs the Kraft sum by moving leaves down (the rule of zlib / miniz), then hands the longest lengths to the rarest
// symbols.  No used symbol, or one: two codes of length 1, so every code is complete.
__device__ void defl_lengths(const u32 *f, int n, u32 maxbits, u32 *ln, HuffScratch &h)
{
    const int t = threadIdx.x;
    for (int s = t; s < n; s += blockDim.x) {
        ln[s] = 0;
        const u32 fs = f[s];
        if (fs) {
            u32 r = 0;
            for (int q = 0; q < n; q++) { const u32 fq = f[q]; r += fq && (fq < fs || (fq == fs && q < s)); }
            h.sym[r] = s;
        }
    }
    if (t == 0) { u32 m = 0; for (int s = 0; s < n; s++) m += f[s] != 0; h.m = m; }
    __syncthreads();
    if (t == 0) {
        const int m = (int)h.m;
        if (m <= 1) {
            const u32 s0 = m ? h.sym[0] : 0;
            ln[s0] = 1;
            ln[s0 == 0 ? 1 : 0] = 1;
        } else {
            u32 *A = h.w;
            for (int k = 0; k < m; k++) A[k] = f[h.sym[k]];
            // in-place minimum-redundancy code (A sorted ascending -> A[k] = depth of the k-th rarest symbol)
            A[0] += A[1];
            int root = 0, leaf = 2, next;
            for (next = 1; next < m - 1; next++) {
                if (leaf >= m || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = next; }
                else A[next] = A[leaf++];
                if (leaf >= m || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = next; }
                else A[next] += A[leaf++];
            }
            A[m - 2] = 0;
            for (next = m - 3; next >= 0; next--) A[next] = A[A[next]] + 1;
            int avbl = 1, used = 0, dpth = 0;
            root = m - 2; next = m - 1;
            while (avbl > 0) {
                while (root >= 0 && (int)A[root] == dpth) { used++; root--; }
                while (avbl > used) { A[next--] = dpth; avbl--; }
                avbl = 2 * used; dpth++; used = 0;
            }
            for (u32 l = 0; l < 16; l++) h.num[l] = 0;
            for (int k = 0; k < m; k++) h.num[min(A[k], maxbits)]++;
            u32 total = 0;
            for (u32 l = 1; l <= maxbits; l++) total += h.num[l] << (maxbits - l);
            while (total != (1u << maxbits)) {
                h.num[maxbits]--;
                for (u32 l = maxbits - 1; l > 0; l--)
                    if (h.num[l]) { h.num[l]--; h.num[l + 1] += 2; break; }
                total--;
            }
            int k = 0;
            for (u32 l = maxbits; l >= 1; l--)
                for (u32 j = 0; j < h.num[l]; j++) ln[h.sym[k++]] = l;
        }
    }
    __syncthreads();
}

// canonical codes (bit-reversed: DEFLATE sends Huffman codes from their top bit) of n lengths; one lane
__device__ void defl_codes(const u32 *ln, int n, u32 *tab, HuffScratch &h)
{
    for (u32 l = 0; l < 16; l++) h.num[l] = 0;
    for (int s = 0; s < n; s++) h.num[ln[s]]++;
    h.num[0] = 0;
    u32 code = 0;
    for (u32 b = 1; b < 16; b++) { code = (code + h.num[b - 1]) << 1; h.next[b] = code; }
    for (int s = 0; s < n; s++) {
        const u32 l = ln[s];
        tab[s] = l ? (__brev(h.next[l]++) >> (32 - l)) | l << 16 : 0;
    }
}

struct HdrWriter {
    u32 *w; u64 acc; u32 fill, nw;
    __device__ void put(u32 v, u32 nb) { acc |= (u64)v << fill; fill += nb; if (fill >= 32) { w[nw++] = (u32)acc; acc >>= 32; fill -= 32; } }
    __device__ u32 done() { if (fill) w[nw] = (u32)acc; return nw * 32 + fill; }
};

__constant__ u8 c_defl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

__global__ void __launch_bounds__(256) k_defl_huff(DeflateArgs a)
{
    __shared__ u32 f[CKZ_SYMS], ln[CKZ_SYMS], tab[CKZ_SYMS];
    __shared__ u32 rle[CKZ_SYMS], clf[19], cl[19], cltab[19];
    __shared__ HuffScratch h;
    const u32 seg = blockIdx.x, t = threadIdx.x;
    const u32 lo = seg * CKZ_SEG, hi = min(lo + CKZ_SEG, a.n), len = hi - lo;
    for (u32 i = t; i < CKZ_SYMS; i += 256) f[i] = a.freq[(u64)seg * CKZ_SYMS + i];
    if (t < 19) clf[t] = 0;
    __syncthreads();
    defl_lengths(f, CKZ_LL, 15, ln, h);
    defl_lengths(f + CKZ_LL, 30, 15, ln + CKZ_LL, h);
    __shared__ u32 s_hlit, s_hdist, s_nrle, s_type;
    if (t == 0) {
        u32 hlit = 257, hdist = 1;
        for (u32 s = 257; s < 286; s++) if (ln[s]) hlit = s + 1;
        for (u32 s = 0; s < 30; s++) if (ln[CKZ_LL + s]) hdist = s + 1;
        // run-length code of the hlit + hdist code lengths (symbols 16 / 17 / 18 with their extra bits in bits 8..)
        const u32 N = hlit + hdist;
        u32 nr = 0;
        for (u32 i = 0; i < N;) {
            const u32 v = ln[i < hlit ? i : CKZ_LL + i - hlit];
            u32 run = 1;
            while (i + run < N && ln[i + run < hlit ? i + run : CKZ_LL + i + run - hlit] == v) run++;
            u32 r = run;
            if (v == 0) {
                while (r >= 11) { const u32 k = min(r, 138u); rle[nr++] = 18 | (k - 11) << 8; clf[18]++; r -= k; }
                if (r >= 3) { rle[nr++] = 17 | (r - 3) << 8; clf[17]++; r = 0; }
            } else {
                rle[nr++] = v; clf[v]++; r--;
                while (r >= 3) { const u32 k = min(r, 6u); rle[nr++] = 16 | (k - 3) << 8; clf[16]++; r -= k; }
            }
            while (r > 0) { rle[nr++] = v; clf[v]++; r--; }
            i += run;
        }
        s_hlit = hlit; s_hdist = hdist; s_nrle = nr;
    }
    __syncthreads();
    defl_lengths(clf, 19, 7, cl, h);
    if (t == 0) {
        const u8 *order = c_defl_order;
        u32 hclen = 19;
        while (hclen > 4 && cl[order[hclen - 1]] == 0) hclen--;
        const u32 nr = s_nrle;
        u64 hdr_bits = 3 + 14 + 3 * hclen;
        for (u32 i = 0; i < nr; i++) {
            const u32 s = rle[i] & 255;
            hdr_bits += cl[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
        }
        u64 dyn = hdr_bits, fix = 3;
        for (u32 s = 0; s < CKZ_LL; s++) {
            if (!f[s]) continue;
            const u32 fl = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
            dyn += (u64)f[s] * (ln[s] + defl_lext(s));
            fix += (u64)f[s] * (fl + defl_lext(s));
        }
        for (u32 d = 0; d < 30; d++) {
            if (!f[CKZ_LL + d]) continue;
            dyn += (u64)f[CKZ_LL + d] * (ln[CKZ_LL + d] + defl_dext(d));
            fix += (u64)f[CKZ_LL + d] * (5 + defl_dext(d));
        }
        const bool last = hi == a.n;
        const u64 dyn_bytes = (dyn + 3 + 7) / 8 + 4, fix_bytes = (fix + 3 + 7) / 8 + 4;
        const u64 sto_bytes = len + 5ull * ((len + 65534) / 65535) + (last ? 5 : 0);
        u32 type = CKZ_DYNAMIC;
        u64 bytes = dyn_bytes;
        if (fix_bytes < bytes) { type = CKZ_FIXED; bytes = fix_bytes; }
        if (sto_bytes < bytes) { type = CKZ_STORED; bytes = sto_bytes; }
        HdrWriter w{a.hdr + (u64)seg * CKZ_HDR_WORDS, 0, 0, 0};
        if (type == CKZ_FIXED) {
            for (u32 s = 0; s < CKZ_LL; s++) ln[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
            for (u32 d = 0; d < 30; d++) ln[CKZ_LL + d] = 5;
            w.put(2, 3);                                  // BFINAL 0, BTYPE 01
        } else if (type == CKZ_DYNAMIC) {
            defl_codes(cl, 19, cltab, h);
            w.put(4, 3);                                  // BFINAL 0, BTYPE 10
            w.put(s_hlit - 257, 5); w.put(s_hdist - 1, 5); w.put(hclen - 4, 4);
            for (u32 i = 0; i < hclen; i++) w.put(cl[order[i]], 3);
            for (u32 i = 0; i < nr; i++) {
                const u32 s = rle[i] & 255, x = rle[i] >> 8;
                w.put(cltab[s] & 0xffff, cltab[s] >> 16);
                if (s == 16) w.put(x, 2); else if (s == 17) w.put(x, 3); else if (s == 18) w.put(x, 7);
            }
        }
        const u32 hb = type == CKZ_STORED ? 0 : w.done();
        if (type != CKZ_STORED) {
            defl_codes(ln, CKZ_LL, tab, h);
            defl_codes(ln + CKZ_LL, 30, tab + CKZ_LL, h);
        }
        u32 *meta = a.meta + 4ull * seg;
        meta[0] = hb; meta[1] = type; meta[2] = (u32)bytes; meta[3] = 0;
        s_type = type;
    }
    __syncthreads();
    if (s_type != CKZ_STORED)
        for (u32 i = t; i < CKZ_SYMS; i += 256) a.table[(u64)seg * CKZ_SYMS + i] = tab[i];
}

// ---- k_defl_place ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_defl_place(DeflateArgs a)
{
    typedef cub::BlockScan<u32, 1024> Scan;
    typedef cub::BlockReduce<u32, 1024> Reduce;
    __shared__ typename Scan::TempStorage scan;
    __shared__ typename Reduce::TempStorage red;
    const u32 s = threadIdx.x;
    const u32 bytes = s < a.nseg ? a.meta[4ull * s + 2] : 0;
    u32 o, total;
    Scan(scan).ExclusiveSum(bytes, o, total);
    if (s < a.nseg) a.off[s] = o;
    u32 c = 0;
    if (s < a.nseg) {
        const u32 hi = min((s + 1) * CKZ_SEG, a.n);
        c = a.seg_crc[s];
        if (a.n > hi) c = crc_multmodp(crc_x8n(a.n - hi), c);
    }
    const u32 raw = Reduce(red).Reduce(c, [](u32 u, u32 v) { return u ^ v; });
    if (s == 0) {
        a.result[0] = total;
        a.result[1] = 0;
        a.result[2] = ~(crc_multmodp(crc_x8n(a.n), ~a.crc_in) ^ raw);
    }
}

// ---- k_defl_pack ----------------------------------------------------------------------------------------------------------
// Bits go LSB first into 32-bit words of the output; a word entirely inside [lo, hi) belongs to this lane alone.
struct BitWriter {
    u32 *out; u64 word, lo, hi, acc; u32 fill;
    __device__ void init(u32 *o, u64 start, u64 end) { out = o; word = start >> 5; fill = start & 31; acc = 0; lo = start; hi = end; }
    __device__ void flush(u32 v)
    {
        const u64 b = word << 5;
        if (b >= lo && b + 32 <= hi) out[word] = v;
        else if (v) atomicOr(out + word, v);
        word++;
    }
    __device__ void put(u32 v, u32 nb) { acc |= (u64)v << fill; fill += nb; if (fill >= 32) { flush((u32)acc); acc >>= 32; fill -= 32; } }
    __device__ void finish() { if (fill) flush((u32)acc); }
};

__device__ __forceinline__ u32 defl_tok_bits(u32 tk, const u32 *tab)
{
    const u32 L = tk & 0x1ff;
    if (!L) return tab[tk >> 16] >> 16;
    u32 lnb, lx, dnb, dx;
    const u32 ls = defl_lsym(L, lnb, lx), ds = defl_dsym(tk >> 16, dnb, dx);
    return (tab[ls] >> 16) + lnb + (tab[CKZ_LL + ds] >> 16) + dnb;
}

__device__ __forceinline__ void defl_tok_put(BitWriter &w, u32 tk, const u32 *tab)
{
    const u32 L = tk & 0x1ff;
    if (!L) { const u32 e = tab[tk >> 16]; w.put(e & 0xffff, e >> 16); return; }
    u32 lnb, lx, dnb, dx;
    const u32 ls = defl_lsym(L, lnb, lx), ds = defl_dsym(tk >> 16, dnb, dx);
    const u32 el = tab[ls], ed = tab[CKZ_LL + ds];
    w.put(el & 0xffff, el >> 16);
    if (lnb) w.put(lx, lnb);
    w.put(ed & 0xffff, ed >> 16);
    if (dnb) w.put(dx, dnb);
}

__device__ __forceinline__ u32 defl_stored_byte(const u8 *in, u32 len, u32 r)   // byte r of a stored segment's output
{
    const u32 nblk = (len + 65534) / 65535, blk = r / 65540, q = r - blk * 65540;
    if (r < len + 5 * nblk) {
        const u32 blen = min(65535u, len - blk * 65535);
        switch (q) {
        case 0: return 0;                                 // BFINAL 0, BTYPE 00, padding
        case 1: return blen & 255;
        case 2: return blen >> 8;
        case 3: return ~blen & 255;
        case 4: return (~blen >> 8) & 255;
        default: return in[blk * 65535 + q - 5];
        }
    }
    return r - (len + 5 * nblk) >= 3 ? 0xff : 0;        // the empty stored block after the last segment
}

__global__ void __launch_bounds__(256) k_defl_pack(DeflateArgs a)
{
    __shared__ u32 tab[CKZ_SYMS];
    typedef cub::BlockScan<u64, 256> Scan;
    __shared__ typename Scan::TempStorage scan;
    const u32 seg = blockIdx.x, t = threadIdx.x;
    const u32 lo = seg * CKZ_SEG, hi = min(lo + CKZ_SEG, a.n), len = hi - lo;
    const u32 *meta = a.meta + 4ull * seg;
    const u32 hb = meta[0], type = meta[1], bytes = meta[2];
    const u64 O = a.off[seg];
    if (type == CKZ_STORED) {
        const u8 *in = a.buf + a.dict + lo;
        for (u64 w = (O >> 2) + t; w <= (O + bytes - 1) >> 2; w += 256) {
            u32 v = 0;
            for (u32 j = 0; j < 4; j++) {
                const u64 b = 4 * w + j;
                if (b >= O && b < O + bytes) v |= defl_stored_byte(in, len, (u32)(b - O)) << (8 * j);
            }
            if (4 * w >= O && 4 * w + 4 <= O + bytes) a.out[w] = v;
            else if (v) atomicOr(a.out + w, v);
        }
        return;
    }
    for (u32 i = t; i < CKZ_SYMS; i += 256) tab[i] = a.table[(u64)seg * CKZ_SYMS + i];
    __syncthreads();
    const u32 nt = a.ntok[seg], run = (nt + 255) / 256;
    const u32 ta = min(t * run, nt), tb = min(ta + run, nt);
    const u32 *tok = a.tok + lo;
    u64 bits = 0;
    for (u32 k = ta; k < tb; k++) bits += defl_tok_bits(tok[k], tab);
    if (t == 255) bits += tab[256] >> 16;                 // end of block
    u64 pre;
    Scan(scan).ExclusiveSum(bits, pre);
    const u64 base = O * 8;
    BitWriter w;
    if (t == 0) {                                         // the block header
        const u32 *hdr = a.hdr + (u64)seg * CKZ_HDR_WORDS;
        w.init(a.out, base, base + hb);
        u32 k = 0;
        for (; k + 32 <= hb; k += 32) w.put(hdr[k >> 5], 32);
        if (hb > k) w.put(hdr[k >> 5] & ((1u << (hb - k)) - 1), hb - k);
        w.finish();
    }
    const u64 start = base + hb + pre;
    w.init(a.out, start, start + bits);
    for (u32 k = ta; k < tb; k++) defl_tok_put(w, tok[k], tab);
    if (t == 255) {
        w.put(tab[256] & 0xffff, tab[256] >> 16);
        w.finish();
        // an empty stored block (3 zero bits, padding, 00 00) already reads as zeros: only its ff ff is left to write
        const u64 e = O + bytes;
        for (u64 b = e - 2; b < e; b++) atomicOr(a.out + (b >> 2), 0xffu << (8 * (b & 3)));
    } else {
        w.finish();
    }
}

}  // namespace ck
