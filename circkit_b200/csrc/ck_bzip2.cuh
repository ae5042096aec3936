// ck_bzip2.cuh -- bzip2 (libbzip2 1.0.8 at level 9, byte for byte) on the device for ck_bzip2_submit / ck_bzip2_wait: the
// `.bz2` output of the CLI.
//
// One call takes up to CK_BZIP2_MAX_BYTES of the stream and writes the bzip2 blocks that are complete in it (every block when
// the call is final) as one bit string.  The stages, in stream order:
//   k_bz_runs / k_bz_tok   run starts (max scan), then RLE1 tokens: a run of one byte value split at 255, coded as
//                          min(L, 4) copies plus a count byte L - 4 when L >= 4; every position holds the RLE1 bytes of the
//                          token that starts there (0 elsewhere), and an inclusive sum gives the RLE1 offsets
//   k_bz_cuts              one lane: greedy walk over those sums (a binary search per block): a block ends right after the
//                          first token that brings its RLE1 bytes to >= 899 981 (libbzip2's nblockMAX at level 9).  A call
//                          that is not final never uses the input's last token, which may still grow
//   k_bz_gather            the RLE1 bytes of every block, back to back
//   k_bz_crc               one CTA per block: CRC-32/BZIP2 (MSB first) of the block's raw range, per-lane CRCs combined by
//                          GF(2) shifts
//   k_bz_key0 + rounds     BWT of all blocks of the call in one sort: (block, 7 bytes read cyclically within the block),
//                          then prefix doubling: (rank[i], rank[(i + h) mod n]) with CUB radix sorts over the rotations still
//                          in groups of more than one, until every group is one rotation or h reaches the block's length
//                          (groups left then are identical rotations)
//   k_bz_orig              the last column of every block and origPtr (the last row of rotation 0's group)
//   k_bz_periodic          a block with equal rotations (rows libbzip2 orders by its fallbackSort): origPtr from that sort
//   k_bz_mtf               one CTA per block: the symbols in use; one warp runs move-to-front over the block with the
//                          256-entry list in registers (8 entries a lane) and codes zero runs as RUNA / RUNB
//   k_bz_huff              one CTA per block: libbzip2's table choice (2..6 tables, its initial partition, 4 iterations of
//                          choosing a table per 50-symbol group, in parallel over groups), BZ2_hbMakeCodeLengths per table
//                          (one lane per table), canonical codes, the block header's bits and the block's exact bit length
//   k_bz_place             one CTA: bit offsets of the blocks after the caller's pending bits; the combined CRC
//   k_bz_pack              one CTA per block: a scan of the groups' bit lengths, then every lane writes its groups MSB first;
//                          words wholly inside a lane's bit range are stored, shared edge words are OR-ed atomically
#pragma once
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "ck_device.cuh"

namespace ck {

#define CKB_BLOCK_MAX 899981u     // libbzip2's nblockMAX at level 9: 100000 * 9 - 19
#define CKB_MAX_BLOCKS 128u       // blocks of one call: every block covers >= 4/5 * CKB_BLOCK_MAX raw bytes
#define CKB_GSIZE 50u             // symbols per selector group
#define CKB_GROUPS 6              // most coding tables
#define CKB_ALPHA 258             // most symbols: 256 in use + RUNA / RUNB - 1 + EOB
#define CKB_MAX_SEL 18002u        // libbzip2's BZ_MAX_SELECTORS
#define CKB_HDR_WORDS 5120u       // block header: 105 + 272 + 18 + 6 * 18002 selector bits + 6 * (5 + 258 * 33) table bits
#define CKB_MAX_LEN 17
#define CKB_KEY0_CHARS 7u         // bytes in the first sort key (the block number takes the top byte)

struct Bzip2Block {               // per block of the call
    u32 raw_lo, raw_hi;           // raw input range
    u32 off, n;                   // RLE1 range
    u32 crc, orig, nmtf, ninuse;  // block CRC, origPtr, MTF symbols (EOB included), symbols in use
    u32 hdr_bits, body_bits, equal, pad;  // equal: rows whose rotation equals rotation 0
    u64 bit_off;                  // bit offset of the block in the call's output
};

struct Bzip2Meta {                // k_bz_cuts -> host
    u32 nblk, consumed, nrle, maxlen;
};

struct Bzip2Args {
    const u8 *in; u32 n, final;
    u32 *rs, *runst, *enc, *cum;  // run-start marks, run starts, token RLE1 bytes, their inclusive sum (n each)
    Bzip2Meta *meta;
    Bzip2Block *blk;              // CKB_MAX_BLOCKS
    u8 *rle, *bid;                // RLE1 bytes of the blocks, block of every RLE1 byte
    u32 *sa, *rank;               // rows -> rotation, rotation -> rank (first row of its group)
    u8 *last;                     // the BWT's last column, as seq numbers once k_bz_mtf mapped it
    u16 *mtfv;                    // block b's MTF symbols from blk[b].off + b
    u32 *freq;                    // CKB_MAX_BLOCKS * CKB_ALPHA
    u8 *sel;                      // CKB_MAX_BLOCKS * CKB_MAX_SEL
    u32 *code;                    // CKB_MAX_BLOCKS * CKB_GROUPS * CKB_ALPHA: code | length << 24
    u32 *hdr;                     // CKB_MAX_BLOCKS * CKB_HDR_WORDS
    int *hb;                      // CKB_MAX_BLOCKS * CKB_GROUPS * BzHeap scratch of BZ2_hbMakeCodeLengths
    u32 *out;                     // zeroed; big-endian words
    u32 *result;                  // [0..1] output bits, [2] combined CRC, [3] rotations left after a sort round
    u32 bits_in, nbits_in, crc_in;
};

// ---- CRC-32/BZIP2 (poly 0x04c11db7, MSB first) in GF(2) ------------------------------------------------------------------
__host__ __device__ __forceinline__ u32 bz_crc_mul(u32 a, u32 b)   // a * b mod P
{
    u32 p = 0;
    for (int k = 31; k >= 0; k--) {
        p = (p & 0x80000000u) ? (p << 1) ^ 0x04c11db7u : p << 1;
        if ((a >> k) & 1) p ^= b;
    }
    return p;
}

// x^(8 nbytes) mod P: the operator that runs an MSB-first CRC register over nbytes zero bytes
__host__ __device__ __forceinline__ u32 bz_crc_x8n(u64 nbytes)
{
    u32 r = 1, sq = 0x100;
    while (nbytes) {
        if (nbytes & 1) r = bz_crc_mul(r, sq);
        nbytes >>= 1;
        if (nbytes) sq = bz_crc_mul(sq, sq);
    }
    return r;
}

// ---- RLE1 tokens -------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_bz_runs(const u8 *in, u32 n, u32 *rs)
{
    const u32 i = blockIdx.x * 256u + threadIdx.x;
    if (i < n) rs[i] = (i == 0 || in[i] != in[i - 1]) ? i : 0;
}

__device__ __forceinline__ u32 bz_tok_len(const u8 *in, u32 n, u32 i)    // raw bytes of the token that starts at i
{
    const u8 c = in[i];
    u32 e = i + 1;
    while (e < n && e - i < 255 && in[e] == c) e++;
    return e - i;
}

__device__ __forceinline__ u32 bz_tok_start(const u32 *runst, u32 i) { return i - (i - runst[i]) % 255; }

__global__ void __launch_bounds__(256) k_bz_tok(Bzip2Args a)
{
    const u32 i = blockIdx.x * 256u + threadIdx.x;
    if (i >= a.n) return;
    u32 e = 0;
    if ((i - a.runst[i]) % 255 == 0) {
        const u32 L = bz_tok_len(a.in, a.n, i);
        e = L < 4 ? L : 5;
    }
    a.enc[i] = e;
}

// one lane: the greedy walk over the tokens' RLE1 sums
__global__ void k_bz_cuts(Bzip2Args a)
{
    const u32 n = a.n;
    const u32 limit = a.final ? n : bz_tok_start(a.runst, n - 1);   // tokens before `limit` can no longer change
    u32 p = 0, nb = 0, maxlen = 0;
    while (p < limit && nb < CKB_MAX_BLOCKS) {
        const u32 base = p ? a.cum[p - 1] : 0, target = base + CKB_BLOCK_MAX;
        u32 e;
        if (a.cum[limit - 1] < target) {
            if (!a.final) break;
            e = n;                                        // the final block: everything that is left
        } else {
            u32 lo = p, hi = limit - 1;                   // smallest j in [p, limit) with cum[j] >= target
            while (lo < hi) {
                const u32 m = lo + (hi - lo) / 2;
                if (a.cum[m] >= target) hi = m; else lo = m + 1;
            }
            e = lo + bz_tok_len(a.in, n, lo);
        }
        Bzip2Block &b = a.blk[nb];
        b.raw_lo = p; b.raw_hi = e; b.off = base; b.n = a.cum[e - 1] - base; b.orig = 0; b.equal = 0;
        maxlen = max(maxlen, b.n);
        nb++;
        p = e;
    }
    a.meta->nblk = nb;
    a.meta->consumed = p;
    a.meta->nrle = p ? a.cum[p - 1] : 0;
    a.meta->maxlen = maxlen;
}

__global__ void __launch_bounds__(256) k_bz_gather(Bzip2Args a, u32 consumed)
{
    const u32 i = blockIdx.x * 256u + threadIdx.x;
    if (i >= consumed) return;
    const u32 e = a.enc[i];
    if (!e) return;
    const u8 c = a.in[i];
    u8 *o = a.rle + a.cum[i] - e;
    if (e < 4) {
        for (u32 k = 0; k < e; k++) o[k] = c;
    } else {
        o[0] = c; o[1] = c; o[2] = c; o[3] = c;
        o[4] = (u8)(bz_tok_len(a.in, a.n, i) - 4);
    }
}

__global__ void __launch_bounds__(1024) k_bz_crc(Bzip2Args a)
{
    __shared__ u32 tab[256];
    typedef cub::BlockReduce<u32, 1024> Reduce;
    __shared__ typename Reduce::TempStorage red;
    const u32 t = threadIdx.x;
    Bzip2Block &b = a.blk[blockIdx.x];
    if (t < 256) {
        u32 c = t << 24;
        for (int k = 0; k < 8; k++) c = (c & 0x80000000u) ? (c << 1) ^ 0x04c11db7u : c << 1;
        tab[t] = c;
    }
    __syncthreads();
    const u32 lo = b.raw_lo, hi = b.raw_hi, len = hi - lo;
    const u32 run = (len + 1023) / 1024, ra = min(lo + t * run, hi), rb = min(ra + run, hi);
    u32 c = 0;
    for (u32 p = ra; p < rb; p++) c = (c << 8) ^ tab[(c >> 24) ^ a.in[p]];
    if (rb > ra && hi > rb) c = bz_crc_mul(bz_crc_x8n(hi - rb), c);
    const u32 x = Reduce(red).Reduce(c, [](u32 u, u32 v) { return u ^ v; });
    if (t == 0) b.crc = ~(bz_crc_mul(bz_crc_x8n(len), 0xffffffffu) ^ x);
}

// ---- BWT by prefix doubling ----------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 bz_block_of(const Bzip2Block *blk, u32 nblk, u32 k)   // block holding RLE1 byte k
{
    u32 lo = 0, hi = nblk - 1;
    while (lo < hi) {
        const u32 m = (lo + hi + 1) / 2;
        if (blk[m].off <= k) lo = m; else hi = m - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(256) k_bz_key0(Bzip2Args a, u32 nblk, u32 N, u64 *key, u32 *val, u32 *pos)
{
    const u32 k = blockIdx.x * 256u + threadIdx.x;
    if (k >= N) return;
    const u32 b = bz_block_of(a.blk, nblk, k), B = a.blk[b].off, nb = a.blk[b].n;
    u32 o = k - B;
    u64 v = (u64)b;
    for (u32 t = 0; t < CKB_KEY0_CHARS; t++) {
        v = v << 8 | a.rle[B + o];
        if (++o == nb) o = 0;
    }
    a.bid[k] = (u8)b;
    key[k] = v;
    val[k] = k;
    pos[k] = k;
}

// rows pos[0, m) (ascending) hold the rotations of the groups being refined; skey / sval are those rotations sorted
__global__ void __launch_bounds__(256) k_bz_mark(Bzip2Args a, u32 m, const u64 *skey, const u32 *sval, const u32 *pos,
                                                 u32 *hp)
{
    const u32 k = blockIdx.x * 256u + threadIdx.x;
    if (k >= m) return;
    a.sa[pos[k]] = sval[k];
    hp[k] = (k == 0 || skey[k] != skey[k - 1]) ? k : 0;
}

// new ranks; keep[k] = the rotation is still in a group of several that a longer prefix may split
__global__ void __launch_bounds__(256) k_bz_rank(Bzip2Args a, u32 m, const u64 *skey, const u32 *sval, const u32 *pos,
                                                 const u32 *hs, u32 sorted_chars, u8 *keep)
{
    const u32 k = blockIdx.x * 256u + threadIdx.x;
    if (k >= m) return;
    const u32 i = sval[k];
    a.rank[i] = pos[hs[k]];
    const bool head = hs[k] == k, tail = k + 1 == m || skey[k + 1] != skey[k];
    keep[k] = !(head && tail) && a.blk[a.bid[i]].n > sorted_chars;
}

__global__ void __launch_bounds__(256) k_bz_key(Bzip2Args a, u32 m, const u32 *pos, u32 h, u32 rbits, u64 *key, u32 *val)
{
    const u32 k = blockIdx.x * 256u + threadIdx.x;
    if (k >= m) return;
    const u32 i = a.sa[pos[k]];
    const Bzip2Block &b = a.blk[a.bid[i]];
    const u32 j = b.off + (u32)(((u64)(i - b.off) + h) % b.n);
    key[k] = (u64)a.rank[i] << rbits | a.rank[j];
    val[k] = i;
}

// origPtr of a block that is a power of a shorter word, where rows of equal rotations make the order libbzip2's: its
// fallbackSort (which it runs on such blocks: below 10 000 bytes always, above once the main sort exhausts its budget), step
// for step.  fmap and eclass hold n words, bhtab n / 32 + 8.
__host__ __device__ inline void bz_fb_simple(u32 *fmap, const u32 *eclass, int lo, int hi)
{
    if (lo == hi) return;
    if (hi - lo > 3) {
        for (int i = hi - 4; i >= lo; i--) {
            const u32 tmp = fmap[i], ec = eclass[tmp];
            int j;
            for (j = i + 4; j <= hi && ec > eclass[fmap[j]]; j += 4) fmap[j - 4] = fmap[j];
            fmap[j - 4] = tmp;
        }
    }
    for (int i = hi - 1; i >= lo; i--) {
        const u32 tmp = fmap[i], ec = eclass[tmp];
        int j;
        for (j = i + 1; j <= hi && ec > eclass[fmap[j]]; j++) fmap[j - 1] = fmap[j];
        fmap[j - 1] = tmp;
    }
}

__host__ __device__ inline void bz_fb_qsort3(u32 *fmap, const u32 *eclass, int loSt, int hiSt)
{
    int stackLo[100], stackHi[100], sp = 0;
    u32 r = 0;
    stackLo[sp] = loSt; stackHi[sp] = hiSt; sp++;
    while (sp > 0) {
        sp--;
        const int lo = stackLo[sp], hi = stackHi[sp];
        if (hi - lo < 10) { bz_fb_simple(fmap, eclass, lo, hi); continue; }
        r = ((r * 7621) + 1) % 32768;
        const u32 r3 = r % 3;
        const u32 med = r3 == 0 ? eclass[fmap[lo]] : r3 == 1 ? eclass[fmap[(lo + hi) >> 1]] : eclass[fmap[hi]];
        int unLo = lo, ltLo = lo, unHi = hi, gtHi = hi, n, m;
        for (;;) {
            for (;;) {
                if (unLo > unHi) break;
                n = (int)eclass[fmap[unLo]] - (int)med;
                if (n == 0) { u32 t = fmap[unLo]; fmap[unLo] = fmap[ltLo]; fmap[ltLo] = t; ltLo++; unLo++; continue; }
                if (n > 0) break;
                unLo++;
            }
            for (;;) {
                if (unLo > unHi) break;
                n = (int)eclass[fmap[unHi]] - (int)med;
                if (n == 0) { u32 t = fmap[unHi]; fmap[unHi] = fmap[gtHi]; fmap[gtHi] = t; gtHi--; unHi--; continue; }
                if (n < 0) break;
                unHi--;
            }
            if (unLo > unHi) break;
            u32 t = fmap[unLo]; fmap[unLo] = fmap[unHi]; fmap[unHi] = t;
            unLo++; unHi--;
        }
        if (gtHi < ltLo) continue;
        n = min(ltLo - lo, unLo - ltLo);
        for (int a = lo, b = unLo - n, k = n; k > 0; a++, b++, k--) { u32 t = fmap[a]; fmap[a] = fmap[b]; fmap[b] = t; }
        m = min(hi - gtHi, gtHi - unHi);
        for (int a = unLo, b = hi - m + 1, k = m; k > 0; a++, b++, k--) { u32 t = fmap[a]; fmap[a] = fmap[b]; fmap[b] = t; }
        n = lo + unLo - ltLo - 1;
        m = hi - (gtHi - unHi) + 1;
        if (n - lo > hi - m) {
            stackLo[sp] = lo; stackHi[sp] = n; sp++;
            stackLo[sp] = m; stackHi[sp] = hi; sp++;
        } else {
            stackLo[sp] = m; stackHi[sp] = hi; sp++;
            stackLo[sp] = lo; stackHi[sp] = n; sp++;
        }
    }
}

__host__ __device__ inline u32 bz_fallback_orig(const u8 *blk, int nblock, u32 *fmap, u32 *eclass, u32 *bhtab)
{
#define BZ_SET(z) (bhtab[(z) >> 5] |= (1u << ((z) & 31)))
#define BZ_CLR(z) (bhtab[(z) >> 5] &= ~(1u << ((z) & 31)))
#define BZ_ISSET(z) (bhtab[(z) >> 5] & (1u << ((z) & 31)))
#define BZ_WORD(z) (bhtab[(z) >> 5])
#define BZ_UNALIGNED(z) ((z) & 0x1f)
    int ftab[257];
    for (int i = 0; i < 257; i++) ftab[i] = 0;
    for (int i = 0; i < nblock; i++) ftab[blk[i]]++;
    for (int i = 1; i < 257; i++) ftab[i] += ftab[i - 1];
    for (int i = 0; i < nblock; i++) { const int j = blk[i], k = ftab[j] - 1; ftab[j] = k; fmap[k] = i; }
    const int nBhtab = 2 + (nblock / 32);
    for (int i = 0; i < nBhtab + 2; i++) bhtab[i] = 0;
    for (int i = 0; i < 256; i++) BZ_SET(ftab[i]);
    for (int i = 0; i < 32; i++) { BZ_SET(nblock + 2 * i); BZ_CLR(nblock + 2 * i + 1); }
    int H = 1;
    for (;;) {
        int j = 0;
        for (int i = 0; i < nblock; i++) {
            if (BZ_ISSET(i)) j = i;
            int k = (int)fmap[i] - H;
            if (k < 0) k += nblock;
            eclass[k] = (u32)j;
        }
        int nNotDone = 0, r = -1;
        for (;;) {
            int k = r + 1;
            while (BZ_ISSET(k) && BZ_UNALIGNED(k)) k++;
            if (BZ_ISSET(k)) {
                while (BZ_WORD(k) == 0xffffffffu) k += 32;
                while (BZ_ISSET(k)) k++;
            }
            const int l = k - 1;
            if (l >= nblock) break;
            while (!BZ_ISSET(k) && BZ_UNALIGNED(k)) k++;
            if (!BZ_ISSET(k)) {
                while (BZ_WORD(k) == 0) k += 32;
                while (!BZ_ISSET(k)) k++;
            }
            r = k - 1;
            if (r >= nblock) break;
            if (r > l) {
                nNotDone += r - l + 1;
                bz_fb_qsort3(fmap, eclass, l, r);
                int cc = -1;
                for (int i = l; i <= r; i++) {
                    const int cc1 = (int)eclass[fmap[i]];
                    if (cc != cc1) { BZ_SET(i); cc = cc1; }
                }
            }
        }
        H *= 2;
        if (H > nblock || nNotDone == 0) break;
    }
    u32 orig = 0;
    for (int i = 0; i < nblock; i++) if (fmap[i] == 0) { orig = (u32)i; break; }
    return orig;
#undef BZ_SET
#undef BZ_CLR
#undef BZ_ISSET
#undef BZ_WORD
#undef BZ_UNALIGNED
}

struct BzMax {
    __host__ __device__ __forceinline__ u32 operator()(u32 x, u32 y) const { return x > y ? x : y; }
};

// the last column (RLE1 byte before each row's rotation) and origPtr (the last row of rotation 0's group)
__global__ void __launch_bounds__(256) k_bz_orig(Bzip2Args a, u32 N)
{
    const u32 k = blockIdx.x * 256u + threadIdx.x;
    if (k >= N) return;
    const u32 i = a.sa[k];
    Bzip2Block &b = a.blk[a.bid[k]];
    const u32 o = i - b.off;
    a.last[k] = a.rle[b.off + (o ? o - 1 : b.n - 1)];
    if (a.rank[i] == a.rank[b.off]) { atomicMax(&b.orig, k - b.off); atomicAdd(&b.equal, 1u); }
}

// one lane per block: a block with equal rotations (a power of a shorter word) takes libbzip2's order of them.  The sort
// buffers are free by now: fmap in sa, eclass in rank, bhtab in hp
__global__ void k_bz_periodic(Bzip2Args a, u32 *hp)
{
    Bzip2Block &b = a.blk[blockIdx.x];
    if (b.equal > 1)
        b.orig = bz_fallback_orig(a.rle + b.off, (int)b.n, a.sa + b.off, a.rank + b.off, hp + b.off / 32 + 8 * blockIdx.x);
}

// ---- move-to-front and zero runs -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_bz_mtf(Bzip2Args a)
{
    __shared__ u8 seen[256], seq[256];
    __shared__ u32 fq[CKB_ALPHA], s_ninuse;
    const u32 t = threadIdx.x, bi = blockIdx.x;
    Bzip2Block &b = a.blk[bi];
    const u32 B = b.off, n = b.n;
    seen[t] = 0;
    for (u32 v = t; v < CKB_ALPHA; v += 256) fq[v] = 0;
    __syncthreads();
    for (u32 k = t; k < n; k += 256) {
        const u8 c = a.rle[B + k];
        if (!seen[c]) seen[c] = 1;
    }
    __syncthreads();
    if (t == 0) {
        u32 q = 0;
        for (u32 c = 0; c < 256; c++) { seq[c] = (u8)q; q += seen[c]; }
        s_ninuse = q;
    }
    __syncthreads();
    const u32 ninuse = s_ninuse, EOB = ninuse + 1;
    for (u32 k = t; k < n; k += 256) a.last[B + k] = seq[a.last[B + k]];
    __syncthreads();
    if (t < 32) {
        const u32 lane = t;
        u64 w = 0;                                        // list entries lane * 8 + j at bits 8 j; unused entries 0xff
        for (u32 j = 0; j < 8; j++) {
            const u32 v = lane * 8 + j;
            w |= (u64)(v < ninuse ? v : 0xffu) << (8 * j);
        }
        u16 *out = a.mtfv + B + bi;
        u32 wr = 0, zpend = 0, front = 0;
        const u8 *L = a.last + B;
        for (u32 k0 = 0; k0 < n; k0 += 32) {
            const u32 mine = k0 + lane < n ? L[k0 + lane] : 0, cnt = min(32u, n - k0);
            for (u32 q = 0; q < cnt; q++) {
                const u32 s = __shfl_sync(0xffffffffu, mine, q);
                if (s == front) { zpend++; continue; }
                const u32 rep = s * 0x01010101u;
                const u32 mlo = __vcmpeq4((u32)w, rep), mhi = __vcmpeq4((u32)(w >> 32), rep);
                const u64 mm = (u64)mhi << 32 | mlo;
                const u32 ball = __ballot_sync(0xffffffffu, mm != 0);
                const u32 Lf = __ffs(ball) - 1;
                const u32 jb = mm ? (u32)(__ffsll(mm) - 1) >> 3 : 0;
                const u32 j = __shfl_sync(0xffffffffu, jb, Lf);
                u64 carry = __shfl_up_sync(0xffffffffu, w >> 56, 1);
                if (lane == 0) carry = s;
                const u64 sh = w << 8 | carry;
                if (lane < Lf) {
                    w = sh;
                } else if (lane == Lf) {
                    const u64 mask = j == 7 ? ~0ull : (1ull << (8 * (j + 1))) - 1;
                    w = (sh & mask) | (w & ~mask);
                }
                front = s;
                if (lane == 0) {
                    if (zpend) {
                        zpend--;
                        for (;;) {
                            const u32 r = zpend & 1;     // RUNB = 1, RUNA = 0
                            out[wr++] = (u16)r; fq[r]++;
                            if (zpend < 2) break;
                            zpend = (zpend - 2) / 2;
                        }
                        zpend = 0;
                    }
                    const u32 v = Lf * 8 + j + 1;
                    out[wr++] = (u16)v; fq[v]++;
                }
                zpend = 0;
            }
        }
        if (lane == 0) {
            if (zpend) {
                zpend--;
                for (;;) {
                    const u32 r = zpend & 1;
                    out[wr++] = (u16)r; fq[r]++;
                    if (zpend < 2) break;
                    zpend = (zpend - 2) / 2;
                }
            }
            out[wr++] = (u16)EOB; fq[EOB]++;
            b.nmtf = wr;
            b.ninuse = ninuse;
        }
    }
    __syncthreads();
    for (u32 v = t; v < CKB_ALPHA; v += 256) a.freq[bi * CKB_ALPHA + v] = fq[v];
}

// ---- Huffman tables (libbzip2's sendMTFValues) ------------------------------------------------------------------------------
struct BzHeap {
    int heap[CKB_ALPHA + 2], weight[CKB_ALPHA * 2], parent[CKB_ALPHA * 2];
};

// BZ2_hbMakeCodeLengths of libbzip2 1.0.8, step for step (equal weights keep its heap order)
__host__ __device__ inline void bz_make_lengths(u8 *len, const u32 *freq, int alpha, int maxlen, BzHeap &H)
{
    int *heap = H.heap, *weight = H.weight, *parent = H.parent;
    for (int i = 0; i < alpha; i++) weight[i + 1] = (freq[i] == 0 ? 1 : (int)freq[i]) << 8;
    for (;;) {
        int nNodes = alpha, nHeap = 0;
        heap[0] = 0; weight[0] = 0; parent[0] = -2;
        for (int i = 1; i <= alpha; i++) {
            parent[i] = -1;
            nHeap++;
            heap[nHeap] = i;
            int zz = nHeap, tmp = heap[zz];
            while (weight[tmp] < weight[heap[zz >> 1]]) { heap[zz] = heap[zz >> 1]; zz >>= 1; }
            heap[zz] = tmp;
        }
        while (nHeap > 1) {
            int nn[2];
            for (int r = 0; r < 2; r++) {
                nn[r] = heap[1];
                heap[1] = heap[nHeap];
                nHeap--;
                int zz = 1, tmp = heap[zz];
                for (;;) {
                    int yy = zz << 1;
                    if (yy > nHeap) break;
                    if (yy < nHeap && weight[heap[yy + 1]] < weight[heap[yy]]) yy++;
                    if (weight[tmp] < weight[heap[yy]]) break;
                    heap[zz] = heap[yy];
                    zz = yy;
                }
                heap[zz] = tmp;
            }
            nNodes++;
            parent[nn[0]] = parent[nn[1]] = nNodes;
            const int w1 = weight[nn[0]], w2 = weight[nn[1]];
            const int d1 = w1 & 0xff, d2 = w2 & 0xff;
            weight[nNodes] = (int)(((u32)w1 & 0xffffff00u) + ((u32)w2 & 0xffffff00u)) | (1 + (d1 > d2 ? d1 : d2));
            parent[nNodes] = -1;
            nHeap++;
            heap[nHeap] = nNodes;
            int zz = nHeap, tmp = heap[zz];
            while (weight[tmp] < weight[heap[zz >> 1]]) { heap[zz] = heap[zz >> 1]; zz >>= 1; }
            heap[zz] = tmp;
        }
        bool tooLong = false;
        for (int i = 1; i <= alpha; i++) {
            int j = 0, k = i;
            while (parent[k] >= 0) { k = parent[k]; j++; }
            len[i - 1] = (u8)j;
            if (j > maxlen) tooLong = true;
        }
        if (!tooLong) break;
        for (int i = 1; i <= alpha; i++) weight[i] = (1 + (weight[i] >> 8) / 2) << 8;
    }
}

__host__ __device__ inline int bz_ngroups(u32 nmtf)
{
    return nmtf < 200 ? 2 : nmtf < 600 ? 3 : nmtf < 1200 ? 4 : nmtf < 2400 ? 5 : 6;
}

// the initial tables: symbol ranges of about equal frequency, cost 0 inside the range and 15 outside
__host__ __device__ inline void bz_initial_tables(u8 (*len)[CKB_ALPHA], const u32 *freq, int alpha, int nG, u32 nmtf)
{
    int nPart = nG, gs = 0;
    int remF = (int)nmtf;
    while (nPart > 0) {
        const int tFreq = remF / nPart;
        int ge = gs - 1, aFreq = 0;
        while (aFreq < tFreq && ge < alpha - 1) { ge++; aFreq += (int)freq[ge]; }
        if (ge > gs && nPart != nG && nPart != 1 && ((nG - nPart) % 2 == 1)) { aFreq -= (int)freq[ge]; ge--; }
        for (int v = 0; v < alpha; v++) len[nPart - 1][v] = (v >= gs && v <= ge) ? 0 : 15;
        nPart--;
        gs = ge + 1;
        remF -= aFreq;
    }
}

// the table a group of symbols costs least with (the lowest on equal cost)
__host__ __device__ inline int bz_best_table(const u16 *v, u32 cnt, const u8 (*len)[CKB_ALPHA], int nG)
{
    u32 cost[CKB_GROUPS] = {0, 0, 0, 0, 0, 0};
    for (u32 i = 0; i < cnt; i++) {
        const u32 s = v[i];
#pragma unroll
        for (int t = 0; t < CKB_GROUPS; t++) if (t < nG) cost[t] += len[t][s];
    }
    int bt = 0;
    u32 bc = cost[0];
#pragma unroll
    for (int t = 1; t < CKB_GROUPS; t++) if (t < nG && cost[t] < bc) { bc = cost[t]; bt = t; }
    return bt;
}

// MSB-first bits into big-endian words
struct BzBits {
    u32 *w; u64 acc; u32 fill, nw;
    __host__ __device__ void put(u32 v, u32 nb) { acc = acc << nb | v; fill += nb; if (fill >= 32) { w[nw++] = (u32)(acc >> (fill - 32)); fill -= 32; } }
    __host__ __device__ u32 done() { if (fill) w[nw] = (u32)(acc << (32 - fill)); return nw * 32 + fill; }
};

// the block header: magic, CRC, origPtr, symbol map, selectors, code lengths; codes[t][v] = code | length << 24
__host__ __device__ inline u32 bz_header(u32 *words, u32 crc, u32 orig, const u8 *seen, int alpha, int nG, const u8 *sel,
                                         u32 nsel, const u8 (*len)[CKB_ALPHA], u32 *codes)
{
    BzBits w{words, 0, 0, 0};
    w.put(0x314159u, 24); w.put(0x265359u, 24);
    w.put(crc >> 16, 16); w.put(crc & 0xffff, 16);
    w.put(0, 1);
    w.put(orig, 24);
    u32 used16 = 0;
    for (int i = 0; i < 16; i++) {
        bool any = false;
        for (int j = 0; j < 16; j++) any |= seen[i * 16 + j] != 0;
        if (any) used16 |= 1u << i;
        w.put(any, 1);
    }
    for (int i = 0; i < 16; i++)
        if (used16 >> i & 1)
            for (int j = 0; j < 16; j++) w.put(seen[i * 16 + j] != 0, 1);
    w.put(nG, 3);
    w.put(nsel, 15);
    u8 pos[CKB_GROUPS];
    for (int i = 0; i < nG; i++) pos[i] = (u8)i;
    for (u32 i = 0; i < nsel; i++) {
        const u8 s = sel[i];
        int j = 0;
        u8 tmp = pos[0];
        while (s != tmp) { j++; const u8 t2 = tmp; tmp = pos[j]; pos[j] = t2; }
        pos[0] = tmp;
        for (int k = 0; k < j; k++) w.put(1, 1);
        w.put(0, 1);
    }
    for (int t = 0; t < nG; t++) {
        int curr = len[t][0];
        w.put(curr, 5);
        for (int i = 0; i < alpha; i++) {
            while (curr < len[t][i]) { w.put(2, 2); curr++; }
            while (curr > len[t][i]) { w.put(3, 2); curr--; }
            w.put(0, 1);
        }
        int minLen = 32, maxLen = 0;
        for (int i = 0; i < alpha; i++) { minLen = min(minLen, (int)len[t][i]); maxLen = max(maxLen, (int)len[t][i]); }
        u32 vec = 0;
        for (int n = minLen; n <= maxLen; n++) {
            for (int i = 0; i < alpha; i++)
                if (len[t][i] == n) codes[t * CKB_ALPHA + i] = vec++ | (u32)n << 24;
            vec <<= 1;
        }
    }
    return w.done();
}

__global__ void __launch_bounds__(256) k_bz_huff(Bzip2Args a)
{
    __shared__ u8 len[CKB_GROUPS][CKB_ALPHA];
    __shared__ u32 rfreq[CKB_GROUPS][CKB_ALPHA], codes[CKB_GROUPS * CKB_ALPHA];
    __shared__ u8 sel[CKB_MAX_SEL], seen[256];
    typedef cub::BlockReduce<u32, 256> Reduce;
    __shared__ typename Reduce::TempStorage red;
    const u32 t = threadIdx.x, bi = blockIdx.x;
    Bzip2Block &b = a.blk[bi];
    const u32 nmtf = b.nmtf, nsel = (nmtf + CKB_GSIZE - 1) / CKB_GSIZE;
    const int alpha = (int)b.ninuse + 2, nG = bz_ngroups(nmtf);
    const u16 *v = a.mtfv + b.off + bi;
    const u32 *freq = a.freq + bi * CKB_ALPHA;
    if (t == 0) bz_initial_tables(len, freq, alpha, nG, nmtf);
    seen[t] = 0;
    __syncthreads();
    for (u32 k = t; k < b.n; k += 256) {
        const u8 c = a.rle[b.off + k];
        if (!seen[c]) seen[c] = 1;
    }
    for (int iter = 0; iter < 4; iter++) {
        for (u32 k = t; k < CKB_GROUPS * CKB_ALPHA; k += 256) (&rfreq[0][0])[k] = 0;
        __syncthreads();
        for (u32 g = t; g < nsel; g += 256) {
            const u32 gs = g * CKB_GSIZE, cnt = min(CKB_GSIZE, nmtf - gs);
            const int bt = bz_best_table(v + gs, cnt, len, nG);
            sel[g] = (u8)bt;
            for (u32 i = 0; i < cnt; i++) atomicAdd(&rfreq[bt][v[gs + i]], 1u);
        }
        __syncthreads();
        if ((int)t < nG)
            bz_make_lengths(len[t], rfreq[t], alpha, CKB_MAX_LEN,
                            *reinterpret_cast<BzHeap *>(a.hb + ((u64)bi * CKB_GROUPS + t) * (sizeof(BzHeap) / 4)));
        __syncthreads();
    }
    if (t == 0) b.hdr_bits = bz_header(a.hdr + (u64)bi * CKB_HDR_WORDS, b.crc, b.orig, seen, alpha, nG, sel, nsel, len, codes);
    __syncthreads();
    u32 bits = 0;
    for (u32 g = t; g < nsel; g += 256) {
        const u32 gs = g * CKB_GSIZE, cnt = min(CKB_GSIZE, nmtf - gs);
        for (u32 i = 0; i < cnt; i++) bits += len[sel[g]][v[gs + i]];
    }
    const u32 body = Reduce(red).Sum(bits);
    if (t == 0) b.body_bits = body;
    for (u32 k = t; k < nsel; k += 256) a.sel[(u64)bi * CKB_MAX_SEL + k] = sel[k];
    for (u32 k = t; k < CKB_GROUPS * CKB_ALPHA; k += 256) a.code[(u64)bi * CKB_GROUPS * CKB_ALPHA + k] = codes[k];
}

// ---- place and pack ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CKB_MAX_BLOCKS) k_bz_place(Bzip2Args a, u32 nblk)
{
    typedef cub::BlockScan<u64, CKB_MAX_BLOCKS> Scan;
    __shared__ typename Scan::TempStorage scan;
    const u32 t = threadIdx.x;
    const u64 bits = t < nblk ? (u64)a.blk[t].hdr_bits + a.blk[t].body_bits : 0;
    u64 o, total;
    Scan(scan).ExclusiveSum(bits, o, total);
    if (t < nblk) a.blk[t].bit_off = a.nbits_in + o;
    if (t == 0) {
        u32 crc = a.crc_in;
        for (u32 k = 0; k < nblk; k++) crc = (crc << 1 | crc >> 31) ^ a.blk[k].crc;
        total += a.nbits_in;
        a.result[0] = (u32)total; a.result[1] = (u32)(total >> 32); a.result[2] = crc;
        if (a.nbits_in) atomicOr(a.out, __byte_perm(a.bits_in << (32 - a.nbits_in), 0, 0x0123));
    }
}

// MSB-first bits into the zeroed output; a word entirely inside [lo, hi) belongs to this lane alone
struct BzWriter {
    u32 *out; u64 word, lo, hi, acc; u32 fill;
    __device__ void init(u32 *o, u64 start, u64 end) { out = o; word = start >> 5; fill = start & 31; acc = 0; lo = start; hi = end; }
    __device__ void flush(u32 v)
    {
        const u64 bb = word << 5;
        const u32 sw = __byte_perm(v, 0, 0x0123);
        if (bb >= lo && bb + 32 <= hi) out[word] = sw;
        else if (v) atomicOr(out + word, sw);
        word++;
    }
    __device__ void put(u32 v, u32 nb) { acc = acc << nb | v; fill += nb; if (fill >= 32) { flush((u32)(acc >> (fill - 32))); fill -= 32; } }
    __device__ void finish() { if (fill) flush((u32)(acc << (32 - fill))); }
};

__global__ void __launch_bounds__(256) k_bz_pack(Bzip2Args a)
{
    __shared__ u32 codes[CKB_GROUPS * CKB_ALPHA];
    typedef cub::BlockScan<u32, 256> Scan;
    __shared__ typename Scan::TempStorage scan;
    const u32 t = threadIdx.x, bi = blockIdx.x;
    const Bzip2Block &b = a.blk[bi];
    for (u32 k = t; k < CKB_GROUPS * CKB_ALPHA; k += 256) codes[k] = a.code[(u64)bi * CKB_GROUPS * CKB_ALPHA + k];
    __syncthreads();
    const u32 nmtf = b.nmtf, nsel = (nmtf + CKB_GSIZE - 1) / CKB_GSIZE, hb = b.hdr_bits;
    const u16 *v = a.mtfv + b.off + bi;
    const u8 *sel = a.sel + (u64)bi * CKB_MAX_SEL;
    const u32 run = (nsel + 255) / 256, ga = min(t * run, nsel), gb = min(ga + run, nsel);
    u32 bits = 0;
    for (u32 g = ga; g < gb; g++) {
        const u32 *c = codes + sel[g] * CKB_ALPHA;
        for (u32 i = g * CKB_GSIZE, e = min(i + CKB_GSIZE, nmtf); i < e; i++) bits += c[v[i]] >> 24;
    }
    u32 pre;
    Scan(scan).ExclusiveSum(bits, pre);
    BzWriter w;
    if (t == 0) {
        const u32 *hdr = a.hdr + (u64)bi * CKB_HDR_WORDS;
        w.init(a.out, b.bit_off, b.bit_off + hb);
        u32 k = 0;
        for (; k + 32 <= hb; k += 32) w.put(hdr[k >> 5], 32);
        if (hb > k) w.put(hdr[k >> 5] >> (32 - (hb - k)), hb - k);
        w.finish();
    }
    const u64 start = b.bit_off + hb + pre;
    w.init(a.out, start, start + bits);
    for (u32 g = ga; g < gb; g++) {
        const u32 *c = codes + sel[g] * CKB_ALPHA;
        for (u32 i = g * CKB_GSIZE, e = min(i + CKB_GSIZE, nmtf); i < e; i++) {
            const u32 x = c[v[i]];
            w.put(x & 0xffffffu, x >> 24);
        }
    }
    w.finish();
}

}  // namespace ck
