// ck_kernels.cuh -- the kernels of the canonicalize / uniq hot path (sm_100a, no tensor cores:
// nothing here is a contraction; the work is integer scan + hash + hash-table traffic).
//
//   k_prepare      normalise (needletail rules) + classify + pack one batch of raw records
//   k_classify     route records to a symbol lane / thread shape by alphabet and length
//   k_canon_warp   warp-per-record LMSR + canonical form + XXH3-64       (viroid / circRNA sizes)
//   k_canon_cta    CTA-per-record, same algorithm                        (plasmid / mtDNA sizes)
//   k_table_insert first-occurrence table: CAS the key, atomicMin the input index
//   k_table_first  read back first_index per record
//   k_table_rehash move a context's table into a larger one (ck_uniq_grow)
#pragma once
#include "ck_hash.cuh"

namespace ck {

// record classes (index into the per-class work lists)
enum : int {
    CLS_W2S = 0,   // 2-bit, warp, n <= 512
    CLS_W2M = 1,   // 2-bit, warp, n <= 2048
    CLS_C2A = 2,   // 2-bit, CTA,  n <= 65536
    CLS_C2B = 3,   // 2-bit, CTA,  n <= 425984
    CLS_W4 = 4,    // 4-bit, warp, n <= 2048
    CLS_C4 = 5,    // 4-bit, CTA,  n <= 212992
    CLS_W8 = 6,    // bytes, warp, n <= 1024
    CLS_C8 = 7,    // bytes, CTA,  n <= 106496
    CLS_HUGE = 8,  // anything longer: strands staged in global scratch
    CLS_EMPTY = 9, // n == 0
    CLS_W2L = 10,  // 2-bit, warp, n <= 4096
    CLS_W2X = 11,  // 2-bit, warp, n <= 8192
    CLS_COUNT = 12
};
__host__ __device__ constexpr u32 cls_max_n(int c)
{
    return c == CLS_W2S ? 512u : c == CLS_W2M ? 2048u : c == CLS_W2L ? 4096u : c == CLS_W2X ? 8192u : c == CLS_C2A ? 65536u
         : c == CLS_C2B ? 425984u : c == CLS_W4 ? 2048u : c == CLS_C4 ? 212992u : c == CLS_W8 ? 1024u : c == CLS_C8 ? 106496u
         : c == CLS_EMPTY ? 0u : 0xffffffffu;
}
// smallest length of a class (the class below it in the same symbol lane ends one short of it)
__host__ __device__ constexpr u32 cls_min_n(int c)
{
    return c == CLS_W2M ? cls_max_n(CLS_W2S) + 1 : c == CLS_W2L ? cls_max_n(CLS_W2M) + 1 : c == CLS_W2X ? cls_max_n(CLS_W2L) + 1
         : c == CLS_C2A ? cls_max_n(CLS_W2X) + 1 : c == CLS_C2B ? cls_max_n(CLS_C2A) + 1 : c == CLS_C4 ? cls_max_n(CLS_W4) + 1
         : c == CLS_C8 ? cls_max_n(CLS_W8) + 1 : c == CLS_EMPTY ? 0u : 1u;
}

// order of the classes in the sorted index list: the lane-kernel classes first, contiguous, by length
__host__ __device__ constexpr u32 cls_rank(int c)
{
    return c == CLS_W2S ? 0u : c == CLS_W2M ? 1u : c == CLS_W2L ? 2u : c == CLS_W2X ? 3u : c == CLS_C2A ? 4u : c == CLS_C2B ? 5u
         : c == CLS_W4 ? 6u : c == CLS_C4 ? 7u : c == CLS_W8 ? 8u : c == CLS_C8 ? 9u : c == CLS_HUGE ? 10u : 11u;
}
__host__ __device__ constexpr int cls_of_rank(u32 r)
{
    return r == 0 ? CLS_W2S : r == 1 ? CLS_W2M : r == 2 ? CLS_W2L : r == 3 ? CLS_W2X : r == 4 ? CLS_C2A : r == 5 ? CLS_C2B
         : r == 6 ? CLS_W4 : r == 7 ? CLS_C4 : r == 8 ? CLS_W8 : r == 9 ? CLS_C8 : r == 10 ? CLS_HUGE : CLS_EMPTY;
}

// First-occurrence table slot (see "First-occurrence table" below).  (Inserting from inside the kernels that produce the
// hashes was measured and dropped: the probes' returned atomics stall the latency-sensitive lane kernel -- config 2: 5.68 ->
// 8.21 ms, config 5: 1.92 -> 4.32 ms -- far more than the separate insert pass costs.)
struct TableSlot { u64 key; u64 first; };
#define CK_EMPTY_KEY 0xffffffffffffffffULL
// home slot in a table of any size: the high half of mix(key) * nslots (no power of two needed: 1.5 slots per key instead of
// 2..4, and the table of a 10 M-key batch is 250 MB instead of 537 MB -- closer to what L2 can hold).  The multiplicative mix
// spreads keys whose top bits are all alike (the keys a rank owns in the multi-GPU exchange are one range of the top bits).
__device__ __forceinline__ u64 table_home(u64 key, u64 nslots) { return __umul64hi((key ^ (key >> 29)) * 0x9E3779B97F4A7C15ULL, nslots); }
// CAS the key into its probe sequence, keep the minimum index; returns the slot (~0: the side slot of key == EMPTY,
// ~0 - 1: table full)
__device__ __forceinline__ u64 table_insert_one(TableSlot *slots, u64 nslots, u64 *side_first, u32 *overflow, u64 key, u64 idx)
{
    if (key == CK_EMPTY_KEY) { atomicMin(side_first, idx); return ~0ULL; }
    u64 s = table_home(key, nslots);
    for (u64 probes = 0; probes < nslots; probes++) {
        const u64 prev = atomicCAS(&slots[s].key, CK_EMPTY_KEY, key);
        if (prev == CK_EMPTY_KEY || prev == key) { atomicMin(&slots[s].first, idx); return s; }
        s = s + 1 == nslots ? 0 : s + 1;
    }
    *overflow = 1;
    return ~0ULL - 1;
}

struct CanonArgs {
    const u64 *packed2;     // 2-bit arena (ck_device.cuh): record i at u64 index p2_word(offsets[i], i, p2_dbl)
    u32 p2_dbl;             // 1: doubled 32-byte-aligned layout, 0: single copy + extension (batches of short records)
    const u8 *bytes;        // normalised byte arena: record i at offsets[i]
    const u64 *offsets;     // n_records + 1 symbol offsets
    const u32 *lens;        // optional normalised lengths (else offsets[i+1] - offsets[i])
    const u32 *list;        // optional: the batch's record indices sorted by (class, length); this class's run starts at count[16]
    const u32 *count;       // device count of this class's entries (with list), else null; count[16] = first entry
    u32 n_direct;           // without list: records [0, n_direct)
    u8 *out;                // canonical ASCII arena (same offsets) or null
    u32 *out_start;         // or null
    u8 *out_strand;         // or null
    u64 *out_hash;          // or null
    u32 *scratch;           // tie-path scratch, `scratch_stride` u32 per warp (warp shape) / per CTA
    u64 scratch_stride;
    u32 smem_units;         // u32 units reserved per strand in (shared) staging memory
    u32 *xglobal;           // CLS_HUGE only: strands staged here, 2 * smem_units u32 per CTA
    u32 mode;               // bit0: forward strand only (lmsr / lmsr_index, lib/src/canonicalize.rs:5,41)
                            // bit1: aligned output arena: record i's bytes start at out_byte(offsets[i], i)
    u32 min_n, max_n;       // length range of this launch's class (checked when there is no list)
    u32 *retry;             // lane-per-record kernel: records it leaves to the warp / CTA kernels, appended per class at
    u32 *retry_counts;      // retry[retry_counts[16 + class] + atomicAdd(retry_counts + class, 1)]
    const u8 *lane_bits;    // optional: only records whose symbol lane is this kernel's BITS (the CLS_HUGE list holds every lane)
};

// ---------------------------------------------------------------------------------------------
// One 16-byte destination-aligned chunk of a record's canonical ASCII.  t0 = record-relative index of the
// chunk's first byte (negative in the record's first chunk when the record does not start on a 16-byte
// line).  Full chunks are one 128-bit store; ragged edges use naturally aligned 1/2/4/8-byte pieces because
// the neighbouring records own the rest of the line.
__device__ __forceinline__ void store_chunk(u8 *dst, int t0, u32 n, u64 lo, u64 hi)
{
    if (t0 >= 0 && (u32)t0 + 16u <= n) {
        *reinterpret_cast<uint4 *>(dst + t0) = make_uint4((u32)lo, (u32)(lo >> 32), (u32)hi, (u32)(hi >> 32));
        return;
    }
    const u32 kb = t0 < 0 ? (u32)(-t0) : 0u;
    const u32 ke = t0 < 0 ? min(16u, n + kb) : min(16u, n - (u32)t0);
    u8 *p = dst + t0;
#define CK_PIECE(k) (((k) & 8u ? hi : lo) >> (8u * ((k) & 7u)))
    u32 k = kb;
    if ((k & 1u) && k + 1 <= ke) { p[k] = (u8)CK_PIECE(k); k += 1; }
    if ((k & 2u) && k + 2 <= ke) { *reinterpret_cast<u16 *>(p + k) = (u16)CK_PIECE(k); k += 2; }
    if ((k & 4u) && k + 4 <= ke) { *reinterpret_cast<u32 *>(p + k) = (u32)CK_PIECE(k); k += 4; }
    if ((k & 8u) && k + 8 <= ke) { *reinterpret_cast<u64 *>(p + k) = hi; k += 8; }
    if (k + 8 <= ke) { *reinterpret_cast<u64 *>(p + k) = CK_PIECE(k); k += 8; }
    if (k + 4 <= ke) { *reinterpret_cast<u32 *>(p + k) = (u32)CK_PIECE(k); k += 4; }
    if (k + 2 <= ke) { *reinterpret_cast<u16 *>(p + k) = (u16)CK_PIECE(k); k += 2; }
    if (k + 1 <= ke) { p[k] = (u8)CK_PIECE(k); }
#undef CK_PIECE
}

// canonical ASCII -> global memory, generic lanes (coalesced 128-bit stores)
template <int BITS, typename G>
__device__ __forceinline__ void emit_ascii(const u32 *X, u32 n, u32 start, u8 *dst)
{
    const u32 rank = G::rank(), gs = G::size();
    const u32 a = (u32)(reinterpret_cast<uintptr_t>(dst) & 15u);
    const u32 nchunks = (n + a + 15u) >> 4;
    for (u32 c = rank; c < nchunks; c += gs) {
        const int t0 = (int)(16u * c) - (int)a;               // t0 < n always
        int ti = t0;
        if (ti < 0) { ti += (int)n; if (ti < 0) { ti %= (int)n; if (ti < 0) ti += (int)n; } }
        const u32 tt = (u32)ti;
        u32 t8 = tt + 8; if (t8 >= n) { t8 -= n; if (t8 >= n) t8 %= n; }
        const u64 lo = ascii8<BITS>(X, n, start, tt), hi = ascii8<BITS>(X, n, start, t8);
        store_chunk(dst, t0, n, lo, hi);
    }
}

// One record, both shapes.
template <int BITS, typename G>
__device__ __forceinline__ void do_record(const CanonArgs &a, u32 rec, u32 *Xf, u32 *Xr, u32 *scr, u64 *hbuf, u32 *red)
{
    const u64 off = a.offsets[rec];
    const u32 n = a.lens ? a.lens[rec] : (u32)(a.offsets[rec + 1] - off);
    if (a.list == nullptr && (n < a.min_n || n > a.max_n)) return;   // direct mode: k_classify reported it (uniform)
    if (a.lane_bits) { const u32 lb = a.lane_bits[rec]; if ((lb == 3u ? 4u : lb) != (u32)BITS) return; }
    RecordIn in;
    in.packed2 = a.packed2 ? a.packed2 + p2_word(off, rec, a.p2_dbl) : nullptr;
    in.bytes = a.bytes ? a.bytes + off : nullptr;
    in.n = n;
    stage_record<BITS, G>(in, Xf, Xr);
    RecordOut o = canonical_start<BITS, G>(Xf, Xr, n, scr, red, (a.mode & 1u) != 0);
    const u32 *X = o.strand ? Xr : Xf;
    if (a.out) emit_ascii<BITS, G>(X, n, o.start, a.out + ((a.mode & 2u) ? out_byte(off, rec) : off));
    u64 h = 0;
    if (a.out_hash) h = xxh3_canonical<BITS, G>(X, n, o.start, hbuf, red);
    if (G::rank() == 0) {
        // strand 1 start is reported in forward coordinates: canonical[j] = comp(s[(start - j) mod n])
        if (a.out_start) a.out_start[rec] = o.strand ? (n - 1 - o.start) : o.start;
        if (a.out_strand) a.out_strand[rec] = (u8)o.strand;
        if (a.out_hash) a.out_hash[rec] = h;
    }
    G::sync();      // staging memory is reused by the next record
}

template <int BITS>
__global__ void __launch_bounds__(256) k_canon_warp(CanonArgs a)
{
    extern __shared__ u32 smem[];
    typedef Grp<false> G;
    if (BITS != 2) stab_load();
    const u32 wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    u32 *Xf = smem + (size_t)wid * 2 * a.smem_units, *Xr = Xf + a.smem_units;
    const u32 gw = blockIdx.x * wpb + wid, nw = gridDim.x * wpb;
    u32 *scr = a.scratch + (size_t)gw * a.scratch_stride;
    const u32 count = a.list ? *a.count : a.n_direct;
    if (a.list) a.list += a.count[16];
    for (u32 e = gw; e < count; e += nw) {
        const u32 rec = a.list ? a.list[e] : e;
        do_record<BITS, G>(a, rec, Xf, Xr, scr, nullptr, nullptr);
    }
}

template <int BITS, bool XGLOBAL>
__global__ void __launch_bounds__(1024) k_canon_cta(CanonArgs a)
{
    extern __shared__ u32 smem[];
    __shared__ u32 red[40];
    __shared__ u64 hbuf[32 * 8];
    typedef Grp<true> G;
    if (BITS != 2) stab_load();
    u32 *Xf = XGLOBAL ? a.xglobal + (size_t)blockIdx.x * 2 * a.smem_units : smem;
    u32 *Xr = Xf + a.smem_units;
    u32 *scr = a.scratch + (size_t)blockIdx.x * a.scratch_stride;
    const u32 count = a.list ? *a.count : a.n_direct;
    if (a.list) a.list += a.count[16];
    for (u32 e = blockIdx.x; e < count; e += gridDim.x) {
        const u32 rec = a.list ? a.list[e] : e;
        do_record<BITS, G>(a, rec, Xf, Xr, scr, hbuf, red);
    }
}

// n == 0 records: canonical form is empty, strand follows the `else` arm, hash is XXH3 of "".
__global__ void k_canon_empty(CanonArgs a)
{
    const u32 count = a.list ? *a.count : a.n_direct;
    if (a.list) a.list += a.count[16];
    for (u32 e = blockIdx.x * blockDim.x + threadIdx.x; e < count; e += gridDim.x * blockDim.x) {
        const u32 rec = a.list ? a.list[e] : e;
        if (a.list == nullptr && a.offsets[rec + 1] != a.offsets[rec]) continue;
        if (a.out_start) a.out_start[rec] = 0;
        if (a.out_strand) a.out_strand[rec] = 1;
        if (a.out_hash) a.out_hash[rec] = xxh64_avalanche(sec64(56) ^ sec64(64));
    }
}

// ---------------------------------------------------------------------------------------------
// k_prepare: one warp per raw record, 512 raw bytes per warp iteration (16 per lane, two aligned 128-bit loads).
//   flags bit0 (normalise): needletail::sequence::normalize(seq, false) -- src/canonicalize.rs:24-27
//                           (whitespace dropped, acgt -> upper, t/u/U -> T, ./~ -> -, anything else -> N)
//   otherwise             : library semantics, bytes are taken as they are (lib/src/canonicalize.rs:54)
//   flags bit1            : write the (normalised) bytes of EVERY record, whatever its alphabet class (ck_dev_normalize)
// Writes lens[i], lane[i] (2, 4 or 8 bits per symbol) and the record in that lane's format:
//   lane 2 -> packed2 at word p2_word(offsets[i], i);   lanes 4/8 -> normalised bytes at offsets[i].
// Pass 1 classifies and counts through a 256-entry shared-memory table (mapped byte | keep | not-ACGT | not-16-symbol);
// pass 2 writes.  A 2-bit record without dropped bytes is packed straight from the raw bytes (the 2-bit code only reads
// bits 1-2 of a byte, which a/A, c/C, g/G, t/T/u/U share); everything else is compacted through a per-warp stage that is
// laid out congruent to the destination (mod 16 symbols / bytes), so that it leaves as aligned 128-bit pieces.
struct PrepareArgs {
    const u8 *raw; const u64 *offsets; u32 n_records; u32 flags;     // flags bit2: doubled packed2 layout
    u64 *packed2; u8 *bytes; u32 *lens; u8 *lane;
};
__device__ __forceinline__ u32 code2_of(u32 b) { return ((b >> 1) & 3u) ^ ((b >> 2) & 1u); }   // A,C,G,T -> 0..3

// 16 raw bytes starting `sh` bytes into the aligned word *w; each of the two aligned words is read only if it holds a byte
// of the record (an aligned word that does cannot leave the mapped page the record is in)
__device__ __forceinline__ uint4 prep_load16(const uint4 *w, u32 sh, bool second, bool first = true)
{
    uint4 a = make_uint4(0, 0, 0, 0), b = make_uint4(0, 0, 0, 0);
    if (first) a = __ldg(w);
    if (second) b = __ldg(w + 1);
    const u32 bs = 8u * (sh & 3u);
    uint4 q;
    switch (sh >> 2) {                                   // warp-uniform (one record per warp)
    case 0: q.x = __funnelshift_r(a.x, a.y, bs); q.y = __funnelshift_r(a.y, a.z, bs); q.z = __funnelshift_r(a.z, a.w, bs); q.w = __funnelshift_r(a.w, b.x, bs); break;
    case 1: q.x = __funnelshift_r(a.y, a.z, bs); q.y = __funnelshift_r(a.z, a.w, bs); q.z = __funnelshift_r(a.w, b.x, bs); q.w = __funnelshift_r(b.x, b.y, bs); break;
    case 2: q.x = __funnelshift_r(a.z, a.w, bs); q.y = __funnelshift_r(a.w, b.x, bs); q.z = __funnelshift_r(b.x, b.y, bs); q.w = __funnelshift_r(b.y, b.z, bs); break;
    default: q.x = __funnelshift_r(a.w, b.x, bs); q.y = __funnelshift_r(b.x, b.y, bs); q.z = __funnelshift_r(b.y, b.z, bs); q.w = __funnelshift_r(b.z, b.w, bs); break;
    }
    return q;
}
// four A/C/G/T bytes (first one in the low bits) -> their 2-bit codes in the top byte, first base in the top bits
__device__ __forceinline__ u32 prep_pack4(u32 x)
{
    const u32 c = ((x >> 1) & 0x03030303u) ^ ((x >> 2) & 0x01010101u);
    return c * 0x40100401u;      // byte k lands at bits 30 - 2k; the cross terms stay below bit 24 and never carry
}
__device__ __forceinline__ u32 prep_pack16(uint4 q)
{
    const u32 lo = __byte_perm(prep_pack4(q.w), prep_pack4(q.z), 0x0073);
    const u32 hi = __byte_perm(prep_pack4(q.y), prep_pack4(q.x), 0x0073);
    return __byte_perm(lo, hi, 0x5410);
}
__device__ __forceinline__ u32 prep_byte(const uint4 &q, int k)
{
    const u32 w = (k >> 2) == 0 ? q.x : (k >> 2) == 1 ? q.y : (k >> 2) == 2 ? q.z : q.w;
    return (w >> (8 * (k & 3))) & 0xffu;
}

// table lookups for 16 raw bytes, of which bytes [lo, hi) belong to the record: mapped bytes (0 = dropped), OR of the
// table flags, bit mask of the kept bytes.  Bytes outside [lo, hi) are looked up as 'A' (kept, no flag).
__device__ __forceinline__ void prep_lookup(const u16 *tab, uint4 q, u32 lo, u32 hi, uint4 &m, u32 &fl, u32 &keep)
{
    u32 w[4] = {q.x, q.y, q.z, q.w};
    const u32 valid = (hi >= 16 ? 0xffffu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        // nibble of `valid` -> byte mask (bit k of the nibble lands on bit 8 k, times 0xff); no carries anywhere
        const u32 vm = ((((valid >> (4 * i)) & 15u) * 0x00204081u) & 0x01010101u) * 0xffu;
        w[i] = (w[i] & vm) | (0x41414141u & ~vm);
    }
    const char *tb = reinterpret_cast<const char *>(tab);
    u32 all = 0x100u, any = 0, mm[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const u32 e0 = *reinterpret_cast<const u16 *>(tb + ((w[i] << 1) & 0x1feu));
        const u32 e1 = *reinterpret_cast<const u16 *>(tb + ((w[i] >> 7) & 0x1feu));
        const u32 e2 = *reinterpret_cast<const u16 *>(tb + ((w[i] >> 15) & 0x1feu));
        const u32 e3 = *reinterpret_cast<const u16 *>(tb + ((w[i] >> 23) & 0x1feu));
        all &= e0 & e1 & e2 & e3;
        any |= e0 | e1 | e2 | e3;
        mm[i] = __byte_perm(__byte_perm(e0, e1, 0x0040), __byte_perm(e2, e3, 0x0040), 0x5410);
    }
    m = make_uint4(mm[0], mm[1], mm[2], mm[3]);
    fl = any;
    keep = valid;
    if (!all) {                                          // some byte is dropped (normalise mode: its mapped byte is 0)
        u32 nz = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const u32 t = ((mm[i] & 0x7f7f7f7fu) + 0x7f7f7f7fu) | mm[i];
            nz |= ((((t >> 7) & 0x01010101u) * 0x01020408u) >> 24) << (4 * i);
        }
        keep = valid & nz;
    }
}

// predicated single-byte stores of the bytes of (w[0..3]) whose bit is set in `mask`, all off one base register (written
// in C the compiler recomputes a 64-bit address per store: 130 of k_prepare's 390 instructions per record were this)
template <int K> __device__ __forceinline__ void prep_store_byte(u8 *g, u32 w, u32 mask)
{
    asm volatile("{ .reg .pred q; .reg .b32 t; and.b32 t, %2, %3; setp.ne.u32 q, t, 0; @q st.global.u8 [%0+%4], %1; }"
                 :: "l"(g), "r"(w >> (8 * (K & 3))), "r"(mask), "n"(1 << K), "n"(K) : "memory");
}
__device__ __forceinline__ void prep_store_bytes(u8 *g, const u32 (&w)[4], u32 mask)
{
    prep_store_byte<0>(g, w[0], mask); prep_store_byte<1>(g, w[0], mask); prep_store_byte<2>(g, w[0], mask); prep_store_byte<3>(g, w[0], mask);
    prep_store_byte<4>(g, w[1], mask); prep_store_byte<5>(g, w[1], mask); prep_store_byte<6>(g, w[1], mask); prep_store_byte<7>(g, w[1], mask);
    prep_store_byte<8>(g, w[2], mask); prep_store_byte<9>(g, w[2], mask); prep_store_byte<10>(g, w[2], mask); prep_store_byte<11>(g, w[2], mask);
    prep_store_byte<12>(g, w[3], mask); prep_store_byte<13>(g, w[3], mask); prep_store_byte<14>(g, w[3], mask); prep_store_byte<15>(g, w[3], mask);
}

#define CK_PREP_STAGE 560u     // 16 carried bytes + 512 + slack, per warp

__global__ void __launch_bounds__(256) k_prepare(PrepareArgs a)
{
    __shared__ u16 tab[256];
    __shared__ __align__(16) u8 stage_all[8][CK_PREP_STAGE];
    const bool norm = a.flags & 1u;
    for (u32 b = threadIdx.x; b < 256; b += blockDim.x) {
        const u32 m = norm ? (u32)c_tab.norm[b] : b;
        const bool keep = norm ? m != 0 : true;
        const bool acgt = (m == 'A') | (m == 'C') | (m == 'G') | (m == 'T');
        u32 e = 0;
        if (keep) e = m | 0x100u | (acgt ? 0u : 0x200u) | ((!acgt && c_tab.code4[m] == 0xffu) ? 0x400u : 0u);
        tab[b] = (u16)e;
    }
    __syncthreads();
    const u32 lane = lane_id();
    u8 *stage = stage_all[threadIdx.x >> 5];
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (u32 rec = gw; rec < a.n_records; rec += nw) {
        const u64 off = a.offsets[rec];
        const u32 rawlen = (u32)(a.offsets[rec + 1] - off);
        const u8 *src = a.raw + off;
        u8 *dstb = a.bytes + off;
        // pass 1 walks the record in pieces congruent to the byte destination: piece w = destination bytes
        // [gbase + 16 w, + 16), i.e. record positions [16 w - A, 16 w - A + 16)
        const u32 A = (u32)((size_t)dstb & 15u);
        u8 *gbase = dstb - A;
        const u8 *srcA = src - A;
        const u32 shA = (u32)((size_t)srcA & 15u);
        const uint4 *srcA16 = reinterpret_cast<const uint4 *>(srcA - shA);
        const u32 spanA = A + rawlen;                    // pieces cover [0, spanA) in these coordinates, record at [A, spanA)
        u32 fl = 0, cnt = 0;
        uint4 m1 = make_uint4(0, 0, 0, 0);
        for (u32 base = 0; base < spanA && rawlen; base += 512) {
            const u32 p = base + 16 * lane;
            if (p < spanA) {
                const u32 lo = p < A ? A - p : 0u, hi = min(16u, spanA - p);
                const uint4 *w0 = srcA16 + (p >> 4);
                const uint4 q = prep_load16(w0, shA, p + 16 < spanA + shA, p + 16 > A + shA);
                u32 f, keep;
                prep_lookup(tab, q, lo, hi, m1, f, keep);
                fl |= f; cnt += __popc(keep);
            }
        }
        cnt = __reduce_add_sync(CK_FULL, cnt);
        fl = __reduce_or_sync(CK_FULL, fl);
        const u32 lanebits = (fl & 0x400u) ? 8u : (fl & 0x200u) ? 4u : 2u;
        if (lane == 0) { a.lens[rec] = cnt; if (a.lane) a.lane[rec] = (u8)lanebits; }
        const bool pack2 = lanebits == 2 && !(a.flags & 2u);       // flags bit1: normalised bytes for every record (ck_dev_normalize)
        if (rawlen == 0) continue;
        // pass 2: write in the lane's format
        const u32 sh = (u32)((size_t)src & 15u);
        const uint4 *src16 = reinterpret_cast<const uint4 *>(src - sh);
        const u32 span = sh + rawlen;                   // bytes from *src16 to the end of the record
        u32 *dst32 = reinterpret_cast<u32 *>(a.packed2 + p2_word(off, rec, (a.flags >> 2) & 1u));     // 16-base units in address order
        if (cnt == rawlen && pack2) {                    // nothing dropped: pack straight from the raw bytes
            for (u32 base = 0; base < rawlen; base += 512) {
                const u32 p = base + 16 * lane;
                if (p < rawlen) {
                    const u32 v = min(16u, rawlen - p);
                    u32 unit = prep_pack16(prep_load16(src16 + (p >> 4), sh, p + 16 < span));
                    if (v < 16) unit &= ~(0xffffffffu >> (2 * v));
                    dst32[p >> 4] = unit;
                }
            }
            continue;
        }
        if (cnt == rawlen && spanA <= 512) {             // nothing dropped, one piece per lane: the mapped bytes are at hand
            const u32 p = 16 * lane;
            if (p < spanA) {
                const u32 lo = p < A ? A - p : 0u, hi = min(16u, spanA - p);
                if (hi - lo == 16) *reinterpret_cast<uint4 *>(gbase + p) = m1;
                else {                                   // first / last piece: whole 32-bit words, then single bytes
                    const u32 valid = (hi >= 16 ? 0xffffu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
                    const u32 w[4] = {m1.x, m1.y, m1.z, m1.w};
                    u8 *g = gbase + p;
                    u32 vb = valid;                      // bytes left to the single-byte stores
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        if (((valid >> (4 * i)) & 15u) == 15u) { *reinterpret_cast<u32 *>(g + 4 * i) = w[i]; vb &= ~(15u << (4 * i)); }
                    prep_store_bytes(g, w, vb);
                }
            }
            continue;
        }
        // general path: compact the kept bytes through the stage, laid out congruent to the destination
        u32 S = pack2 ? 0u : A;                          // stage[S ..) <-> next symbol to place
        u32 done = 0;                                    // 2-bit: full units stored; bytes: bytes stored
        for (u32 base = 0; base < rawlen; base += 512) {
            const u32 p = base + 16 * lane;
            uint4 m = make_uint4(0, 0, 0, 0);
            u32 mask = 0;
            if (p < rawlen) {
                u32 f;
                prep_lookup(tab, prep_load16(src16 + (p >> 4), sh, p + 16 < span), 0u, min(16u, rawlen - p), m, f, mask);
            }
            // exclusive scan of the kept counts
            const u32 kc = __popc(mask);
            u32 incl = kc;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const u32 t = __shfl_up_sync(CK_FULL, incl, d); if (lane >= (u32)d) incl += t; }
            const u32 T = __shfl_sync(CK_FULL, incl, 31);
            u32 idx = S + incl - kc;
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 16; k++)
                if ((mask >> k) & 1u) stage[idx++] = (u8)prep_byte(m, k);
            __syncwarp();
            const u32 fill = S + T;                                  // stage[0, fill) is valid
            if (pack2) {
                const u32 U = fill >> 4;
                for (u32 j = lane; j < U; j += 32) dst32[done + j] = prep_pack16(*reinterpret_cast<const uint4 *>(stage + 16 * j));
                const u32 r = fill & 15u;
                u8 c = 0;
                if (lane < r) c = stage[16 * U + lane];
                __syncwarp();
                if (lane < r) stage[lane] = c;
                done += U; S = r;
            } else {
                u8 *g = dstb + done - S;                             // 16-byte aligned, congruent to the stage
                for (u32 w = lane; 16 * w < fill; w += 32) {
                    const u32 lo = max(16 * w, S), hi = min(16 * w + 16, fill);
                    if (hi - lo == 16) *reinterpret_cast<uint4 *>(g + 16 * w) = *reinterpret_cast<const uint4 *>(stage + 16 * w);
                    else for (u32 i = lo; i < hi; i++) g[i] = stage[i];
                }
                done += T; S = (u32)((size_t)(dstb + done) & 15u);
            }
        }
        __syncwarp();
        if (pack2 && S && lane == 0)
            dst32[done] = prep_pack16(*reinterpret_cast<const uint4 *>(stage)) & ~(0xffffffffu >> (2 * S));
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// k_classify: class of every record.  With a class promise (direct_mask) records outside it are counted as
// "left unprocessed"; otherwise every record gets a sort key (class << 8 | length bin) and the classes are counted:
// a radix sort of (key, index) then yields ONE index list in which each class is a contiguous run ordered by length,
// so the lanes of a lane-per-record warp walk records of (nearly) equal length.
struct ClassifyArgs {
    const u64 *offsets; const u32 *lens; const u8 *lane;   // lane == null: every record is 2-bit
    u32 n_records;
    u32 *keys, *vals;  // n_records sort keys / record indices (list mode)
    u32 *counts;       // 16 class counters (zeroed by the caller), followed by 16 run starts (k_list_starts)
    u32 direct_mask;   // != 0: no keys are written (the classes of the mask run over all records directly);
                       // records of any other class are counted in counts[CLS_HUGE] = "left unprocessed"
    u32 window_shift;  // < 32: the lane-kernel classes are keyed (index >> window_shift, length bin) instead of (class, length bin):
    u32 top_bit;       //       the records a warp walks together then come from one window of the arenas, which L2 can hold;
                       //       every other class gets bit `top_bit` set and keeps (class, bin), i.e. sorts behind them
};
__global__ void __launch_bounds__(256) k_classify(ClassifyArgs a)
{
    __shared__ u32 cnt[16];                                    // per-CTA class counts: one global atomic per class and CTA
    if (threadIdx.x < 16) cnt[threadIdx.x] = 0;
    __syncthreads();
    const u32 nthreads = gridDim.x * blockDim.x;
    const u32 rounds = (a.n_records + nthreads - 1) / nthreads;
    for (u32 r = 0; r < rounds; r++) {
        const u32 i = r * nthreads + blockIdx.x * blockDim.x + threadIdx.x;
        int cls = -1;
        u32 n = 0;
        if (i < a.n_records) {
            n = a.lens ? a.lens[i] : (u32)(a.offsets[i + 1] - a.offsets[i]);
            const u32 bits = a.lane ? a.lane[i] : 2u;
            if (n == 0) cls = CLS_EMPTY;
            else if (bits == 2) cls = n <= cls_max_n(CLS_W2S) ? CLS_W2S : n <= cls_max_n(CLS_W2M) ? CLS_W2M
                                    : n <= cls_max_n(CLS_W2L) ? CLS_W2L : n <= cls_max_n(CLS_W2X) ? CLS_W2X
                                    : n <= cls_max_n(CLS_C2A) ? CLS_C2A : n <= cls_max_n(CLS_C2B) ? CLS_C2B : CLS_HUGE;
            else if (bits == 4 || bits == 3) cls = n <= cls_max_n(CLS_W4) ? CLS_W4 : n <= cls_max_n(CLS_C4) ? CLS_C4 : CLS_HUGE;
            else cls = n <= cls_max_n(CLS_W8) ? CLS_W8 : n <= cls_max_n(CLS_C8) ? CLS_C8 : CLS_HUGE;
        }
        if (a.direct_mask) {
            const u32 m = __ballot_sync(CK_FULL, cls >= 0 && !((a.direct_mask >> cls) & 1u));
            if (m && lane_id() == (u32)(__ffs(m) - 1)) atomicAdd(cnt + CLS_HUGE, __popc(m));
            continue;
        }
        if (cls >= 0) {
            // key = (rank of the class in list order) : (length on a 1/4-octave log scale: lanes of a warp differ by < 19 % in
            // length, and a bin is dense enough that its consecutive members sit close together in the arenas; measured on
            // config 2: 1/32 octave 9.7 ms, 1/8 octave 8.6 ms, 1/4 octave 8.4 ms)
            const u32 msb = 31u - __clz(n | 1u);
            const u32 bin = (msb << 5) | ((((n << (31u - msb)) >> 29) & 3u) << 3);
            u32 key = (cls_rank(cls) << 10) | bin;
            if (a.window_shift < 32u) {
                const bool lane_cls = cls == CLS_W2S || cls == CLS_W2M || cls == CLS_W2L || cls == CLS_W2X;
                const u32 q = (msb << 2) | (((n << (31u - msb)) >> 29) & 3u);            // quarter octaves; n <= 8192: q <= 52
                key = lane_cls ? (((i >> a.window_shift) << 5) | (q > 28u ? q - 28u : 0u)) : (key | (1u << a.top_bit));
            }
            a.keys[i] = key; a.vals[i] = i;
        }
        // warp-aggregated counting: one shared-memory atomic per (warp, class present)
        u32 todo = __ballot_sync(CK_FULL, cls >= 0);
        while (todo) {
            const int c = __shfl_sync(CK_FULL, cls, __ffs(todo) - 1);
            const u32 m = __ballot_sync(CK_FULL, cls == c);
            if (lane_id() == (u32)(__ffs(m) - 1)) atomicAdd(cnt + c, __popc(m));
            todo &= ~m;
        }
    }
    __syncthreads();
    if (threadIdx.x < 16 && cnt[threadIdx.x]) atomicAdd(a.counts + threadIdx.x, cnt[threadIdx.x]);
}
// run starts of the sorted index list (classes in cls_rank order).  Layout of the 64 counters:
//   [0, 12)  records per class        [12]  records of the lane-kernel classes together (one launch)   [13] of the long 2-bit classes
//   [16, 28) first entry per class    [28]  first entry of the lane-kernel classes                     [29] of the long 2-bit classes
//   [32, 44) retry entries per class  [48, 60)  first retry entry per class (= first entry of the class)
__global__ void k_list_starts(u32 *counts)
{
    if (threadIdx.x == 0) {
        u32 s = 0;
        for (u32 r = 0; r < (u32)CLS_COUNT; r++) {
            const int c = cls_of_rank(r);
            counts[16 + c] = s; counts[48 + c] = s;
            s += counts[c];
        }
        counts[12] = counts[CLS_W2S] + counts[CLS_W2M] + counts[CLS_W2L] + counts[CLS_W2X];
        counts[28] = counts[16 + CLS_W2S];
        counts[13] = counts[CLS_C2A] + counts[CLS_C2B];            // the long 2-bit classes together (k_canon_seg)
        counts[29] = counts[16 + CLS_C2A];
    }
}

// k_extend_packed2: complete every packed record of the arena (ck_device.cuh, "packed2 arena"): units up to `last` hold
// the bases S[b mod n], last = the unit of base 2 n + 143 (at least jn + 5, jn = n >> 4) -- the record twice, then some.
//   dense == null : the packer (k_prepare / k_synth_packed2) wrote the first copy in place; units jn .. last are appended
//                   (the partial unit jn keeps its real bases);
//   dense != null : CK_F_PACKED_IN -- the host packer's dense layout (record i at 64-bit word (offsets[i] >> 5) + i, first
//                   copy only, ck_host_pack.cpp) is spread into the arena: units 0 .. last.
// One warp per record, one lane per destination unit; every source is a unit of the first copy (in place, unit jn is read
// while another lane completes it: the bits a reader uses are the same before and after).
__device__ __forceinline__ u32 p2_last_unit(u32 n) { return max((2u * n + 143u) >> 4, (n >> 4) + 5u); }
__device__ __forceinline__ void extend_one(u64 *packed2, const u64 *offsets, const u32 *lens, u32 i, const u64 *dense, u32 dbl, u32 lane)
{
    const u64 off = offsets[i];
    const u32 n = lens ? lens[i] : (u32)(offsets[i + 1] - off);
    if (n == 0) return;
    u32 *U = reinterpret_cast<u32 *>(packed2 + p2_word(off, i, dbl));
    const u32 *S = dense ? reinterpret_cast<const u32 *>(dense + (off >> 5) + i) : U;
    const u32 jn = n >> 4, last = dbl ? p2_last_unit(n) : jn + 4;          // single copy: the circular extension only
    if (n >= 80) {
        for (u32 j = (dense ? 0u : jn) + lane; j <= last; j += 32) {
            const u32 r = (16u * j) % n;                          // first base of the unit, modulo n
            const u32 q = r >> 4, sh = 2u * (r & 15u);
            u32 w = __funnelshift_l(__ldcg(S + q + 1), __ldcg(S + q), sh);
            if (r + 16u > n) {                                    // the seam: k bases of the tail, then the head
                const u32 k = n - r;
                w = (w & ~(0xffffffffu >> (2u * k))) | (__ldcg(S) >> (2u * k));
            }
            U[j] = w;
        }
    } else {
        // tiny records: base by base (at most 20 units)
        for (u32 j = (dense ? 0u : jn) + lane; j <= last; j += 32) {
            u32 v = 0;
            for (u32 b = 0; b < 16; b++) {
                const u32 t = (16 * j + b) % n;
                v = (v << 2) | ((__ldcg(S + (t >> 4)) >> (30 - 2 * (t & 15))) & 3u);
            }
            __syncwarp(__activemask());
            U[j] = v;
        }
    }
    __syncwarp();
}
__global__ void __launch_bounds__(256) k_extend_packed2(u64 *packed2, const u64 *offsets, const u32 *lens, const u8 *lane_bits, u32 n_records,
                                                        const u64 *dense, u32 dbl)
{
    const u32 lane = lane_id();
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    if (n_records < 65536u) {                                     // small batches: a warp per record, all of them at once
        for (u32 i = gw; i < n_records; i += nw) {
            if (lane_bits && lane_bits[i] != 2) continue;
            extend_one(packed2, offsets, lens, i, dense, dbl, lane);
        }
        return;
    }
    // large batches: a warp looks at the lane tags of 32 records at once, so that a batch without 2-bit records (config 3:
    // 5 M IUPAC records) costs 32 times fewer dependent loads (0.2 ms -> 10 us)
    for (u32 i0 = 32u * gw; i0 < n_records; i0 += 32u * nw) {
        const u32 ii = i0 + lane;
        u32 m = __ballot_sync(CK_FULL, ii < n_records && (!lane_bits || lane_bits[ii] == 2));
        while (m) {
            const u32 i = i0 + (u32)__ffs(m) - 1u;
            m &= m - 1u;
            extend_one(packed2, offsets, lens, i, dense, dbl, lane);
        }
    }
}

// CK_F_PACKED_IN, byte-level lanes: the (normalised) bytes of the records whose lane is not 2 arrive concatenated in record
// order; put record i's bytes at offsets[i] of the byte arena, where the byte-lane kernels look for them.
__global__ void __launch_bounds__(256) k_scatter_lane_bytes(const u8 *lane_bytes, const u64 *lane_offsets, const u64 *offsets, const u32 *lens,
                                                            const u8 *lane_bits, u32 n_records, u8 *bytes)
{
    const u32 lane = lane_id();
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (u32 i = gw; i < n_records; i += nw) {
        if (lane_bits[i] == 2) continue;
        const u8 *src = lane_bytes + lane_offsets[i];
        u8 *dst = bytes + offsets[i];
        const u32 n = lens[i];
        for (u32 k = lane; k < n; k += 32) dst[k] = src[k];
    }
}

// ---------------------------------------------------------------------------------------------
// First-occurrence table (replaces HashMap<u64, String, NoHash>, src/uniq.rs:27,47-48,66).
// slot = {key, first}; key == EMPTY_KEY marks a free slot, and the one real key equal to EMPTY_KEY is
// kept in a side slot, so every u64 stays a legal XXH3 value.  Keeping the MIN input index per key
// reproduces "first record seen wins" of the serial consumer for any insertion order.
struct TableArgs {
    TableSlot *slots; u64 nslots;        // slots of the table (any number)
    u64 *side_first;                     // first index of key == EMPTY_KEY
    const u64 *hash; const u64 *index;   // index == null: base_index + i
    u32 stride;                          // elements between consecutive records in hash / index (2: interleaved pairs)
    u64 base_index; u32 n;
    u64 *slot_of;                        // out: slot found per record (for k_table_first)
    u64 *first_out;                      // out (k_table_first)
    u32 *overflow;                       // set if the table is full
    u64 *keys;                           // optional: += keys this launch adds to the table (a context's table; ck_uniq_grow)
};
__global__ void __launch_bounds__(256) k_table_insert(TableArgs a)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const u64 key = a.hash[(size_t)i * a.stride];
    const u64 idx = a.index ? a.index[(size_t)i * a.stride] : a.base_index + i;
    if (idx == ~0ULL) { a.slot_of[i] = ~0ULL - 1; return; }     // padding of a fixed-capacity exchange bucket (k_owner_pad)
    if (key == CK_EMPTY_KEY) { atomicMin(a.side_first, idx); a.slot_of[i] = ~0ULL; return; }
    u64 s = table_home(key, a.nslots);
    for (u64 probes = 0; probes < a.nslots; probes++) {
        u64 prev = atomicCAS(&a.slots[s].key, CK_EMPTY_KEY, key);
        if (prev == CK_EMPTY_KEY || prev == key) {
            atomicMin(&a.slots[s].first, idx);
            a.slot_of[i] = s;
            if (a.keys && prev == CK_EMPTY_KEY) {     // claimed a free slot: one add per group of lanes that got here together
                const u32 m = __activemask();
                if ((threadIdx.x & 31) == (u32)(__ffs(m) - 1)) atomicAdd(a.keys, (u64)__popc(m));
            }
            return;
        }
        s = s + 1 == a.nslots ? 0 : s + 1;
    }
    *a.overflow = 1; a.slot_of[i] = ~0ULL - 1;
}
__global__ void __launch_bounds__(256) k_table_first(TableArgs a)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const u64 s = a.slot_of[i];
    a.first_out[i] = s == ~0ULL ? *a.side_first : (s == ~0ULL - 1 ? ~0ULL : a.slots[s].first);
}
__global__ void k_table_clear(TableSlot *slots, u64 n, u64 *side_first)
{
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        slots[i].key = CK_EMPTY_KEY; slots[i].first = ~0ULL;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *side_first = ~0ULL;
}
// Growth of a context's table (ck_uniq_grow): every key of the old table moves to its home in the new one, with the same
// probing.  Keys are unique, so each move claims a free slot and carries its minimum index over as it is; the new table
// starts all ones (empty key, empty first) and is larger than the old one, so the probe always ends.
__global__ void __launch_bounds__(256) k_table_rehash(const TableSlot *old, u64 old_slots, TableSlot *slots, u64 nslots)
{
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < old_slots; i += (u64)gridDim.x * blockDim.x) {
        const TableSlot e = old[i];
        if (e.key == CK_EMPTY_KEY) continue;
        u64 s = table_home(e.key, nslots);
        while (atomicCAS(&slots[s].key, CK_EMPTY_KEY, e.key) != CK_EMPTY_KEY) s = s + 1 == nslots ? 0 : s + 1;
        slots[s].first = e.first;
    }
}

// ---------------------------------------------------------------------------------------------
// Order-preserving compaction of the survivors (SURVEY K6; src/uniq.rs:47-61: only first occurrences are written, in input
// order): flags -> cub::DeviceSelect (indices of the survivors, increasing) -> their lengths (rounded up to 16) -> exclusive
// scan -> gather of the canonical bytes into a compact arena, survivor k at compact_off[k].
__global__ void __launch_bounds__(256) k_survivor_flags(const u64 *first, u64 base_index, u32 n, u8 *flags)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = first[i] == base_index + i;
}
__global__ void __launch_bounds__(256) k_survivor_lens(const u32 *sel, const u32 *n_sel, const u32 *lens, u32 n, u64 *len16)
{
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > n) return;
    len16[k] = k < *n_sel ? (u64)((lens[sel[k]] + 15u) & ~15u) : 0ull;
}
__global__ void __launch_bounds__(256) k_gather_survivors(const u32 *sel, const u32 *n_sel, const u32 *lens, const u64 *offsets, const u8 *out,
                                                          u32 aligned, const u64 *compact_off, u8 *compact)
{
    const u32 lane = lane_id();
    const u32 gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const u32 ns = *n_sel;
    for (u32 k = gw; k < ns; k += nw) {
        const u32 rec = sel[k], n = lens[rec];
        const u64 off = offsets[rec];
        const u8 *src = out + (aligned ? out_byte(off, rec) : off);
        u8 *dst = compact + compact_off[k];                       // 16-byte aligned
        if (aligned) {
            for (u32 c = lane; 16u * c < n; c += 32) reinterpret_cast<uint4 *>(dst)[c] = reinterpret_cast<const uint4 *>(src)[c];
        } else {
            for (u32 b = lane; b < n; b += 32) dst[b] = src[b];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Hash-range partition for multi-GPU uniq (SURVEY section 8e): owner = floor(hash * world / 2^64).  Two passes over
// the local hashes: counts per owner, then a scatter of (hash, global index) into per-owner runs of the send
// buffers (order inside a run is free: the owner keeps the minimum index per key).  pos[i] = where record i went, so
// the answer that comes back in send-buffer order can be gathered back into input order.
struct OwnerArgs {
    const u64 *hash; u32 n; u32 world; u64 base_index;
    u32 *counts;       // [world] records per owner, then [world] scatter cursors (both zeroed by the caller)
    u64 *send_pairs; u32 *pos;   // send buffer: (hash, global index) pairs, 16 bytes per record
};
// floor(hash * world / 2^64) on the top 32 bits.  Written with __umulhi: nvcc 12.9 turned the 64-bit form
// (((h >> 32) * world) >> 32), used as a shared-memory index, into a low multiply (every record went to owner 0).
__device__ __forceinline__ u32 owner_of_hash(u64 h, u32 world) { return __umulhi((u32)(h >> 32), world); }
__global__ void __launch_bounds__(256) k_owner_count(OwnerArgs a)
{
    __shared__ u32 cnt[32];
    if (threadIdx.x < 32) cnt[threadIdx.x] = 0;
    __syncthreads();
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += gridDim.x * blockDim.x)
        atomicAdd(cnt + owner_of_hash(a.hash[i], a.world), 1u);
    __syncthreads();
    if (threadIdx.x < a.world && cnt[threadIdx.x]) atomicAdd(a.counts + threadIdx.x, cnt[threadIdx.x]);
}
__global__ void __launch_bounds__(256) k_owner_scatter(OwnerArgs a)
{
    __shared__ u32 cnt[32], basep[32];
    const u32 per = (a.n + gridDim.x - 1) / gridDim.x;         // this CTA's contiguous slice
    const u32 lo = min(a.n, blockIdx.x * per), hi = min(a.n, lo + per);
    if (threadIdx.x < 32) cnt[threadIdx.x] = 0;
    __syncthreads();
    for (u32 i = lo + threadIdx.x; i < hi; i += blockDim.x) atomicAdd(cnt + owner_of_hash(a.hash[i], a.world), 1u);
    __syncthreads();
    if (threadIdx.x < a.world) {
        u32 start = 0;                                         // run start of this owner = counts of the owners below it
        for (u32 o = 0; o < threadIdx.x; o++) start += a.counts[o];
        basep[threadIdx.x] = start + atomicAdd(a.counts + a.world + threadIdx.x, cnt[threadIdx.x]);
        cnt[threadIdx.x] = 0;
    }
    __syncthreads();
    for (u32 i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const u64 h = a.hash[i];
        const u32 o = owner_of_hash(h, a.world);
        const u32 p = basep[o] + atomicAdd(cnt + o, 1u);
        reinterpret_cast<ulonglong2 *>(a.send_pairs)[p] = make_ulonglong2(h, a.base_index + i);
        a.pos[i] = p;
    }
}


// The same partition into FIXED-capacity buckets (bucket o = send_pairs[o * cap, (o + 1) * cap)): one pass, no counts to
// exchange and nothing for the host to wait for -- the buckets go out as an equal-split all-to-all.  XXH3 keys spread
// evenly, so cap = n / world plus a few standard deviations wastes well under 1 % of the volume; a bucket that would
// overflow (a heavily duplicated key set) raises *overflow and the caller repeats the batch through the exact path.
struct OwnerPadArgs {
    const u64 *hash; u32 n; u32 world; u64 base_index; u32 cap;
    u32 *cursors;      // [world] records placed per bucket so far (zeroed by the caller), [world] = overflow flag
    u64 *send_pairs; u32 *pos;
};
__global__ void __launch_bounds__(256) k_owner_scatter_padded(OwnerPadArgs a)
{
    __shared__ u32 cnt[32], basep[32];
    const u32 per = (a.n + gridDim.x - 1) / gridDim.x;
    const u32 lo = min(a.n, blockIdx.x * per), hi = min(a.n, lo + per);
    if (threadIdx.x < 32) cnt[threadIdx.x] = 0;
    __syncthreads();
    for (u32 i = lo + threadIdx.x; i < hi; i += blockDim.x) atomicAdd(cnt + owner_of_hash(a.hash[i], a.world), 1u);
    __syncthreads();
    if (threadIdx.x < a.world) {
        basep[threadIdx.x] = cnt[threadIdx.x] ? atomicAdd(a.cursors + threadIdx.x, cnt[threadIdx.x]) : 0u;
        if (basep[threadIdx.x] + cnt[threadIdx.x] > a.cap) a.cursors[a.world] = 1u;
        cnt[threadIdx.x] = 0;
    }
    __syncthreads();
    for (u32 i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const u64 h = a.hash[i];
        const u32 o = owner_of_hash(h, a.world);
        const u32 k = basep[o] + atomicAdd(cnt + o, 1u);
        u32 p = 0xffffffffu;
        if (k < a.cap) {
            p = o * a.cap + k;
            reinterpret_cast<ulonglong2 *>(a.send_pairs)[p] = make_ulonglong2(h, a.base_index + i);
        }
        a.pos[i] = p;
    }
}
// the unused tail of every bucket: index ~0 = "no record" (k_table_insert skips it)
__global__ void __launch_bounds__(256) k_owner_pad(OwnerPadArgs a)
{
    const u32 o = blockIdx.y;
    const u32 used = min(a.cursors[o], a.cap);
    for (u32 k = used + blockIdx.x * blockDim.x + threadIdx.x; k < a.cap; k += gridDim.x * blockDim.x)
        reinterpret_cast<ulonglong2 *>(a.send_pairs)[(size_t)o * a.cap + k] = make_ulonglong2(0ULL, ~0ULL);
}

// ---------------------------------------------------------------------------------------------
// The exchange fused into the two kernels around it, over peer-mapped memory (NVLink / NVSwitch loads and stores):
//   k_owner_scatter_peers  the partition writes every (hash, index) pair straight into its owner's receive buffer
//                          (region `rank` of it, same fixed capacity as above) and pads the tail of that region;
//   k_table_first_peers    the owner's query writes every answer straight into the asking rank's return buffer, in the
//                          order the pairs were sent, so that pos[] gathers them back into input order.
// Between the two sit one device-side barrier each (all pairs have landed / all answers have landed); no collective
// moves data and no send or receive staging buffer exists.
struct PeerPtrs { u64 *p[32]; };
struct OwnerPeerArgs {
    const u64 *hash; u32 n; u32 world; u32 rank; u64 base_index; u32 cap;
    u32 *cursors;      // [world] + overflow flag, zeroed by the caller
    u32 *pos;
    PeerPtrs recv;     // recv.p[o] = owner o's receive buffer: world regions of cap (hash, index) pairs
};
// Tiles of 2048 records are bucketed in shared memory first, so that what crosses NVLink are runs of consecutive 16-byte
// pairs per owner (a tile holds ~256 pairs per owner at 8 ranks) written by consecutive threads, not single pairs
// scattered over eight destinations (8 GPUs, 12.5 M records: 0.55 ms with per-record remote stores).
#define CK_SCAT_TILE 2048u
__global__ void __launch_bounds__(256) k_owner_scatter_peers(OwnerPeerArgs a)
{
    __shared__ ulonglong2 stage[CK_SCAT_TILE];
    __shared__ u8 own[CK_SCAT_TILE];
    __shared__ u32 cnt[32], start[33], basep[32], fill[32];
    const u32 per = (a.n + gridDim.x - 1) / gridDim.x;
    const u32 lo = min(a.n, blockIdx.x * per), hi = min(a.n, lo + per);
    for (u32 tile = lo; tile < hi; tile += CK_SCAT_TILE) {
        const u32 tn = min(hi - tile, CK_SCAT_TILE);
        if (threadIdx.x < 32) { cnt[threadIdx.x] = 0; fill[threadIdx.x] = 0; }
        __syncthreads();
        u64 hreg[CK_SCAT_TILE / 256];
        u32 oreg[CK_SCAT_TILE / 256];
#pragma unroll
        for (u32 k = 0; k < CK_SCAT_TILE / 256; k++) {
            const u32 j = threadIdx.x + 256u * k;
            if (j < tn) {
                hreg[k] = a.hash[tile + j];
                oreg[k] = owner_of_hash(hreg[k], a.world);
                atomicAdd(cnt + oreg[k], 1u);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            u32 acc = 0;
            for (u32 o = 0; o < a.world; o++) { start[o] = acc; acc += cnt[o]; }
            start[a.world] = acc;
        }
        if (threadIdx.x < a.world) {
            const u32 c = cnt[threadIdx.x];
            basep[threadIdx.x] = c ? atomicAdd(a.cursors + threadIdx.x, c) : 0u;
            if (basep[threadIdx.x] + c > a.cap) a.cursors[a.world] = 1u;
        }
        __syncthreads();
#pragma unroll
        for (u32 k = 0; k < CK_SCAT_TILE / 256; k++) {
            const u32 j = threadIdx.x + 256u * k;
            if (j < tn) {
                const u32 o = oreg[k];
                const u32 r = atomicAdd(fill + o, 1u);
                const u32 slot = start[o] + r;
                stage[slot] = make_ulonglong2(hreg[k], a.base_index + tile + j);
                own[slot] = (u8)o;
                const u32 g = basep[o] + r;
                a.pos[tile + j] = g < a.cap ? o * a.cap + g : 0xffffffffu;
            }
        }
        __syncthreads();
        for (u32 sl = threadIdx.x; sl < tn; sl += 256) {
            const u32 o = own[sl];
            const u32 g = basep[o] + (sl - start[o]);
            if (g < a.cap) reinterpret_cast<ulonglong2 *>(a.recv.p[o])[(size_t)a.rank * a.cap + g] = stage[sl];
        }
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) k_owner_pad_peers(OwnerPeerArgs a)
{
    const u32 o = blockIdx.y;
    const u32 used = min(a.cursors[o], a.cap);
    ulonglong2 *dst = reinterpret_cast<ulonglong2 *>(a.recv.p[o]) + (size_t)a.rank * a.cap;
    for (u32 k = used + blockIdx.x * blockDim.x + threadIdx.x; k < a.cap; k += gridDim.x * blockDim.x)
        dst[k] = make_ulonglong2(0ULL, ~0ULL);
}
struct FirstPeerArgs {
    const TableSlot *slots; const u64 *side_first; const u64 *slot_of;
    u32 world; u32 rank; u32 cap;
    PeerPtrs ret;      // ret.p[s] = rank s's return buffer: world regions of cap first indices (region = owner)
};
__global__ void __launch_bounds__(256) k_table_first_peers(FirstPeerArgs a)
{
    const u32 s = blockIdx.y;                                  // asking rank: region s of the local receive buffer
    u64 *dst = a.ret.p[s] + (size_t)a.rank * a.cap;
    const u64 *slot_of = a.slot_of + (size_t)s * a.cap;
    for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < a.cap; k += gridDim.x * blockDim.x) {
        const u64 sl = slot_of[k];
        dst[k] = sl == ~0ULL ? *a.side_first : (sl == ~0ULL - 1 ? ~0ULL : a.slots[sl].first);
    }
}
// Barrier over the ranks of a peer group (one process per GPU, every rank's exchange block mapped into every process by
// CUDA IPC): thread t tells rank t "rank `rank` has reached epoch e of barrier b" -- and, when `send_counts` is given, how
// many (hash, index) pairs it has stored into rank t's receive region -- and then waits until rank t has said the same
// here.  Launched behind the kernel whose remote stores it publishes: those stores were performed before this kernel
// started (stream order), the system-scope fence + release store order them before the flag.  Every rank must launch it the
// same number of times per barrier id; ranks must run on different GPUs (a rank that spins here waits for its peers' kernels).
// Block layout (u64 words): [0, 128) flags[barrier id 0..3][src rank]; [128, 192) counts[slot 0..1][src rank].
struct PeerBlockPtrs { u64 *p[32]; };
#define CK_PEER_FLAG_WORDS 128u
#define CK_PEER_HEADER_BYTES 4096u
__global__ void k_peer_barrier(PeerBlockPtrs blocks, u32 world, u32 rank, u32 barrier_id, u64 epoch, const u32 *send_counts, u32 count_slot)
{
    const u32 t = threadIdx.x;
    if (t >= world) return;
    if (send_counts) blocks.p[t][CK_PEER_FLAG_WORDS + 32u * count_slot + rank] = send_counts[t];
    __threadfence_system();
    u64 *theirs = blocks.p[t] + barrier_id * 32u + rank;
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(theirs), "l"(epoch) : "memory");
    const u64 *mine = blocks.p[rank] + barrier_id * 32u + t;
    u64 seen;
    do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(mine) : "memory");
    } while (seen < epoch);
}
// Owner side of the fused exchange with EXACT counts (no padding, no overflow: a region holds up to `cap` = every record a
// sender can have): insert the pairs of all regions, region s holding counts[s] of them; then answer them into the asking
// ranks' return regions.
struct RegionArgs {
    TableSlot *slots; u64 nslots; u64 *side_first; u32 *overflow;
    const u64 *recv;        // local receive buffer: world regions of cap (hash, index) pairs
    const u64 *counts;      // counts[s] (low 32 bits) = pairs in region s
    u64 *slot_of;           // world * cap entries
    u32 world, rank, cap;
    PeerBlockPtrs ret;      // ret.p[s] = rank s's return buffer: world regions of cap first indices (region = owner)
};
__global__ void __launch_bounds__(256) k_table_insert_regions(RegionArgs a)
{
    const u32 s = blockIdx.y;
    const u32 cnt = (u32)a.counts[s];
    const ulonglong2 *pairs = reinterpret_cast<const ulonglong2 *>(a.recv) + (size_t)s * a.cap;
    u64 *slot_of = a.slot_of + (size_t)s * a.cap;
    for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < cnt; k += gridDim.x * blockDim.x) {
        const ulonglong2 pr = pairs[k];
        const u64 key = pr.x, idx = pr.y;
        if (key == CK_EMPTY_KEY) { atomicMin(a.side_first, idx); slot_of[k] = ~0ULL; continue; }
        u64 sl = table_home(key, a.nslots);
        u64 found = ~0ULL - 1;
        for (u64 probes = 0; probes < a.nslots; probes++) {
            const u64 prev = atomicCAS(&a.slots[sl].key, CK_EMPTY_KEY, key);
            if (prev == CK_EMPTY_KEY || prev == key) { atomicMin(&a.slots[sl].first, idx); found = sl; break; }
            sl = sl + 1 == a.nslots ? 0 : sl + 1;
        }
        if (found == ~0ULL - 1) *a.overflow = 1;
        slot_of[k] = found;
    }
}
__global__ void __launch_bounds__(256) k_table_first_regions(RegionArgs a)
{
    const u32 s = blockIdx.y;
    const u32 cnt = (u32)a.counts[s];
    u64 *dst = a.ret.p[s] + (size_t)a.rank * a.cap;
    const u64 *slot_of = a.slot_of + (size_t)s * a.cap;
    for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < cnt; k += gridDim.x * blockDim.x) {
        const u64 sl = slot_of[k];
        dst[k] = sl == ~0ULL ? *a.side_first : (sl == ~0ULL - 1 ? ~0ULL : a.slots[sl].first);
    }
}

// first_index[i] = ret[pos[i]]: the answers, which arrive in send order, back in input order
__global__ void __launch_bounds__(256) k_gather_first(const u64 *ret, const u32 *pos, u32 n, u64 *out)
{
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u32 p = pos[i];
        out[i] = p == 0xffffffffu ? ~0ULL : ret[p];
    }
}

}  // namespace ck
