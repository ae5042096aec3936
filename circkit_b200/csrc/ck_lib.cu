// ck_lib.cu -- C ABI (include/circkit_b200.h) over the kernels in ck_kernels.cuh.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "../../include/circkit_b200.h"
#include "ck_kernels.cuh"
#include "ck_warp2.cuh"
#include "ck_lane2.cuh"
#include "ck_stream2.cuh"
#include "ck_stream3.cuh"
#include "ck_seg2.cuh"
#include "ck_lane4.cuh"
#include "ck_synth.cuh"
#include "ck_monomerize.cuh"
#include "ck_fasta.cuh"
#include "ck_deflate.cuh"
#include "ck_bzip2.cuh"

using namespace ck;

namespace {

thread_local std::string g_init_error;

inline const u64 *U(const uint64_t *p) { return reinterpret_cast<const u64 *>(p); }
inline u64 *U(uint64_t *p) { return reinterpret_cast<u64 *>(p); }

struct ClsCfg { int bits; bool cta; u32 threads; u32 ctas_per_sm; };
const ClsCfg kCls[CLS_COUNT] = {
    {2, false, 256, 8},   // CLS_W2S
    {2, false, 256, 6},   // CLS_W2M
    {2, true, 512, 4},    // CLS_C2A
    {2, true, 1024, 1},   // CLS_C2B
    {4, false, 256, 32},  // CLS_W4
    {4, true, 1024, 1},   // CLS_C4
    {8, false, 256, 32},  // CLS_W8
    {8, true, 1024, 1},   // CLS_C8
    {0, true, 0, 0},      // CLS_HUGE (handled separately)
    {0, false, 256, 1},   // CLS_EMPTY
    {2, false, 256, 6},   // CLS_W2L
    {2, false, 256, 6},   // CLS_W2X
};

u32 cls_units(int c)
{
    const u32 n = cls_max_n(c);
    switch (kCls[c].bits) {
    case 2: return strand_units<2>(n);
    case 4: return strand_units<4>(n);
    default: return strand_units<8>(n);
    }
}
u64 cls_tie_words(int c)
{
    const u64 n = cls_max_n(c);
    switch (kCls[c].bits) {
    case 2: return tie_scratch_words<2>(n);
    case 4: return tie_scratch_words<4>(n);
    default: return tie_scratch_words<8>(n);
    }
}
u32 cls_smem_bytes(int c)
{
    const u32 per = 2u * cls_units(c) * 4u;
    if (c == CLS_W2S || c == CLS_W2M || c == CLS_W2L || c == CLS_W2X) return (u32)sizeof(W2Const) + per * (kCls[c].threads / 32u);
    return kCls[c].cta ? per : per * (kCls[c].threads / 32u);
}

// One set of tie-path scratch buffers: kernels of one in-flight batch use one set.
struct ExecScratch {
    u32 *tie[CLS_COUNT] = {};
    u64 *seg = nullptr;                 // k_canon_seg: per-warp partial XXH3 sums
    u32 *huge_x = nullptr, *huge_tie = nullptr;     // CLS_HUGE: strands staged in global memory + tie scratch, grown on demand
    u64 huge_x_words = 0, huge_tie_words = 0;
    // the per-class launches that follow the lane kernel are independent of each other (own lists, own scratch): they are
    // forked onto side streams and joined back, so that the small retry / tail launches overlap instead of queueing.  One set
    // per in-flight batch (slot 0, slot 1, the device-resident API), so batches never queue behind each other's forks.
    cudaStream_t side_stream[CLS_COUNT] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[CLS_COUNT] = {};
};

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t inserted = nullptr;     // recorded after this slot's table insert
    u8 *d_raw = nullptr; u64 *d_off = nullptr; u64 *d_p2 = nullptr; u8 *d_norm = nullptr; u8 *d_p4 = nullptr;
    u32 *d_len = nullptr; u8 *d_lane = nullptr; u8 *d_out = nullptr; u32 *d_start = nullptr;
    u8 *d_strand = nullptr; u64 *d_hash = nullptr; u64 *d_first = nullptr; u64 *d_slotof = nullptr;
    u32 *d_lists = nullptr; u32 *d_counts = nullptr;
    u64 *d_dense = nullptr; u64 *d_laneoff = nullptr;   // CK_F_PACKED_IN: the host packer's dense 2-bit layout, byte-lane offsets
    u32 *h_counts = nullptr;            // pinned
    ExecScratch scr;
    bool busy = false, uniq = false, mono = false;   // mono: ck_mono_submit's batch (ck_mono_wait collects it)
    bool text = false;                  // ck_fasta_submit's batch (ck_fasta_wait collects it)
    u32 cmd = 0;                        // its CK_CMD_*
    // text batches, allocated by the first ck_fasta_submit on the slot: the text, the framed output, the record starts,
    // head / seq ranges (2 per record), 64-bit lengths (seq, then framed), framed offsets, tile counts / offsets, the longest seq
    u8 *d_text = nullptr, *d_frame = nullptr;
    u64 *d_rstart = nullptr, *d_head = nullptr, *d_seq = nullptr, *d_len64 = nullptr, *d_fofs = nullptr, *d_meta = nullptr;
    u32 *d_tiles = nullptr;
    u32 dbl = 1;                        // packed2 layout of the batch in flight
    u64 longest = 0;                    // longest raw record of the batch in flight
    u32 *sel = nullptr; u64 *coff = nullptr;    // CK_F_SURVIVORS: survivor indices / compact offsets of the batch in flight
    u32 n = 0, flags = 0; u64 total = 0;
    u64 rec_mark = 0;                   // uniq batch in flight: ck_ctx::submitted_rec once it was counted (0: not counted)
    bool defl = false;                  // ck_deflate_submit's call (ck_deflate_wait collects it)
    // ck_deflate_*: own stream and buffers, allocated by the slot's first deflate call and grown to the largest since
    struct Deflate {
        cudaStream_t stream = nullptr;
        u64 cap = 0;                    // input bytes the buffers hold
        u8 *buf = nullptr;              // dict || input
        u32 *kA = nullptr, *kB = nullptr, *vA = nullptr, *vB = nullptr;   // sort buffers; then match table / tokens
        u32 *prev8 = nullptr, *prev4 = nullptr;
        u32 *seg = nullptr;             // per segment: freq, table, header, meta, CRC, token count, offset
        u32 *out = nullptr, *result = nullptr;
        u32 *h_result = nullptr;        // pinned
        void *tmp = nullptr; size_t tmp_bytes = 0;
        u64 n = 0;
    } z;
    bool bz = false;                    // ck_bzip2_submit's call (ck_bzip2_wait collects it)
    // ck_bzip2_*: own stream and buffers, allocated by the slot's first bzip2 call and grown to the largest since
    struct Bzip2 {
        cudaStream_t stream = nullptr;
        cudaEvent_t ev[6] = {};         // stage boundaries of the last call
        u64 cap = 0, rcap = 0;          // raw input bytes / RLE1 bytes the buffers hold
        u8 *in = nullptr, *rle = nullptr, *bid = nullptr, *flag = nullptr;
        u32 *rank = nullptr, *sa = nullptr, *pos = nullptr, *pos2 = nullptr, *valA = nullptr, *valB = nullptr;
        u32 *hp = nullptr, *hs = nullptr;
        u64 *keyA = nullptr, *keyB = nullptr;
        u8 *small = nullptr;            // blocks, meta, freq, selectors, codes, headers, heap scratch
        u32 *out = nullptr, *result = nullptr;
        u32 *h_host = nullptr;          // pinned: [0..3] Bzip2Meta, [4..7] result, [8] selected count
        void *tmp = nullptr; size_t tmp_bytes = 0;
        u64 n = 0;
        u32 nblk = 0, consumed = 0, rounds = 0, bits_in = 0, nbits_in = 0, crc_in = 0;
    } bz2;
};

// Multi-GPU uniq through the C ABI: this rank's exchange block (exported by CUDA IPC) and every peer's, mapped here.
struct PeerGroup {
    u32 world = 1, rank = 0, cap = 0;     // cap = pairs a (sender, owner) region can hold = the largest batch
    u8 *block = nullptr; u64 block_bytes = 0, recv_bytes = 0, ret_bytes = 0;
    void *mapped[32] = {};                // mapped[r] = rank r's block in this process (mapped[rank] == block)
    bool exported = false, attached = false;
    u64 epoch[4] = {};                    // launches so far per barrier id (2 * slot + phase)
    u32 *pos[2] = {}; u32 *cursors[2] = {}; u64 *slot_of[2] = {};   // per exchange slot
    u64 *recv(u32 r, u32 slot) const { return reinterpret_cast<u64 *>((u8 *)mapped[r] + CK_PEER_HEADER_BYTES + (u64)slot * recv_bytes); }
    u64 *ret(u32 r, u32 slot) const { return reinterpret_cast<u64 *>((u8 *)mapped[r] + CK_PEER_HEADER_BYTES + 2 * recv_bytes + (u64)slot * ret_bytes); }
    u64 *counts(u32 r, u32 slot) const { return reinterpret_cast<u64 *>(mapped[r]) + CK_PEER_FLAG_WORDS + 32u * slot; }
};

}  // namespace

struct ck_ctx {
    int device = 0;
    int num_sms = 148;
    ck_config cfg{};
    std::string err;
    Slot slot[2];
    ExecScratch dev_scr;                // device-resident API (one stream at a time)
    cudaEvent_t last_insert = nullptr;  // insert event of the most recently submitted uniq batch
    bool have_last_insert = false;
    TableSlot *table = nullptr; u64 table_slots = 0; u64 *side = nullptr; u32 *d_overflow = nullptr;
    u64 *d_keys = nullptr;              // keys in `table` (k_table_insert counts its claims); 8 bytes after d_overflow, so one
                                        // 16-byte copy brings both back to h_counts[16] / h_counts[18..19]
    // ck_uniq_grow: grow_max = most keys the table may grow to hold (0: fixed size).  table_reserve bounds the keys in the table
    // from above by known_keys (the device's count as collected with the batch that ended at known_rec uniq records) plus the
    // uniq records submitted since (submitted_rec counts them all).
    u64 grow_max = 0, grows = 0;
    u64 known_keys = 0, known_rec = 0, submitted_rec = 0;
    PeerGroup peer;                    // world > 1 after ck_peer_attach: uniq runs the hash-range exchange
    // library drop-ins (ck_lmsr_index / ck_lmsr / ck_canonicalize): persistent staging + stream, one call at a time per
    // context (any number of host threads may call; lib/src/canonicalize.rs:54 is called from T worker threads)
    std::mutex lib_mu;
    cudaStream_t lib_stream = nullptr;
    u8 *lib_h = nullptr, *lib_d = nullptr; size_t lib_h_bytes = 0, lib_d_bytes = 0;
    ExecScratch lib_scr;
    u64 launches = 0;
    bool attrs_set = false;
    u32 s3_debug = 0;                   // CK_S3_DEBUG: bits 8.. switch the lane kernel's L2 prefetches off (traffic experiments)
    bool l4_kernel = true;              // CK_L4_KERNEL=0: {-ACGNT} records go to the generic 4-bit kernels only (A/B runs)
    bool seg_kernel = true;             // CK_SEG_KERNEL=0: long 2-bit records go to the CTA kernels only (A/B runs)
    int lane_kernel = 3;                // 2: ck_stream2.cuh (CK_LANE_KERNEL=2), else ck_stream3.cuh
    // optional per-class kernel timing (bench.py's roofline): event pairs around each class launch
    bool timing = false;
    std::vector<cudaEvent_t> ev_pairs[CLS_COUNT + 7];     // [CLS_COUNT] = lane kernel, table insert, table first, segment kernel, 4-bit lane kernel, k_pack4, k_prepare + k_extend_packed2 (device-resident entry)
};

namespace {

int fail(ck_ctx *ctx, int code, const char *what, cudaError_t e = cudaSuccess)
{
    std::string m = what;
    if (e != cudaSuccess) { m += ": "; m += cudaGetErrorString(e); }
    if (ctx) ctx->err = m; else g_init_error = m;
    return code;
}
#define CK_CUDA(ctx, call)                                                     \
    do {                                                                       \
        cudaError_t e__ = (call);                                              \
        if (e__ != cudaSuccess) return fail((ctx), CK_ERR_CUDA, #call, e__);   \
    } while (0)

void fill_tables(Tables &t, u8 secret[200])
{
    // needletail 0.5.1 normalize(_, false)
    for (int c = 0; c < 256; c++) t.norm[c] = 'N';
    for (const char *p = "ACGTN-"; *p; p++) t.norm[(u8)*p] = (u8)*p;
    t.norm['a'] = 'A'; t.norm['c'] = 'C'; t.norm['g'] = 'G';
    t.norm['t'] = 'T'; t.norm['u'] = 'T'; t.norm['U'] = 'T';
    t.norm['.'] = '-'; t.norm['~'] = '-';
    t.norm[' '] = 0; t.norm['\t'] = 0; t.norm['\r'] = 0; t.norm['\n'] = 0;
    // bio 1.3.1 complement
    for (int c = 0; c < 256; c++) t.comp[c] = (u8)c;
    const char *a = "AGCTYRWSKMDVHBN", *b = "TCGARYWSMKHBDVN";
    for (int i = 0; a[i]; i++) { t.comp[(u8)a[i]] = (u8)b[i]; t.comp[(u8)a[i] + 32] = (u8)(b[i] + 32); }
    // 16-symbol ordered alphabet of the 4-bit lane (closed under complement)
    const char *alpha = "-ABCDGHKMNRSTVWY";
    for (int c = 0; c < 256; c++) t.code4[c] = 0xff;
    for (int i = 0; i < 16; i++) { t.sym4[i] = (u8)alpha[i]; t.code4[(u8)alpha[i]] = (u8)i; }
    for (int i = 0; i < 16; i++) t.comp4[i] = t.code4[t.comp[t.sym4[i]]];
    static const u8 sec[192] = {
        0xb8, 0xfe, 0x6c, 0x39, 0x23, 0xa4, 0x4b, 0xbe, 0x7c, 0x01, 0x81, 0x2c, 0xf7, 0x21, 0xad, 0x1c,
        0xde, 0xd4, 0x6d, 0xe9, 0x83, 0x90, 0x97, 0xdb, 0x72, 0x40, 0xa4, 0xa4, 0xb7, 0xb3, 0x67, 0x1f,
        0xcb, 0x79, 0xe6, 0x4e, 0xcc, 0xc0, 0xe5, 0x78, 0x82, 0x5a, 0xd0, 0x7d, 0xcc, 0xff, 0x72, 0x21,
        0xb8, 0x08, 0x46, 0x74, 0xf7, 0x43, 0x24, 0x8e, 0xe0, 0x35, 0x90, 0xe6, 0x81, 0x3a, 0x26, 0x4c,
        0x3c, 0x28, 0x52, 0xbb, 0x91, 0xc3, 0x00, 0xcb, 0x88, 0xd0, 0x65, 0x8b, 0x1b, 0x53, 0x2e, 0xa3,
        0x71, 0x64, 0x48, 0x97, 0xa2, 0x0d, 0xf9, 0x4e, 0x38, 0x19, 0xef, 0x46, 0xa9, 0xde, 0xac, 0xd8,
        0xa8, 0xfa, 0x76, 0x3f, 0xe3, 0x9c, 0x34, 0x3f, 0xf9, 0xdc, 0xbb, 0xc7, 0xc7, 0x0b, 0x4f, 0x1d,
        0x8a, 0x51, 0xe0, 0x4b, 0xcd, 0xb4, 0x59, 0x31, 0xc8, 0x9f, 0x7e, 0xc9, 0xd9, 0x78, 0x73, 0x64,
        0xea, 0xc5, 0xac, 0x83, 0x34, 0xd3, 0xeb, 0xc3, 0xc5, 0x81, 0xa0, 0xff, 0xfa, 0x13, 0x63, 0xeb,
        0x17, 0x0d, 0xdd, 0x51, 0xb7, 0xf0, 0xda, 0x49, 0xd3, 0x16, 0x55, 0x26, 0x29, 0xd4, 0x68, 0x9e,
        0x2b, 0x16, 0xbe, 0x58, 0x7d, 0x47, 0xa1, 0xfc, 0x8f, 0xf8, 0xb8, 0xd1, 0x7a, 0xd0, 0x31, 0xce,
        0x45, 0xcb, 0x3a, 0x8f, 0x95, 0x16, 0x04, 0x28, 0xaf, 0xd7, 0xfb, 0xca, 0xbb, 0x4b, 0x40, 0x7e,
    };
    memset(secret, 0, 200);
    memcpy(secret, sec, 192);
}

int alloc_scratch(ck_ctx *ctx, ExecScratch &s)
{
    CK_CUDA(ctx, cudaEventCreateWithFlags(&s.ev_fork, cudaEventDisableTiming));
    for (int c = 0; c < CLS_COUNT; c++) {
        CK_CUDA(ctx, cudaStreamCreateWithFlags(&s.side_stream[c], cudaStreamNonBlocking));
        CK_CUDA(ctx, cudaEventCreateWithFlags(&s.ev_join[c], cudaEventDisableTiming));
    }
    CK_CUDA(ctx, cudaMalloc(&s.seg, (size_t)2 * ctx->num_sms * CK_SEG_WARPS * CK_SEG_SCRATCH_U64 * 8));
    for (int c = 0; c < CLS_COUNT; c++) {
        if (kCls[c].bits == 0) continue;
        const u64 groups = (u64)kCls[c].ctas_per_sm * ctx->num_sms * (kCls[c].cta ? 1u : kCls[c].threads / 32u);
        CK_CUDA(ctx, cudaMalloc(&s.tie[c], groups * cls_tie_words(c) * 4));
    }
    return CK_OK;
}
void free_scratch(ExecScratch &s)
{
    for (int c = 0; c < CLS_COUNT; c++) {
        if (s.tie[c]) cudaFree(s.tie[c]);
        if (s.side_stream[c]) cudaStreamDestroy(s.side_stream[c]);
        if (s.ev_join[c]) cudaEventDestroy(s.ev_join[c]);
        s.tie[c] = nullptr; s.side_stream[c] = nullptr; s.ev_join[c] = nullptr;
    }
    if (s.ev_fork) cudaEventDestroy(s.ev_fork);
    if (s.seg) cudaFree(s.seg);
    if (s.huge_x) cudaFree(s.huge_x);
    if (s.huge_tie) cudaFree(s.huge_tie);
    s.huge_x = s.huge_tie = nullptr; s.huge_x_words = s.huge_tie_words = 0;
    s.ev_fork = nullptr; s.seg = nullptr;
}

template <typename K> int set_smem(ck_ctx *ctx, K kernel, u32 bytes)
{
    if (bytes > 48 * 1024) CK_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return CK_OK;
}
// lane-per-record streaming kernel, variant v (CK_W2_* bits): ck_stream3.cuh, or its predecessor ck_stream2.cuh when
// the environment says CK_LANE_KERNEL=2 (A/B runs)
void s2_launch(ck_ctx *ctx, cudaStream_t st, const CanonArgs &a, int v)
{
    if (ctx->lane_kernel != 2 && a.p2_dbl) {
        const u32 g3 = 2u * (u32)ctx->num_sms, th3 = 32u * CK_S3_WARPS, sm3 = CK_S3_WARPS * CK_S3_WARP_BYTES;
#define CK_S3(V) k_canon_s3<V><<<g3, th3, sm3, st>>>(a)
        switch (v) {
        case 0: CK_S3(0); break; case 1: CK_S3(1); break; case 2: CK_S3(2); break; case 3: CK_S3(3); break;
        case 4: CK_S3(4); break; case 5: CK_S3(5); break; case 6: CK_S3(6); break; default: CK_S3(7);
        }
#undef CK_S3
        return;
    }
    const u32 g = 2u * (u32)ctx->num_sms, th = 32u * CK_S2_WARPS, sm = CK_S2_WARPS * CK_S2_WARP_BYTES;
#define CK_S2(V) k_canon_s2<V><<<g, th, sm, st>>>(a)
    switch (v) {
    case 0: CK_S2(0); break; case 1: CK_S2(1); break; case 2: CK_S2(2); break; case 3: CK_S2(3); break;
    case 4: CK_S2(4); break; case 5: CK_S2(5); break; case 6: CK_S2(6); break; default: CK_S2(7);
    }
#undef CK_S2
}

int set_attrs(ck_ctx *ctx)
{
    if (ctx->attrs_set) return CK_OK;
    int rc;
    if ((rc = set_smem(ctx, k_canon_cta<2, false>, cls_smem_bytes(CLS_C2B)))) return rc;
    if ((rc = set_smem(ctx, k_canon_cta<4, false>, cls_smem_bytes(CLS_C4)))) return rc;
    if ((rc = set_smem(ctx, k_canon_cta<8, false>, cls_smem_bytes(CLS_C8)))) return rc;
    const u32 s2 = CK_S2_WARPS * CK_S2_WARP_BYTES;
    if ((rc = set_smem(ctx, k_canon_s2<0>, s2)) || (rc = set_smem(ctx, k_canon_s2<1>, s2)) || (rc = set_smem(ctx, k_canon_s2<2>, s2)) ||
        (rc = set_smem(ctx, k_canon_s2<3>, s2)) || (rc = set_smem(ctx, k_canon_s2<4>, s2)) || (rc = set_smem(ctx, k_canon_s2<5>, s2)) ||
        (rc = set_smem(ctx, k_canon_s2<6>, s2)) || (rc = set_smem(ctx, k_canon_s2<7>, s2))) return rc;
    const u32 s3 = CK_S3_WARPS * CK_S3_WARP_BYTES;
    if ((rc = set_smem(ctx, k_canon_s3<0>, s3)) || (rc = set_smem(ctx, k_canon_s3<1>, s3)) || (rc = set_smem(ctx, k_canon_s3<2>, s3)) ||
        (rc = set_smem(ctx, k_canon_s3<3>, s3)) || (rc = set_smem(ctx, k_canon_s3<4>, s3)) || (rc = set_smem(ctx, k_canon_s3<5>, s3)) ||
        (rc = set_smem(ctx, k_canon_s3<6>, s3)) || (rc = set_smem(ctx, k_canon_s3<7>, s3))) return rc;
    const u32 l4 = CK_L4_WARPS * CK_L4_WARP_BYTES;
    if ((rc = set_smem(ctx, k_canon_l4<0>, l4)) || (rc = set_smem(ctx, k_canon_l4<1>, l4)) || (rc = set_smem(ctx, k_canon_l4<2>, l4)) ||
        (rc = set_smem(ctx, k_canon_l4<3>, l4))) return rc;
    ctx->attrs_set = true;
    return CK_OK;
}

struct CanonIO {
    const u64 *packed2; const u8 *bytes; const u64 *offsets; const u32 *lens; const u8 *lane;
    u32 n; u32 mode;
    u32 dbl = 1;                      // packed2 layout of the batch: 1 doubled (ck_stream3 / ck_seg2), 0 single copy (ck_stream2)
    u64 longest = 0;                  // longest raw record of the batch when the host knows it (host-buffer entries): records beyond
                                      // the staged-length classes are then processed from global memory instead of being reported
    u8 *p4 = nullptr;                 // optional packed4 arena (ck_lane4.cuh), p4_bytes_total(total, n) bytes: enables k_canon_l4
    u8 *out; u32 *out_start; u8 *out_strand; u64 *out_hash;
    u32 *lists; u64 lists_bytes;      // sort workspace: >= ck_lists_bytes(n)
    u32 *counts;                      // 32 u32: class counts, run starts
};

// sort workspace of a batch of n records: two (key, index) buffer pairs + radix-sort temporaries
u64 lists_bytes_for(u64 n) { return ((16 * (n + 4) + 24 * (n + 4) + 255) & ~255ull) + (1ull << 20); }   // keeps what follows 256-byte aligned

// classify + one launch per class.  counts[CLS_HUGE] > 0 afterwards means unprocessed records.
int run_canon(ck_ctx *ctx, cudaStream_t st, ExecScratch &scr, const CanonIO &io, u32 class_mask)
{
    if (io.n == 0) return CK_OK;
    int rc = set_attrs(ctx);
    if (rc) return rc;
    CK_CUDA(ctx, cudaMemsetAsync(io.counts, 0, 64 * sizeof(u32), st));
    // a promise of exactly one class lets that class index the records directly (no work lists)
    int only = -1;
    if (class_mask && (class_mask & (class_mask - 1)) == 0)
        for (int c = 0; c < CLS_COUNT; c++) if (class_mask == (1u << c)) only = c;
    const u64 stride = ((u64)io.n + 4) & ~3ull;                // u32 elements per sort buffer
    u32 *k0 = io.lists, *k1 = k0 + stride, *v0 = k1 + stride, *v1 = v0 + stride;
    if (io.lists_bytes < 16 * stride) return fail(ctx, CK_ERR_ARG, "sort workspace too small");
    // both strands, aligned bytes or none: the lane-per-record streaming kernel; everything else (forward-only library
    // calls, output at the input's offsets): the run-time-option warp-per-record kernel
    const bool fastv = io.packed2 && !(io.mode & 1u) && (!io.out || (io.mode & 2u)) && io.out_start && io.out_strand;
    u32 window_shift = 32, top_bit = 13;
    if (fastv && only < 0) {
        // windows of 64 K records (config 2, lane kernel: none 6.30 ms, 1 K 5.97, 4 K 5.89, 16 K 5.88, 64 K 5.86, 256 K 5.96; 1/8-octave bins inside the windows 5.89;
        // DRAM reads of the launch 13.1 -> 11.0 GB, of its scan pass alone 7.4 -> 5.1 GB: profiles/r01_j_traffic.txt)
        window_shift = 16;
        u32 wbits = 0;
        while ((((u64)io.n - 1) >> window_shift) >> wbits) wbits++;
        top_bit = std::max(14u, 5u + wbits);
    }
    // records over {-, A, C, G, N, T} (what needletail's normalisation leaves of IUPAC input): both strands packed at 4 bits
    // for the lane-per-record kernel of ck_lane4.cuh; their lane tag becomes 3
    const bool l4_run = fastv && only < 0 && ctx->l4_kernel && io.p4 && io.lane && io.bytes && (!class_mask || (class_mask & (1u << CLS_W4)));
    if (l4_run) {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (ctx->timing) { CK_CUDA(ctx, cudaEventCreate(&e0)); CK_CUDA(ctx, cudaEventCreate(&e1)); CK_CUDA(ctx, cudaEventRecord(e0, st)); }
        k_pack4<<<std::min<u32>((io.n + 15) / 16, 16u * (u32)ctx->num_sms), 256, 0, st>>>(io.bytes, io.offsets, io.lens, const_cast<u8 *>(io.lane), io.n, io.p4);
        if (ctx->timing) { CK_CUDA(ctx, cudaEventRecord(e1, st)); ctx->ev_pairs[CLS_COUNT + 5].push_back(e0); ctx->ev_pairs[CLS_COUNT + 5].push_back(e1); }
        ctx->launches++;
    }
    const int sort_bits = (int)top_bit + 1;
    // a promise of one of the lane classes over a pure 2-bit batch: the lane kernel walks every record anyway and reports the
    // ones outside the promise itself (configs 1 and 5: one launch less per batch, 0.1 ms of a 2.8 ms step)
    const bool lane_checks = fastv && only >= 0 && io.lane == nullptr &&
                             (only == CLS_W2S || only == CLS_W2M || only == CLS_W2L || only == CLS_W2X);
    if (!lane_checks) {
        ClassifyArgs ca{io.offsets, io.lens, io.lane, io.n, k0, v0, io.counts, only >= 0 ? (1u << only) : 0u, window_shift, top_bit};
        k_classify<<<std::min<u32>((io.n + 255) / 256, 16u * (u32)ctx->num_sms), 256, 0, st>>>(ca);
        ctx->launches++;
    }
    const u32 *sorted = nullptr;
    u32 *retry = v0;                                           // direct mode: the sort buffers are free
    if (only < 0) {
        // one index list for the whole batch: classes are contiguous runs, each ordered by length
        cub::DoubleBuffer<u32> keys(k0, k1), vals(v0, v1);
        void *tmp = v1 + stride;
        size_t tmp_bytes = (size_t)(io.lists_bytes - 16 * stride), need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, keys, vals, (int)io.n, 0, sort_bits, st);
        if (need > tmp_bytes) return fail(ctx, CK_ERR_ARG, "sort workspace too small");
        CK_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, need, keys, vals, (int)io.n, 0, sort_bits, st));
        sorted = vals.Current();
        retry = vals.Alternate();
        k_list_starts<<<1, 32, 0, st>>>(io.counts);
        ctx->launches += 2;
    }
    const u32 lane_classes = (1u << CLS_W2S) | (1u << CLS_W2M) | (1u << CLS_W2L) | (1u << CLS_W2X);
    auto timed = [&](int slot, cudaEvent_t &e0, cudaEvent_t &e1, bool begin, cudaStream_t on) -> cudaError_t {
        if (!ctx->timing) return cudaSuccess;
        if (begin) {
            cudaError_t e = cudaEventCreate(&e0); if (e != cudaSuccess) return e;
            e = cudaEventCreate(&e1); if (e != cudaSuccess) return e;
            return cudaEventRecord(e0, on);
        }
        ctx->ev_pairs[slot].push_back(e0); ctx->ev_pairs[slot].push_back(e1);
        return cudaEventRecord(e1, on);
    };
    auto base_args = [&](int c) {
        CanonArgs a{};
        a.packed2 = io.packed2; a.p2_dbl = io.dbl; a.bytes = io.bytes; a.offsets = io.offsets; a.lens = io.lens;
        a.max_n = cls_max_n(c); a.min_n = cls_min_n(c);
        a.out = io.out; a.out_start = io.out_start; a.out_strand = io.out_strand; a.out_hash = io.out_hash;
        a.scratch = scr.tie[c]; a.scratch_stride = kCls[c].bits ? cls_tie_words(c) : 0;
        a.smem_units = kCls[c].bits ? cls_units(c) : 0; a.xglobal = nullptr; a.mode = io.mode;
        a.retry = retry; a.retry_counts = io.counts + 32;
        return a;
    };
    const bool lane_run = fastv && (only >= 0 ? ((lane_classes >> only) & 1u) != 0 : (!class_mask || (class_mask & lane_classes)));
    if (lane_run) {
        CanonArgs a = base_args(only >= 0 ? only : CLS_W2S);
        if (only >= 0) { a.list = nullptr; a.count = nullptr; a.n_direct = io.n; }
        else { a.list = sorted; a.count = io.counts + 12; a.n_direct = 0; a.min_n = 1; a.max_n = cls_max_n(CLS_W2X); }
        const int v = (a.out_hash ? CK_W2_HASH : 0) | (a.out ? CK_W2_OUT : 0) | (a.list ? CK_W2_LIST : 0);
        a.mode |= ctx->s3_debug;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        CK_CUDA(ctx, timed(CLS_COUNT, e0, e1, true, st));
        s2_launch(ctx, st, a, v);
        CK_CUDA(ctx, timed(CLS_COUNT, e0, e1, false, st));
        ctx->launches++;
    }
    // long 2-bit records (8 k .. 426 k bases): one warp per record, a lane per segment (ck_seg2.cuh); what ties goes to the
    // CTA kernels' duel path through the retry lists
    const u32 seg_classes = (1u << CLS_C2A) | (1u << CLS_C2B);
    const bool seg_run = fastv && only < 0 && ctx->seg_kernel && io.dbl && (!class_mask || (class_mask & seg_classes));
    if (seg_run) {
        CanonArgs a = base_args(CLS_C2A);
        a.list = sorted; a.count = io.counts + 13; a.n_direct = 0;
        const u32 g = 2u * (u32)ctx->num_sms, th = 32u * CK_SEG_WARPS, sm = CK_SEG_WARPS * CK_SEG_WARP_BYTES;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        CK_CUDA(ctx, timed(CLS_COUNT + 3, e0, e1, true, st));
        switch ((a.out_hash ? CK_W2_HASH : 0) | (a.out ? CK_W2_OUT : 0)) {
        case 0: k_canon_seg<0><<<g, th, sm, st>>>(a, scr.seg); break;
        case 1: k_canon_seg<1><<<g, th, sm, st>>>(a, scr.seg); break;
        case 2: k_canon_seg<2><<<g, th, sm, st>>>(a, scr.seg); break;
        default: k_canon_seg<3><<<g, th, sm, st>>>(a, scr.seg); break;
        }
        CK_CUDA(ctx, timed(CLS_COUNT + 3, e0, e1, false, st));
        ctx->launches++;
    }
    if (l4_run) {
        CanonArgs a = base_args(CLS_W4);
        a.list = sorted; a.count = io.counts + CLS_W4; a.n_direct = 0;
        const u32 g = 2u * (u32)ctx->num_sms, th = 32u * CK_L4_WARPS, sm = CK_L4_WARPS * CK_L4_WARP_BYTES;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        CK_CUDA(ctx, timed(CLS_COUNT + 4, e0, e1, true, st));
        switch ((a.out_hash ? CK_W2_HASH : 0) | (a.out ? CK_W2_OUT : 0)) {
        case 0: k_canon_l4<0><<<g, th, sm, st>>>(a, io.p4, io.lane); break;
        case 1: k_canon_l4<1><<<g, th, sm, st>>>(a, io.p4, io.lane); break;
        case 2: k_canon_l4<2><<<g, th, sm, st>>>(a, io.p4, io.lane); break;
        default: k_canon_l4<3><<<g, th, sm, st>>>(a, io.p4, io.lane); break;
        }
        CK_CUDA(ctx, timed(CLS_COUNT + 4, e0, e1, false, st));
        ctx->launches++;
    }
    u32 to_launch = 0;
    for (int c = 0; c < CLS_COUNT; c++)
        if (c != CLS_HUGE && !(class_mask && !(class_mask & (1u << c)))) to_launch++;
    const bool fork = scr.ev_fork != nullptr && to_launch >= 2;
    if (fork) CK_CUDA(ctx, cudaEventRecord(scr.ev_fork, st));
    u32 joined = 0;
    for (int c = 0; c < CLS_COUNT; c++) {
        if (c == CLS_HUGE) continue;
        if (class_mask && !(class_mask & (1u << c))) continue;
        CanonArgs a = base_args(c);
        const bool is_lane_cls = ((lane_classes >> c) & 1u) != 0;
        if ((lane_run && is_lane_cls) || (seg_run && ((seg_classes >> c) & 1u)) || (l4_run && c == CLS_W4)) { a.list = retry; a.count = io.counts + 32 + c; a.n_direct = 0; }   // what the lane / segment kernel left over
        else if (only >= 0) { a.list = nullptr; a.count = nullptr; a.n_direct = io.n; }
        else { a.list = sorted; a.count = io.counts + c; a.n_direct = 0; }
        const u32 grid = kCls[c].ctas_per_sm * (u32)ctx->num_sms, thr = kCls[c].threads;
        const u32 smem = kCls[c].bits ? cls_smem_bytes(c) : 0;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        // CTA-per-record kernels fill the GPU by themselves and keep their place on the caller's stream; the warp-per-record
        // launches (retry lists, byte lanes, empty records) are the small ones that gain from running side by side
        // (behind the segment kernel the CTA kernels of the long 2-bit classes only see its retry list -- the adversarial
        // repeats -- and no longer fill the GPU: they fork too)
        const bool side = fork && (!kCls[c].cta || (seg_run && ((seg_classes >> c) & 1u)));
        cudaStream_t sc = side ? scr.side_stream[c] : st;
        if (side) CK_CUDA(ctx, cudaStreamWaitEvent(sc, scr.ev_fork, 0));
        CK_CUDA(ctx, timed(c, e0, e1, true, sc));
        switch (c) {
        case CLS_W2S: k_canon_w2<true, -1><<<grid, thr, smem, sc>>>(a); break;
        case CLS_W2M: case CLS_W2L: case CLS_W2X: k_canon_w2<false, -1><<<grid, thr, smem, sc>>>(a); break;
        case CLS_C2A: case CLS_C2B: k_canon_cta<2, false><<<grid, thr, smem, sc>>>(a); break;
        case CLS_W4: k_canon_warp<4><<<grid, thr, smem, sc>>>(a); break;
        case CLS_C4: k_canon_cta<4, false><<<grid, thr, smem, sc>>>(a); break;
        case CLS_W8: k_canon_warp<8><<<grid, thr, smem, sc>>>(a); break;
        case CLS_C8: k_canon_cta<8, false><<<grid, thr, smem, sc>>>(a); break;
        case CLS_EMPTY: k_canon_empty<<<(u32)ctx->num_sms, 256, 0, sc>>>(a); break;
        }
        CK_CUDA(ctx, timed(c, e0, e1, false, sc));
        if (side) { CK_CUDA(ctx, cudaEventRecord(scr.ev_join[c], sc)); joined |= 1u << c; }
        ctx->launches++;
    }
    for (int c = 0; c < CLS_COUNT; c++)
        if ((joined >> c) & 1u) CK_CUDA(ctx, cudaStreamWaitEvent(st, scr.ev_join[c], 0));
    // records beyond the staged-length classes (2-bit > 425 984, 4-bit > 212 992, bytes > 106 496 symbols): the CTA kernel with
    // both strands staged in global memory, a few CTAs, one launch per symbol lane over the CLS_HUGE run of the list
    if (only < 0 && io.longest > cls_max_n(CLS_C8) && (!class_mask || (class_mask & (1u << CLS_HUGE)))) {
        const u64 nl = io.longest;
        const u32 G = (u32)std::max<u64>(1, std::min<u64>(32, (1ull << 30) / (2 * nl + 64)));
        const u64 xw = (u64)G * 2 * strand_units<8>((u32)nl), tw = (u64)G * tie_scratch_words<8>(nl);
        if (xw > scr.huge_x_words) {
            if (scr.huge_x) CK_CUDA(ctx, cudaFree(scr.huge_x));
            scr.huge_x = nullptr; scr.huge_x_words = 0;
            CK_CUDA(ctx, cudaMalloc(&scr.huge_x, xw * 4));
            scr.huge_x_words = xw;
        }
        if (tw > scr.huge_tie_words) {
            if (scr.huge_tie) CK_CUDA(ctx, cudaFree(scr.huge_tie));
            scr.huge_tie = nullptr; scr.huge_tie_words = 0;
            CK_CUDA(ctx, cudaMalloc(&scr.huge_tie, tw * 4));
            scr.huge_tie_words = tw;
        }
        CanonArgs a = base_args(CLS_HUGE);
        a.list = sorted; a.count = io.counts + CLS_HUGE; a.n_direct = 0; a.min_n = 1; a.max_n = 0xffffffffu;
        a.xglobal = scr.huge_x; a.scratch = scr.huge_tie; a.lane_bits = io.lane;
        a.smem_units = strand_units<2>((u32)nl); a.scratch_stride = tie_scratch_words<2>(nl);
        if (nl > cls_max_n(CLS_C2B)) { k_canon_cta<2, true><<<G, 1024, 0, st>>>(a); ctx->launches++; }
        if (io.lane && nl > cls_max_n(CLS_C4)) {
            a.smem_units = strand_units<4>((u32)nl); a.scratch_stride = tie_scratch_words<4>(nl);
            k_canon_cta<4, true><<<G, 1024, 0, st>>>(a);
            ctx->launches++;
        }
        if (io.lane) {
            a.smem_units = strand_units<8>((u32)nl); a.scratch_stride = tie_scratch_words<8>(nl);
            k_canon_cta<8, true><<<G, 1024, 0, st>>>(a);
            ctx->launches++;
        }
        CK_CUDA(ctx, cudaMemsetAsync(io.counts + CLS_HUGE, 0, 4, st));      // processed: nothing to report
    }
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}

// k_extend_packed2 runs one warp per record (8 per CTA)
u32 extend_grid(const ck_ctx *ctx, u32 n_records) { return std::max(1u, std::min<u32>((n_records + 7) / 8, 32u * (u32)ctx->num_sms)); }

// slots of a first-occurrence table that is to hold `keys` keys: 1.5 per key (load <= 0.67, linear probing), any number
u64 table_slots_for(u64 keys) { return std::max<u64>(1024, keys + keys / 2 + 16); }

int table_insert(ck_ctx *ctx, cudaStream_t st, TableSlot *slots, u64 nslots, u64 *side, u32 *overflow,
                 const u64 *hash, const u64 *index, u64 base, u32 n, u64 *slot_of, u32 stride = 1, u64 *keys = nullptr)
{
    if (!n) return CK_OK;
    TableArgs t{slots, nslots, side, hash, index, stride, base, n, slot_of, nullptr, overflow, keys};
    k_table_insert<<<(n + 255) / 256, 256, 0, st>>>(t);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int table_first(ck_ctx *ctx, cudaStream_t st, TableSlot *slots, u64 nslots, u64 *side, const u64 *slot_of, u32 n, u64 *first)
{
    if (!n) return CK_OK;
    TableArgs t{slots, nslots, side, nullptr, nullptr, 1, 0, n, const_cast<u64 *>(slot_of), first, nullptr};
    k_table_first<<<(n + 255) / 256, 256, 0, st>>>(t);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}

// keys a table of `slots` slots holds at load <= 2/3
u64 table_capacity_keys(u64 slots) { return slots * 2 / 3; }

// Growth (ck_uniq_grow): a table of `slots` slots, the context's keys rehashed into it on `st`, the old table freed.  The
// caller has synchronised both slot streams: no insert or k_table_first of an earlier batch still refers to the old table.
int table_grow(ck_ctx *ctx, cudaStream_t st, u64 slots)
{
    TableSlot *t = nullptr;
    cudaError_t e = cudaMalloc(&t, slots * sizeof(TableSlot));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, CK_ERR_TABLE_FULL, "uniq table cannot grow: its new size cannot be allocated", e);
    }
    e = cudaMemsetAsync(t, 0xff, slots * sizeof(TableSlot), st);   // empty key and empty first are both all ones
    if (e == cudaSuccess) {
        const u64 grid = std::min<u64>((ctx->table_slots + 255) / 256, 32ull * (u64)ctx->num_sms);
        k_table_rehash<<<(u32)grid, 256, 0, st>>>(ctx->table, ctx->table_slots, t, slots);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cudaFree(t); return fail(ctx, CK_ERR_CUDA, "uniq table growth", e); }
    cudaFree(ctx->table);
    ctx->table = t; ctx->table_slots = slots; ctx->grows++;
    return CK_OK;
}

// Every uniq batch of n records calls this before it enqueues anything (not in a peer group).  With growth on, the table is
// grown here whenever the batch could take it past 2/3 load: the host's bound on the keys decides when to look, the device's
// exact count whether to grow.  The new size leaves room for twice the keys and two more batches of this size, so growths
// are O(log keys) and a stream of duplicates near the bound does not synchronise on every batch.  A refused batch leaves the
// table as it was.
int table_reserve(ck_ctx *ctx, Slot &s, u64 n)
{
    const u64 cap = table_capacity_keys(ctx->table_slots);
    if (ctx->grow_max && ctx->known_keys + (ctx->submitted_rec - ctx->known_rec) + n > cap) {
        // the other slot's insert and k_table_first (its slot indices point into this table) finish first
        for (Slot &o : ctx->slot) if (o.stream) CK_CUDA(ctx, cudaStreamSynchronize(o.stream));
        u64 exact = 0;
        CK_CUDA(ctx, cudaMemcpy(&exact, ctx->d_keys, 8, cudaMemcpyDeviceToHost));
        ctx->known_keys = exact; ctx->known_rec = ctx->submitted_rec;
        const u64 need = exact + n;
        if (need > cap) {
            if (need > ctx->grow_max) return fail(ctx, CK_ERR_TABLE_FULL, "uniq batch would take the table past max_keys");
            const int rc = table_grow(ctx, s.stream, table_slots_for(std::min(ctx->grow_max, 2 * need + 2 * n)));
            if (rc) return rc;
        }
    }
    ctx->submitted_rec += n;
    s.rec_mark = ctx->submitted_rec;
    return CK_OK;
}

// a collected uniq batch brings the device's key count as of its table_first back in h_counts[18..19]
void note_keys(ck_ctx *ctx, const Slot &s)
{
    if (s.rec_mark <= ctx->known_rec) return;     // an older count than the one known (or the batch was not counted)
    memcpy(&ctx->known_keys, s.h_counts + 18, 8);
    ctx->known_rec = s.rec_mark;
}

// The hash-range exchange of multi-GPU uniq, fused into the kernels around it (SURVEY 8e; replaces the single `seen` map of
// src/uniq.rs:27 across ranks).  Per batch, on every rank, in stream order:
//   k_owner_scatter_peers   (hash, index) pairs -> region `rank` of their OWNER's receive buffer, over NVLink
//   k_peer_barrier (2 slot) + how many pairs went to each owner
//   k_table_insert_regions  the owner keeps the minimum index per key
//   [insert_done, when given, is recorded here; wait_before_query, when given, is waited for here]
//   k_table_first_regions   first index per received pair -> region `rank` of the ASKING rank's return buffer
//   k_peer_barrier (2 slot + 1)
//   k_gather_first          answers back into input order
int peer_first_index(ck_ctx *ctx, cudaStream_t st, u32 slot, const u64 *hash, u32 n, u64 base_index, TableSlot *table, u64 nslots,
                     u64 *side, u32 *overflow, u64 *out_first, cudaEvent_t insert_done, cudaEvent_t wait_before_query)
{
    PeerGroup &P = ctx->peer;
    if (!P.attached) return fail(ctx, CK_ERR_STATE, "peer group not attached");
    if (n > P.cap) return fail(ctx, CK_ERR_ARG, "batch larger than the peer group's max_records");
    CK_CUDA(ctx, cudaMemsetAsync(P.cursors[slot], 0, (P.world + 1) * sizeof(u32), st));
    OwnerPeerArgs oa{};
    oa.hash = hash; oa.n = n; oa.world = P.world; oa.rank = P.rank; oa.base_index = base_index; oa.cap = P.cap;
    oa.cursors = P.cursors[slot]; oa.pos = P.pos[slot];
    PeerBlockPtrs blocks{};
    RegionArgs ra{};
    for (u32 r = 0; r < P.world; r++) {
        oa.recv.p[r] = P.recv(r, slot);
        blocks.p[r] = reinterpret_cast<u64 *>(P.mapped[r]);
        ra.ret.p[r] = P.ret(r, slot);
    }
    if (n) {
        k_owner_scatter_peers<<<std::min<u32>((n + 255) / 256, 8u * (u32)ctx->num_sms), 256, 0, st>>>(oa);
        ctx->launches++;
    }
    k_peer_barrier<<<1, 32, 0, st>>>(blocks, P.world, P.rank, 2 * slot, ++P.epoch[2 * slot], P.cursors[slot], slot);
    ra.slots = table; ra.nslots = nslots; ra.side_first = side; ra.overflow = overflow;
    ra.recv = P.recv(P.rank, slot); ra.counts = P.counts(P.rank, slot); ra.slot_of = P.slot_of[slot];
    ra.world = P.world; ra.rank = P.rank; ra.cap = P.cap;
    const u32 gx = std::max<u32>(1u, std::min<u32>((P.cap + 255) / 256, (8u * (u32)ctx->num_sms + P.world - 1) / P.world));
    k_table_insert_regions<<<dim3(gx, P.world), 256, 0, st>>>(ra);
    if (insert_done) CK_CUDA(ctx, cudaEventRecord(insert_done, st));
    if (wait_before_query) CK_CUDA(ctx, cudaStreamWaitEvent(st, wait_before_query, 0));
    k_table_first_regions<<<dim3(gx, P.world), 256, 0, st>>>(ra);
    k_peer_barrier<<<1, 32, 0, st>>>(blocks, P.world, P.rank, 2 * slot + 1, ++P.epoch[2 * slot + 1], nullptr, 0);
    if (n) k_gather_first<<<std::min<u32>((n + 255) / 256, 16u * (u32)ctx->num_sms), 256, 0, st>>>(P.ret(P.rank, slot), P.pos[slot], n, out_first);
    ctx->launches += 5;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}

// Longest record of a monomerize batch: every kernel of that path keeps lengths and in-record positions in u32 and steps
// through a record 512 bytes at a time, so positions up to length + 511 must fit.  (Canonicalize / uniq: 2^30 symbols.)
constexpr u64 kMonoMaxRecord = (1ull << 32) - 1024;

// the builder's rules (lib/src/monomerize.rs:20-40) and the known option flags
int mono_options_check(ck_ctx *ctx, const ck_mono_options *opt)
{
    if (!opt) return fail(ctx, CK_ERR_ARG, "null options");
    if (opt->seed_len < 1 || opt->seed_len > 63) return fail(ctx, CK_ERR_ARG, "Seed length must be at least 1 and at most 63");
    if (opt->overlap_min_identity >= 0.0 && opt->overlap_dist)
        return fail(ctx, CK_ERR_ARG, "Both overlap_dist and overlap_min_identity are set. They are mutually exclusive");
    if (opt->flags & ~(CK_MONO_SENSITIVE | CK_MONO_FIRST_ONLY | CK_MONO_KEEP_ALL)) return fail(ctx, CK_ERR_ARG, "unknown option flags");
    return CK_OK;
}

// shared front of every submit: slot and batch checks.  Returns CK_OK with s.busy still false; n_records == 0 is complete.
int submit_check(ck_ctx *ctx, int slot, const uint64_t *offsets, uint32_t n_records, uint32_t flags, bool uniq, bool have_bytes,
                 bool mono = false)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    Slot &s = ctx->slot[slot];
    if (s.busy) return fail(ctx, CK_ERR_STATE, "slot already holds a batch; call the matching wait first");
    if (n_records > ctx->cfg.max_batch_records) return fail(ctx, CK_ERR_ARG, "n_records exceeds max_batch_records");
    if (n_records && (!offsets || (!have_bytes && offsets[n_records] != offsets[0])))
        return fail(ctx, CK_ERR_ARG, "null batch pointers");
    if (uniq && !ctx->table) return fail(ctx, CK_ERR_STATE, "context was created with table_capacity 0");
    s.n = n_records; s.flags = flags; s.uniq = uniq; s.mono = false; s.text = false; s.defl = false; s.bz = false; s.total = 0; s.rec_mark = 0;
    if (n_records == 0) return CK_OK;
    if (offsets[0] != 0) return fail(ctx, CK_ERR_ARG, "offsets[0] must be 0");
    const u64 total = offsets[n_records];
    if (total > ctx->cfg.max_batch_bytes) return fail(ctx, CK_ERR_ARG, "batch exceeds max_batch_bytes");
    u64 longest = 0;
    for (u32 i = 0; i < n_records; i++) {
        if (offsets[i + 1] < offsets[i]) return fail(ctx, CK_ERR_ARG, "offsets must be non-decreasing");
        longest = std::max<u64>(longest, offsets[i + 1] - offsets[i]);
    }
    if (mono && longest > kMonoMaxRecord) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^32 - 1024 bytes");
    if (!mono && longest > (1ull << 30)) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^30 symbols");
    s.total = total;
    s.longest = longest;
    s.dbl = longest > 512 ? 1u : 0u;     // batches of short records: single-copy arena (ck_device.cuh)
    return CK_OK;
}

// Order-preserving compaction of the records a batch writes (uniq's survivors, monomerize's written records): a flag per
// record -> cub::DeviceSelect (their indices, increasing) -> their lengths rounded up to 16 -> exclusive scan = 16-byte-aligned
// compact offsets.  The sort workspace of the batch is free by now (stream order): indices | lengths / offsets | flags | cub
// temporaries live in it.  compaction_carve lays it out (the caller fills `flags` in stream order); compaction_select_scan
// selects and scans, copies the count to h_counts[20] and leaves s.sel / s.coff for the wait; the caller gathers the bytes.
struct Compaction {
    u32 *sel; u64 *len16; u64 *coff; u8 *flags; u32 *n_sel; void *tmp; size_t tmp_bytes;
};
int compaction_carve(ck_ctx *ctx, Slot &s, Compaction &c)
{
    const u32 n = s.n;
    u8 *w = reinterpret_cast<u8 *>(s.d_lists);
    c.sel = reinterpret_cast<u32 *>(w); w += ((size_t)n * 4 + 255) & ~(size_t)255;
    c.len16 = reinterpret_cast<u64 *>(w); w += ((size_t)(n + 1) * 8 + 255) & ~(size_t)255;
    c.coff = reinterpret_cast<u64 *>(w); w += ((size_t)(n + 1) * 8 + 255) & ~(size_t)255;
    c.flags = w; w += ((size_t)n + 255) & ~(size_t)255;
    c.n_sel = reinterpret_cast<u32 *>(w); w += 256;
    c.tmp = w;
    const size_t used = (size_t)(w - reinterpret_cast<u8 *>(s.d_lists));
    const size_t have = lists_bytes_for(ctx->cfg.max_batch_records);
    size_t need_a = 0, need_b = 0;
    cub::CountingInputIterator<u32> ids(0);
    cub::DeviceSelect::Flagged(nullptr, need_a, ids, c.flags, c.sel, c.n_sel, (int)n, s.stream);
    cub::DeviceScan::ExclusiveSum(nullptr, need_b, c.len16, c.coff, (int)n + 1, s.stream);
    if (used + std::max(need_a, need_b) > have) return fail(ctx, CK_ERR_ARG, "sort workspace too small for the compaction");
    c.tmp_bytes = have - used;
    return CK_OK;
}
int compaction_select_scan(ck_ctx *ctx, Slot &s, const Compaction &c, const u32 *lens)
{
    cudaStream_t st = s.stream;
    const u32 n = s.n;
    size_t tb = c.tmp_bytes;
    cub::CountingInputIterator<u32> ids(0);
    CK_CUDA(ctx, cub::DeviceSelect::Flagged(c.tmp, tb, ids, c.flags, c.sel, c.n_sel, (int)n, st));
    k_survivor_lens<<<(n + 256) / 256, 256, 0, st>>>(c.sel, c.n_sel, lens, n, c.len16);
    tb = c.tmp_bytes;
    CK_CUDA(ctx, cub::DeviceScan::ExclusiveSum(c.tmp, tb, c.len16, c.coff, (int)n + 1, st));
    ctx->launches += 3;
    CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts + 20, c.n_sel, 4, cudaMemcpyDeviceToHost, st));
    s.sel = c.sel; s.coff = c.coff;
    return CK_OK;
}

// CK_F_SURVIVORS: compact the batch's survivors on the device (indices, 16-byte-aligned compact offsets, canonical bytes); the
// compact bytes go to the byte arena d_norm (no byte-lane kernel is running any more).
int enqueue_compaction(ck_ctx *ctx, Slot &s, uint64_t base_index)
{
    cudaStream_t st = s.stream;
    const u32 n = s.n;
    Compaction c;
    int rc = compaction_carve(ctx, s, c);
    if (rc) return rc;
    k_survivor_flags<<<(n + 255) / 256, 256, 0, st>>>(s.d_first, base_index, n, c.flags);
    rc = compaction_select_scan(ctx, s, c, s.d_len);
    if (rc) return rc;
    if (!(s.flags & CK_F_NO_BYTES))
        k_gather_survivors<<<std::min<u32>((n + 7) / 8, 32u * (u32)ctx->num_sms), 256, 0, st>>>(c.sel, c.n_sel, s.d_len, s.d_off, s.d_out,
                                                                                               (s.flags & CK_F_ALIGNED_OUT) ? 1u : 0u, c.coff, s.d_norm);
    ctx->launches += 2;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}

// The device path of a monomerize batch whose raw bytes and offsets are in d_raw / d_off (ck_mono_submit copies them in,
// ck_fasta_submit splits them out of the text), in stream order on the slot's stream: normalise (k_prepare as ck_dev_normalize runs it: bytes to d_norm, lengths to d_len) -> k_monomerize -> k_mono_select ->
// compaction -> k_mono_gather.  Per record: the worker's end index in d_start, full_len in d_slotof and monomer_len in d_hash
// (as u32; no canonical form is computed for a monomerize batch).  The compact bytes go to d_out: they need up to
// offsets[n] + 15 n bytes, and d_out holds out_bytes_total(B, R) >= B + 32 R.
// The callers carve the compaction workspace (`c`) before they enqueue anything, so a refused batch leaves nothing running
// on the slot.
int enqueue_mono(ck_ctx *ctx, Slot &s, const Compaction &c, const ck_mono_options &o)
{
    cudaStream_t st = s.stream;
    const u32 n = s.n;
    const bool norm = s.flags & CK_F_NORMALIZE;
    u32 *end = s.d_start, *full_len = reinterpret_cast<u32 *>(s.d_slotof), *mono_len = reinterpret_cast<u32 *>(s.d_hash);
    int rc;
    if (norm) {
        PrepareArgs pa{s.d_raw, s.d_off, n, 1u | 2u | 4u, nullptr, s.d_norm, s.d_len, nullptr};
        k_prepare<<<ctx->num_sms * 32, 256, 0, st>>>(pa);
        ctx->launches++;
    }
    MonoArgs ma{};
    ma.bytes = norm ? s.d_norm : s.d_raw; ma.offsets = s.d_off; ma.lens = norm ? s.d_len : nullptr; ma.n_records = n;
    ma.seed_len = o.seed_len; ma.use_identity = o.overlap_min_identity >= 0.0 ? 1u : 0u; ma.overlap_dist = o.overlap_dist;
    ma.identity = o.overlap_min_identity; ma.flags = o.flags & (CK_MONO_SENSITIVE | CK_MONO_FIRST_ONLY); ma.out_end = end;
    k_monomerize<<<std::min<u32>((n + 7) / 8, 16u * (u32)ctx->num_sms), 256, 0, st>>>(ma);
    MonoSelectArgs sa{};
    sa.raw = s.d_raw; sa.offsets = s.d_off; sa.lens = norm ? s.d_len : nullptr; sa.n_records = n; sa.normalize = norm ? 1u : 0u;
    sa.keep_all = (o.flags & CK_MONO_KEEP_ALL) ? 1u : 0u; sa.seed_len = o.seed_len; sa.min_length = o.min_length;
    sa.max_length = o.max_length; sa.min_overlap = o.min_overlap; sa.min_overlap_percent = o.min_overlap_percent;
    sa.end = end; sa.full_len = full_len; sa.monomer_len = mono_len; sa.written = c.flags;
    const u32 grid = std::min<u32>((n + 7) / 8, 32u * (u32)ctx->num_sms);
    k_mono_select<<<grid, 256, 0, st>>>(sa);
    ctx->launches += 2;
    rc = compaction_select_scan(ctx, s, c, mono_len);
    if (rc) return rc;
    if (!(s.flags & CK_F_NO_BYTES)) {
        k_mono_gather<<<grid, 256, 0, st>>>(s.d_raw, s.d_off, c.sel, c.n_sel, mono_len, c.coff, norm ? 1u : 0u, s.d_out);
        ctx->launches++;
    }
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}

// shared back of every submit: the lane formats of the batch are in the slot (d_p2 / d_norm / d_len / d_lane); canonicalise,
// then (uniq) the first-occurrence table, then the small result copies
int submit_tail(ck_ctx *ctx, Slot &s, bool lens_given, uint64_t base_index)
{
    cudaStream_t st = s.stream;
    const u32 n_records = s.n, flags = s.flags;
    CanonIO io{};
    // without normalisation every byte is a symbol: lengths are the offset differences and the lane-per-record kernel applies
    io.packed2 = s.d_p2; io.bytes = s.d_norm; io.offsets = s.d_off; io.lens = lens_given ? s.d_len : nullptr; io.lane = s.d_lane;
    io.n = n_records; io.mode = (flags & CK_F_ALIGNED_OUT) ? 2u : 0u; io.dbl = s.dbl; io.p4 = s.d_p4; io.longest = s.longest;
    io.out = (flags & CK_F_NO_BYTES) ? nullptr : s.d_out;
    io.out_start = s.d_start; io.out_strand = s.d_strand; io.out_hash = s.d_hash;
    io.lists = s.d_lists; io.lists_bytes = lists_bytes_for(ctx->cfg.max_batch_records); io.counts = s.d_counts;
    const bool peer_mode = s.uniq && ctx->peer.attached && ctx->peer.world > 1;
    int rc = run_canon(ctx, st, s.scr, io, 0);
    if (rc) return rc;
    if (peer_mode) {
        // multi-GPU: this batch is one of a ROUND of batches, one per rank (include/circkit_b200.h, ck_peer_attach)
        const u32 slot = (u32)(&s - ctx->slot);
        cudaEvent_t prev = (ctx->have_last_insert && ctx->last_insert != s.inserted) ? ctx->last_insert : nullptr;
        rc = peer_first_index(ctx, st, slot, s.d_hash, n_records, base_index, ctx->table, ctx->table_slots, ctx->side, ctx->d_overflow,
                              s.d_first, s.inserted, prev);
        if (rc) return rc;
        ctx->last_insert = s.inserted; ctx->have_last_insert = true;
        CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts + 16, ctx->d_overflow, 4, cudaMemcpyDeviceToHost, st));
    } else if (s.uniq) {
        rc = table_insert(ctx, st, ctx->table, ctx->table_slots, ctx->side, ctx->d_overflow, s.d_hash, nullptr,
                          base_index, n_records, s.d_slotof, 1, ctx->d_keys);
        if (rc) return rc;
        CK_CUDA(ctx, cudaEventRecord(s.inserted, st));
        // first_index of this batch may point into the previous batch: wait for that batch's insert
        if (ctx->have_last_insert && ctx->last_insert != s.inserted) CK_CUDA(ctx, cudaStreamWaitEvent(st, ctx->last_insert, 0));
        ctx->last_insert = s.inserted; ctx->have_last_insert = true;
        rc = table_first(ctx, st, ctx->table, ctx->table_slots, ctx->side, s.d_slotof, n_records, s.d_first);
        if (rc) return rc;
        CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts + 16, ctx->d_overflow, 16, cudaMemcpyDeviceToHost, st));   // + d_keys
    }
    CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts, s.d_counts, 16 * 4, cudaMemcpyDeviceToHost, st));
    if (s.uniq && (flags & CK_F_SURVIVORS)) {
        rc = enqueue_compaction(ctx, s, base_index);
        if (rc) return rc;
    }
    s.busy = true;
    return CK_OK;
}

// an empty batch: nothing to do, except that in a peer group it still is this rank's part of the round (the barriers of
// the exchange are collective)
int submit_empty(ck_ctx *ctx, Slot &s, uint64_t base_index)
{
    s.busy = true;
    if (!(s.uniq && ctx->peer.attached && ctx->peer.world > 1)) return CK_OK;
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    const u32 slot = (u32)(&s - ctx->slot);
    cudaEvent_t prev = (ctx->have_last_insert && ctx->last_insert != s.inserted) ? ctx->last_insert : nullptr;
    int rc = peer_first_index(ctx, s.stream, slot, s.d_hash, 0, base_index, ctx->table, ctx->table_slots, ctx->side, ctx->d_overflow,
                              s.d_first, s.inserted, prev);
    if (rc) { s.busy = false; return rc; }
    ctx->last_insert = s.inserted; ctx->have_last_insert = true;
    return CK_OK;
}

// canonicalize / uniq over raw bytes and offsets already in d_raw / d_off (ck_canon_submit / ck_uniq_submit copy them in,
// ck_fasta_submit splits them out of the text): k_prepare -> k_extend_packed2 -> submit_tail
int enqueue_canon(ck_ctx *ctx, Slot &s, uint64_t base_index)
{
    cudaStream_t st = s.stream;
    const u32 n_records = s.n, flags = s.flags;
    PrepareArgs pa{s.d_raw, s.d_off, n_records, (flags & CK_F_NORMALIZE) | (s.dbl << 2), s.d_p2, s.d_norm, s.d_len, s.d_lane};
    k_prepare<<<ctx->num_sms * 32, 256, 0, st>>>(pa);
    k_extend_packed2<<<extend_grid(ctx, n_records), 256, 0, st>>>(s.d_p2, s.d_off, s.d_len, s.d_lane, n_records, nullptr, s.dbl);
    ctx->launches += 2;
    return submit_tail(ctx, s, (flags & CK_F_NORMALIZE) != 0, base_index);
}

int submit_common(ck_ctx *ctx, int slot, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records,
                  uint32_t flags, bool uniq, uint64_t base_index)
{
    int rc = submit_check(ctx, slot, offsets, n_records, flags, uniq, bytes != nullptr);
    if (rc) return rc;
    Slot &s = ctx->slot[slot];
    if (n_records == 0) return submit_empty(ctx, s, base_index);
    const u64 total = s.total;
    cudaStream_t st = s.stream;
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    if (uniq && !ctx->peer.attached && (rc = table_reserve(ctx, s, n_records))) return rc;
    CK_CUDA(ctx, cudaMemcpyAsync(s.d_off, offsets, (size_t)(n_records + 1) * 8, cudaMemcpyHostToDevice, st));
    if (total) CK_CUDA(ctx, cudaMemcpyAsync(s.d_raw, bytes, total, cudaMemcpyHostToDevice, st));
    return enqueue_canon(ctx, s, base_index);
}

// CK_F_PACKED_IN: the batch arrives as the host packer (ck_pack2_host) left it -- 2 bits per base for the A/C/G/T records,
// bytes only for the others
int submit_packed(ck_ctx *ctx, int slot, const ck_packed_batch *b, uint32_t flags, bool uniq, uint64_t base_index)
{
    if (!ctx) return CK_ERR_ARG;
    if (!b) return fail(ctx, CK_ERR_ARG, "null batch");
    const u32 n_records = b->n_records;
    int rc = submit_check(ctx, slot, b->offsets, n_records, flags | CK_F_PACKED_IN, uniq, true);
    if (rc) return rc;
    Slot &s = ctx->slot[slot];
    if (n_records == 0) return submit_empty(ctx, s, base_index);
    if (!b->packed2 || !b->lens || !b->lane) return fail(ctx, CK_ERR_ARG, "null batch pointers");
    if (b->lane_bytes_total && (!b->lane_bytes || !b->lane_offsets)) return fail(ctx, CK_ERR_ARG, "byte-lane records without lane_bytes / lane_offsets");
    if (b->lane_bytes_total > ctx->cfg.max_batch_bytes) return fail(ctx, CK_ERR_ARG, "lane_bytes exceed max_batch_bytes");
    cudaStream_t st = s.stream;
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    if (uniq && !ctx->peer.attached && (rc = table_reserve(ctx, s, n_records))) return rc;
    CK_CUDA(ctx, cudaMemcpyAsync(s.d_off, b->offsets, (size_t)(n_records + 1) * 8, cudaMemcpyHostToDevice, st));
    CK_CUDA(ctx, cudaMemcpyAsync(s.d_len, b->lens, (size_t)n_records * 4, cudaMemcpyHostToDevice, st));
    CK_CUDA(ctx, cudaMemcpyAsync(s.d_lane, b->lane, (size_t)n_records, cudaMemcpyHostToDevice, st));
    CK_CUDA(ctx, cudaMemcpyAsync(s.d_dense, b->packed2, (size_t)ck_pack2_words(s.total, n_records) * 8, cudaMemcpyHostToDevice, st));
    k_extend_packed2<<<extend_grid(ctx, n_records), 256, 0, st>>>(s.d_p2, s.d_off, s.d_len, s.d_lane, n_records, s.d_dense, s.dbl);
    ctx->launches++;
    if (b->lane_bytes_total) {
        CK_CUDA(ctx, cudaMemcpyAsync(s.d_laneoff, b->lane_offsets, (size_t)(n_records + 1) * 8, cudaMemcpyHostToDevice, st));
        CK_CUDA(ctx, cudaMemcpyAsync(s.d_raw, b->lane_bytes, (size_t)b->lane_bytes_total, cudaMemcpyHostToDevice, st));
        k_scatter_lane_bytes<<<extend_grid(ctx, n_records), 256, 0, st>>>(s.d_raw, s.d_laneoff, s.d_off, s.d_len, s.d_lane, n_records, s.d_norm);
        ctx->launches++;
    }
    return submit_tail(ctx, s, true, base_index);
}

int wait_common(ck_ctx *ctx, int slot, bool uniq, uint8_t *out_bytes, uint32_t *out_len, uint32_t *out_start,
                uint8_t *out_strand, uint64_t *out_hash, uint64_t *out_first)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    Slot &s = ctx->slot[slot];
    if (!s.busy || s.uniq != uniq || s.mono || s.text || s.defl || s.bz) return fail(ctx, CK_ERR_STATE, "no matching submit on this slot");
    s.busy = false;
    if (s.n == 0) {
        if (uniq && ctx->peer.attached && ctx->peer.world > 1) CK_CUDA(ctx, cudaStreamSynchronize(s.stream));
        return CK_OK;
    }
    cudaStream_t st = s.stream;
    const size_t n = s.n;
    if (out_bytes && !(s.flags & CK_F_NO_BYTES) && s.total)
        CK_CUDA(ctx, cudaMemcpyAsync(out_bytes, s.d_out, (s.flags & CK_F_ALIGNED_OUT) ? ck_out_arena_bytes(s.total, s.n) : s.total,
                                     cudaMemcpyDeviceToHost, st));
    if (out_len) CK_CUDA(ctx, cudaMemcpyAsync(out_len, s.d_len, n * 4, cudaMemcpyDeviceToHost, st));
    if (out_start) CK_CUDA(ctx, cudaMemcpyAsync(out_start, s.d_start, n * 4, cudaMemcpyDeviceToHost, st));
    if (out_strand) CK_CUDA(ctx, cudaMemcpyAsync(out_strand, s.d_strand, n, cudaMemcpyDeviceToHost, st));
    if (out_hash) CK_CUDA(ctx, cudaMemcpyAsync(out_hash, s.d_hash, n * 8, cudaMemcpyDeviceToHost, st));
    if (out_first && uniq) CK_CUDA(ctx, cudaMemcpyAsync(out_first, s.d_first, n * 8, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    if (uniq) note_keys(ctx, s);
    if (s.h_counts[CLS_HUGE]) return fail(ctx, CK_ERR_TOO_LONG, "batch holds a record beyond the staged-length classes");
    if (uniq && s.h_counts[16]) return fail(ctx, CK_ERR_TABLE_FULL, "uniq table is full; raise table_capacity");
    return CK_OK;
}

}  // namespace

// =============================================================================================
static bool table_view(void *table, u64 bytes, TableSlot *&slots, u64 &nslots, u64 *&side, u32 *&overflow)
{
    if (!table || bytes < 64 + sizeof(TableSlot) * 16) return false;
    nslots = (bytes - 64) / sizeof(TableSlot);
    side = (u64 *)table; overflow = (u32 *)((u8 *)table + 8);
    slots = (TableSlot *)((u8 *)table + 64);
    return true;
}

extern "C" {

int ck_init(const ck_config *cfg, ck_ctx **out)
{
    if (!cfg || !out) return fail(nullptr, CK_ERR_ARG, "null argument");
    *out = nullptr;
    ck_ctx *ctx = new (std::nothrow) ck_ctx();
    if (!ctx) return fail(nullptr, CK_ERR_ARG, "out of host memory");
    ctx->cfg = *cfg;
    ctx->device = cfg->device;
    if (const char *dbg = getenv("CK_S3_DEBUG")) ctx->s3_debug = (u32)strtoul(dbg, nullptr, 0) & 0xff00u;
    if (const char *sk = getenv("CK_SEG_KERNEL")) ctx->seg_kernel = atoi(sk) != 0;
    if (const char *lk = getenv("CK_L4_KERNEL")) ctx->l4_kernel = atoi(lk) != 0;
    if (const char *lk = getenv("CK_LANE_KERNEL")) ctx->lane_kernel = atoi(lk) == 2 ? 2 : 3;
#define CK_INIT(call)                                                                          \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) { fail(nullptr, CK_ERR_CUDA, #call, e__); ck_destroy(ctx); return CK_ERR_CUDA; } \
    } while (0)
    CK_INIT(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CK_INIT(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->num_sms = prop.multiProcessorCount;
    Tables t; u8 secret[200];
    fill_tables(t, secret);
    CK_INIT(cudaMemcpyToSymbol(c_tab, &t, sizeof(t)));
    CK_INIT(cudaMemcpyToSymbol(c_secret, secret, sizeof(secret)));
    {
        u64 last[8], merge[8], mid[16];
        for (int i = 0; i < 8; i++) { memcpy(&last[i], secret + 121 + 8 * i, 8); memcpy(&merge[i], secret + 11 + 8 * i, 8); }
        for (int i = 0; i < 14; i++) memcpy(&mid[i], secret + 3 + 8 * i, 8);
        memcpy(&mid[14], secret + 119, 8); memcpy(&mid[15], secret + 127, 8);
        CK_INIT(cudaMemcpyToSymbol(c_lastsec, last, sizeof(last)));
        CK_INIT(cudaMemcpyToSymbol(c_mergesec, merge, sizeof(merge)));
        CK_INIT(cudaMemcpyToSymbol(c_midsec, mid, sizeof(mid)));
    }
    if (alloc_scratch(ctx, ctx->dev_scr)) { g_init_error = ctx->err; ck_destroy(ctx); return CK_ERR_CUDA; }
    if (alloc_scratch(ctx, ctx->lib_scr)) { g_init_error = ctx->err; ck_destroy(ctx); return CK_ERR_CUDA; }
    CK_INIT(cudaStreamCreateWithFlags(&ctx->lib_stream, cudaStreamNonBlocking));
    const u64 B = cfg->max_batch_bytes, R = cfg->max_batch_records;
    if (B || R) {
        for (int k = 0; k < 2; k++) {
            Slot &s = ctx->slot[k];
            CK_INIT(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
            CK_INIT(cudaEventCreateWithFlags(&s.inserted, cudaEventDisableTiming));
            CK_INIT(cudaMalloc(&s.d_raw, B + 16));
            CK_INIT(cudaMalloc(&s.d_norm, B + 16));
            CK_INIT(cudaMalloc(&s.d_out, out_bytes_total(B, R) + 64));
            CK_INIT(cudaMalloc(&s.d_p2, p2_words(B, R) * 8));
            CK_INIT(cudaMalloc(&s.d_p4, p4_bytes_total(B, R)));
            CK_INIT(cudaMalloc(&s.d_off, (R + 1) * 8));
            CK_INIT(cudaMalloc(&s.d_len, (R + 1) * 4));
            CK_INIT(cudaMalloc(&s.d_lane, R + 1));
            CK_INIT(cudaMalloc(&s.d_start, (R + 1) * 4));
            CK_INIT(cudaMalloc(&s.d_strand, R + 1));
            CK_INIT(cudaMalloc(&s.d_hash, (R + 1) * 8));
            CK_INIT(cudaMalloc(&s.d_first, (R + 1) * 8));
            CK_INIT(cudaMalloc(&s.d_slotof, (R + 1) * 8));
            CK_INIT(cudaMalloc(&s.d_lists, lists_bytes_for(R)));
            CK_INIT(cudaMalloc(&s.d_counts, 64 * 4));
            CK_INIT(cudaMalloc(&s.d_dense, ((B >> 5) + R + 2) * 8));
            CK_INIT(cudaMalloc(&s.d_laneoff, (R + 1) * 8));
            CK_INIT(cudaMallocHost(&s.h_counts, 32 * 4));
            memset(s.h_counts, 0, 32 * 4);
            if (alloc_scratch(ctx, s.scr)) { g_init_error = ctx->err; ck_destroy(ctx); return CK_ERR_CUDA; }
        }
    }
    CK_INIT(cudaMalloc(&ctx->side, 8));
    CK_INIT(cudaMalloc(&ctx->d_overflow, 16));
    CK_INIT(cudaMemset(ctx->d_overflow, 0, 16));
    ctx->d_keys = reinterpret_cast<u64 *>(ctx->d_overflow + 2);
    if (cfg->table_capacity) {
        ctx->table_slots = table_slots_for(cfg->table_capacity);
        CK_INIT(cudaMalloc(&ctx->table, ctx->table_slots * sizeof(TableSlot)));
        k_table_clear<<<ctx->num_sms * 4, 256>>>(ctx->table, ctx->table_slots, ctx->side);
        CK_INIT(cudaGetLastError());
    }
    CK_INIT(cudaDeviceSynchronize());
#undef CK_INIT
    *out = ctx;
    return CK_OK;
}

void ck_destroy(ck_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (int k = 0; k < 2; k++) {
        Slot &s = ctx->slot[k];
        void *ptrs[] = {s.d_raw, s.d_off, s.d_p2, s.d_norm, s.d_len, s.d_lane, s.d_out, s.d_start, s.d_strand,
                        s.d_hash, s.d_first, s.d_slotof, s.d_lists, s.d_counts, s.d_dense, s.d_laneoff, s.d_p4,
                        s.d_text, s.d_frame, s.d_rstart, s.d_head, s.d_seq, s.d_len64, s.d_fofs, s.d_meta, s.d_tiles};
        for (void *p : ptrs) if (p) cudaFree(p);
        if (s.h_counts) cudaFreeHost(s.h_counts);
        if (s.stream) cudaStreamDestroy(s.stream);
        {
            Slot::Deflate &z = s.z;
            void *zp[] = {z.buf, z.kA, z.kB, z.vA, z.vB, z.prev8, z.prev4, z.seg, z.out, z.result, z.tmp};
            for (void *p : zp) if (p) cudaFree(p);
            if (z.h_result) cudaFreeHost(z.h_result);
            if (z.stream) cudaStreamDestroy(z.stream);
        }
        {
            Slot::Bzip2 &z = s.bz2;
            void *zp[] = {z.in, z.rle, z.bid, z.flag, z.rank, z.sa, z.pos, z.pos2, z.valA, z.valB, z.hp, z.hs, z.keyA, z.keyB,
                          z.small, z.out, z.result, z.tmp};
            for (void *p : zp) if (p) cudaFree(p);
            if (z.h_host) cudaFreeHost(z.h_host);
            for (cudaEvent_t e : z.ev) if (e) cudaEventDestroy(e);
            if (z.stream) cudaStreamDestroy(z.stream);
        }
        if (s.inserted) cudaEventDestroy(s.inserted);
        free_scratch(s.scr);
    }
    free_scratch(ctx->dev_scr);
    free_scratch(ctx->lib_scr);
    if (ctx->lib_stream) cudaStreamDestroy(ctx->lib_stream);
    if (ctx->lib_h) cudaFreeHost(ctx->lib_h);
    if (ctx->lib_d) cudaFree(ctx->lib_d);
    {
        PeerGroup &P = ctx->peer;
        for (u32 r = 0; r < P.world && P.attached; r++) if (r != P.rank && P.mapped[r]) cudaIpcCloseMemHandle(P.mapped[r]);
        for (int k = 0; k < 2; k++) { if (P.pos[k]) cudaFree(P.pos[k]); if (P.cursors[k]) cudaFree(P.cursors[k]); if (P.slot_of[k]) cudaFree(P.slot_of[k]); }
        if (P.block) cudaFree(P.block);
    }
    if (ctx->table) cudaFree(ctx->table);
    if (ctx->side) cudaFree(ctx->side);
    if (ctx->d_overflow) cudaFree(ctx->d_overflow);
    delete ctx;
}

const char *ck_last_error(const ck_ctx *ctx) { return ctx ? ctx->err.c_str() : g_init_error.c_str(); }

void *ck_alloc_pinned(ck_ctx *ctx, size_t bytes)
{
    void *p = nullptr;
    if (ctx) cudaSetDevice(ctx->device);
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { if (ctx) ctx->err = "cudaMallocHost failed"; return nullptr; }
    return p;
}
void ck_free_pinned(ck_ctx *, void *p) { if (p) cudaFreeHost(p); }

int ck_canon_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records, uint32_t flags)
{
    return submit_common(ctx, slot, bytes, offsets, n_records, flags, false, 0);
}
int ck_canon_wait(ck_ctx *ctx, int slot, uint8_t *out_bytes, uint32_t *out_len, uint32_t *out_start,
                  uint8_t *out_strand, uint64_t *out_hash64)
{
    return wait_common(ctx, slot, false, out_bytes, out_len, out_start, out_strand, out_hash64, nullptr);
}
int ck_uniq_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records,
                   uint32_t flags, uint64_t base_index)
{
    return submit_common(ctx, slot, bytes, offsets, n_records, flags, true, base_index);
}
int ck_uniq_wait(ck_ctx *ctx, int slot, uint8_t *out_bytes, uint32_t *out_len, uint64_t *out_hash64, uint64_t *out_first_index)
{
    return wait_common(ctx, slot, true, out_bytes, out_len, nullptr, nullptr, out_hash64, out_first_index);
}
int ck_canon_submit_packed(ck_ctx *ctx, int slot, const ck_packed_batch *batch, uint32_t flags)
{
    return submit_packed(ctx, slot, batch, flags, false, 0);
}
int ck_uniq_submit_packed(ck_ctx *ctx, int slot, const ck_packed_batch *batch, uint32_t flags, uint64_t base_index)
{
    return submit_packed(ctx, slot, batch, flags, true, base_index);
}
int ck_peer_export(ck_ctx *ctx, uint32_t world, uint32_t rank, uint32_t max_records, void *handle_out)
{
    if (!ctx || !handle_out || world < 1 || world > 32 || rank >= world || !max_records || (u64)world * max_records > 0xffffffffull)
        return ctx ? fail(ctx, CK_ERR_ARG, "bad peer group arguments") : CK_ERR_ARG;
    PeerGroup &P = ctx->peer;
    if (P.exported) return fail(ctx, CK_ERR_STATE, "peer block already exported");
    if (ctx->grow_max) return fail(ctx, CK_ERR_STATE, "a context whose uniq table grows (ck_uniq_grow) cannot join a peer group");
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    P.world = world; P.rank = rank; P.cap = max_records;
    P.recv_bytes = ((u64)world * P.cap * 16 + 255) & ~255ull;
    P.ret_bytes = ((u64)world * P.cap * 8 + 255) & ~255ull;
    P.block_bytes = CK_PEER_HEADER_BYTES + 2 * P.recv_bytes + 2 * P.ret_bytes;
    CK_CUDA(ctx, cudaMalloc(&P.block, P.block_bytes));
    CK_CUDA(ctx, cudaMemset(P.block, 0, CK_PEER_HEADER_BYTES));
    for (int k = 0; k < 2; k++) {
        CK_CUDA(ctx, cudaMalloc(&P.pos[k], (size_t)P.cap * 4 + 16));
        CK_CUDA(ctx, cudaMalloc(&P.cursors[k], 64 * 4));
        CK_CUDA(ctx, cudaMalloc(&P.slot_of[k], (size_t)world * P.cap * 8 + 16));
    }
    CK_CUDA(ctx, cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    CK_CUDA(ctx, cudaIpcGetMemHandle(&h, P.block));
    static_assert(sizeof(cudaIpcMemHandle_t) == CK_PEER_HANDLE_BYTES, "handle size");
    memcpy(handle_out, &h, sizeof(h));
    P.exported = true;
    return CK_OK;
}
int ck_peer_attach(ck_ctx *ctx, const void *all_handles)
{
    if (!ctx || !all_handles) return ctx ? fail(ctx, CK_ERR_ARG, "null argument") : CK_ERR_ARG;
    PeerGroup &P = ctx->peer;
    if (!P.exported || P.attached) return fail(ctx, CK_ERR_STATE, "ck_peer_export first, attach once");
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    for (u32 r = 0; r < P.world; r++) {
        if (r == P.rank) { P.mapped[r] = P.block; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const u8 *)all_handles + (size_t)r * CK_PEER_HANDLE_BYTES, sizeof(h));
        CK_CUDA(ctx, cudaIpcOpenMemHandle(&P.mapped[r], h, cudaIpcMemLazyEnablePeerAccess));
    }
    P.attached = true;
    return CK_OK;
}
int ck_dev_peer_first_index(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index, void *table,
                            uint64_t table_bytes, uint64_t *out_first_index)
{
    TableSlot *slots; u64 nslots; u64 *side; u32 *ov;
    if (!ctx || !table_view(table, table_bytes, slots, nslots, side, ov)) return ctx ? fail(ctx, CK_ERR_ARG, "bad table") : CK_ERR_ARG;
    if (n && (!hash64 || !out_first_index)) return fail(ctx, CK_ERR_ARG, "null argument");
    return peer_first_index(ctx, (cudaStream_t)stream, 0, U(hash64), n, base_index, slots, nslots, side, ov, U(out_first_index), nullptr, nullptr);
}
int ck_uniq_wait_survivors(ck_ctx *ctx, int slot, uint32_t *out_n_survivors, uint32_t *out_index, uint64_t *out_compact_offsets,
                           uint8_t *out_compact_bytes, uint32_t *out_len, uint64_t *out_hash64, uint64_t *out_first_index)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    Slot &s = ctx->slot[slot];
    if (!s.busy || !s.uniq || s.text) return fail(ctx, CK_ERR_STATE, "no matching submit on this slot");
    if (!out_n_survivors) return fail(ctx, CK_ERR_ARG, "null argument");
    if (s.n && !(s.flags & CK_F_SURVIVORS)) return fail(ctx, CK_ERR_STATE, "the batch was not submitted with CK_F_SURVIVORS");
    *out_n_survivors = 0;
    cudaStream_t st = s.stream;
    const size_t n = s.n;
    if (n == 0) return wait_common(ctx, slot, true, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
    // everything that is per record first (same as ck_uniq_wait, without the canonical bytes of all records) ...
    if (out_len) CK_CUDA(ctx, cudaMemcpyAsync(out_len, s.d_len, n * 4, cudaMemcpyDeviceToHost, st));
    if (out_hash64) CK_CUDA(ctx, cudaMemcpyAsync(out_hash64, s.d_hash, n * 8, cudaMemcpyDeviceToHost, st));
    if (out_first_index) CK_CUDA(ctx, cudaMemcpyAsync(out_first_index, s.d_first, n * 8, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    s.busy = false;
    note_keys(ctx, s);
    if (s.h_counts[CLS_HUGE]) return fail(ctx, CK_ERR_TOO_LONG, "batch holds a record beyond the staged-length classes");
    if (s.h_counts[16]) return fail(ctx, CK_ERR_TABLE_FULL, "uniq table is full; raise table_capacity");
    // ... then what the survivors need, sized by their number
    const u32 ns = s.h_counts[20];
    *out_n_survivors = ns;
    if (ns == 0) return CK_OK;
    u64 bytes = 0;
    if (out_index) CK_CUDA(ctx, cudaMemcpyAsync(out_index, s.sel, (size_t)ns * 4, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaMemcpyAsync(&bytes, s.coff + ns, 8, cudaMemcpyDeviceToHost, st));
    if (out_compact_offsets) CK_CUDA(ctx, cudaMemcpyAsync(out_compact_offsets, s.coff, ((size_t)ns + 1) * 8, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    if (out_compact_bytes && !(s.flags & CK_F_NO_BYTES) && bytes) {
        CK_CUDA(ctx, cudaMemcpyAsync(out_compact_bytes, s.d_norm, bytes, cudaMemcpyDeviceToHost, st));
        CK_CUDA(ctx, cudaStreamSynchronize(st));
    }
    return CK_OK;
}
int ck_uniq_reset(ck_ctx *ctx)
{
    if (!ctx) return CK_ERR_ARG;
    if (!ctx->table) return CK_OK;
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    CK_CUDA(ctx, cudaDeviceSynchronize());
    k_table_clear<<<ctx->num_sms * 4, 256>>>(ctx->table, ctx->table_slots, ctx->side);
    ctx->launches++;
    CK_CUDA(ctx, cudaMemset(ctx->d_overflow, 0, 16));   // and d_keys
    CK_CUDA(ctx, cudaDeviceSynchronize());
    ctx->have_last_insert = false;
    ctx->known_keys = 0; ctx->known_rec = ctx->submitted_rec;
    return CK_OK;
}

int ck_uniq_grow(ck_ctx *ctx, uint64_t max_keys)
{
    if (!ctx) return CK_ERR_ARG;
    if (!ctx->table) return fail(ctx, CK_ERR_STATE, "context was created with table_capacity 0");
    if (ctx->peer.exported) return fail(ctx, CK_ERR_STATE, "the tables of a peer group do not grow");
    ctx->grow_max = max_keys;
    return CK_OK;
}

int ck_uniq_table_info(ck_ctx *ctx, uint64_t *out_keys, uint64_t *out_capacity_keys, uint64_t *out_grows)
{
    if (!ctx) return CK_ERR_ARG;
    u64 keys = 0;
    if (ctx->table) {
        CK_CUDA(ctx, cudaSetDevice(ctx->device));
        for (Slot &o : ctx->slot) if (o.stream) CK_CUDA(ctx, cudaStreamSynchronize(o.stream));
        CK_CUDA(ctx, cudaMemcpy(&keys, ctx->d_keys, 8, cudaMemcpyDeviceToHost));
    }
    if (out_keys) *out_keys = keys;
    if (out_capacity_keys) *out_capacity_keys = table_capacity_keys(ctx->table_slots);
    if (out_grows) *out_grows = ctx->grows;
    return CK_OK;
}

int ck_mono_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records, uint32_t flags,
                   const ck_mono_options *opt)
{
    if (!ctx) return CK_ERR_ARG;
    int rc = mono_options_check(ctx, opt);
    if (rc) return rc;
    if (flags & ~(CK_F_NORMALIZE | CK_F_NO_BYTES)) return fail(ctx, CK_ERR_ARG, "flags must be CK_F_NORMALIZE / CK_F_NO_BYTES");
    rc = submit_check(ctx, slot, offsets, n_records, flags, false, bytes != nullptr, true);
    if (rc) return rc;
    Slot &s = ctx->slot[slot];
    s.mono = true;
    if (n_records == 0) return submit_empty(ctx, s, 0);
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    Compaction c;
    if ((rc = compaction_carve(ctx, s, c))) return rc;
    cudaStream_t st = s.stream;
    CK_CUDA(ctx, cudaMemcpyAsync(s.d_off, offsets, (size_t)(n_records + 1) * 8, cudaMemcpyHostToDevice, st));
    if (s.total) CK_CUDA(ctx, cudaMemcpyAsync(s.d_raw, bytes, s.total, cudaMemcpyHostToDevice, st));
    rc = enqueue_mono(ctx, s, c, *opt);
    if (rc) return rc;
    s.busy = true;
    return CK_OK;
}
int ck_mono_wait(ck_ctx *ctx, int slot, uint32_t *out_n_written, uint32_t *out_index, uint64_t *out_compact_offsets,
                 uint8_t *out_compact_bytes, uint32_t *out_monomer_len, uint32_t *out_full_len, uint32_t *out_end_index)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    Slot &s = ctx->slot[slot];
    if (!s.busy || !s.mono || s.text) return fail(ctx, CK_ERR_STATE, "no matching submit on this slot");
    s.busy = false;
    if (out_n_written) *out_n_written = 0;
    const size_t n = s.n;
    if (n == 0) return CK_OK;
    cudaStream_t st = s.stream;
    if (out_monomer_len) CK_CUDA(ctx, cudaMemcpyAsync(out_monomer_len, s.d_hash, n * 4, cudaMemcpyDeviceToHost, st));
    if (out_full_len) CK_CUDA(ctx, cudaMemcpyAsync(out_full_len, s.d_slotof, n * 4, cudaMemcpyDeviceToHost, st));
    if (out_end_index) CK_CUDA(ctx, cudaMemcpyAsync(out_end_index, s.d_start, n * 4, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    const u32 nw = s.h_counts[20];
    if (out_n_written) *out_n_written = nw;
    if (nw == 0) return CK_OK;
    u64 bytes = 0;
    if (out_index) CK_CUDA(ctx, cudaMemcpyAsync(out_index, s.sel, (size_t)nw * 4, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaMemcpyAsync(&bytes, s.coff + nw, 8, cudaMemcpyDeviceToHost, st));
    if (out_compact_offsets) CK_CUDA(ctx, cudaMemcpyAsync(out_compact_offsets, s.coff, ((size_t)nw + 1) * 8, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    if (out_compact_bytes && !(s.flags & CK_F_NO_BYTES) && bytes) {
        CK_CUDA(ctx, cudaMemcpyAsync(out_compact_bytes, s.d_out, bytes, cudaMemcpyDeviceToHost, st));
        CK_CUDA(ctx, cudaStreamSynchronize(st));
    }
    return CK_OK;
}

// ---- FASTA text batches (ck_fasta_submit / ck_fasta_wait; csrc/ck_fasta.cuh) -----------------------
uint64_t ck_fasta_out_bytes(uint64_t text_bytes, uint32_t n_records) { return text_bytes + 2ull * n_records + 64; }

static int text_alloc(ck_ctx *ctx, Slot &s)
{
    const u64 B = ctx->cfg.max_batch_bytes, R = ctx->cfg.max_batch_records;
    const u64 tiles = (B + CK_FASTA_TILE - 1) / CK_FASTA_TILE + 1;
    // 64 bytes of slack past the text: the start masks read whole 16-byte words, the copies read one aligned word ahead
    if (!s.d_text) CK_CUDA(ctx, cudaMalloc(&s.d_text, B + 64));
    if (!s.d_frame) CK_CUDA(ctx, cudaMalloc(&s.d_frame, ck_fasta_out_bytes(B, (u32)R)));
    if (!s.d_rstart) CK_CUDA(ctx, cudaMalloc(&s.d_rstart, (R + 1) * 8));
    if (!s.d_head) CK_CUDA(ctx, cudaMalloc(&s.d_head, (R + 1) * 16));
    if (!s.d_seq) CK_CUDA(ctx, cudaMalloc(&s.d_seq, (R + 1) * 16));
    if (!s.d_len64) CK_CUDA(ctx, cudaMalloc(&s.d_len64, (R + 1) * 8));
    if (!s.d_fofs) CK_CUDA(ctx, cudaMalloc(&s.d_fofs, (R + 1) * 8));
    if (!s.d_meta) CK_CUDA(ctx, cudaMalloc(&s.d_meta, 64));
    if (!s.d_tiles) CK_CUDA(ctx, cudaMalloc(&s.d_tiles, 2 * tiles * 4));
    return CK_OK;
}

// Record split of the text in d_text (nbytes >= 1): starts, ranges, the record count to h_counts[24] and the longest seq to
// h_counts[26..27]; the caller synchronises.  Scan temporaries live in the slot's sort workspace (free: the slot is idle).
static int enqueue_split(ck_ctx *ctx, Slot &s, u64 nbytes)
{
    cudaStream_t st = s.stream;
    const u32 R = ctx->cfg.max_batch_records;
    const u64 tiles = (nbytes + CK_FASTA_TILE - 1) / CK_FASTA_TILE;
    u32 *count = s.d_tiles, *off = s.d_tiles + tiles + 1;
    const size_t have = lists_bytes_for(R);
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, count, off, (int)(tiles + 1), st);
    if (need > have) return fail(ctx, CK_ERR_ARG, "sort workspace too small for the record split");
    k_fasta_count<<<(u32)tiles, 256, 0, st>>>(s.d_text, nbytes, count);
    CK_CUDA(ctx, cub::DeviceScan::ExclusiveSum(s.d_lists, need, count, off, (int)(tiles + 1), st));
    k_fasta_starts<<<(u32)tiles, 256, 0, st>>>(s.d_text, nbytes, off, R, s.d_rstart);
    CK_CUDA(ctx, cudaMemsetAsync(s.d_meta, 0, 8, st));
    FastaRangeArgs ra{s.d_text, nbytes, s.d_rstart, off + tiles, R, s.d_head, s.d_seq, s.d_len64, s.d_meta};
    k_fasta_ranges<<<std::min<u32>((R + 7) / 8, 32u * (u32)ctx->num_sms), 256, 0, st>>>(ra);
    ctx->launches += 4;
    CK_CUDA(ctx, cudaGetLastError());
    CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts + 24, off + tiles, 4, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts + 26, s.d_meta, 8, cudaMemcpyDeviceToHost, st));
    return CK_OK;
}

// Framing of the written records: c.sel / c.n_sel hold them (selected already), d_len64 takes the framed lengths, d_fofs their
// exclusive scan, d_frame the bytes; the byte count goes to h_counts[22..23].
static int enqueue_frame(ck_ctx *ctx, Slot &s, const Compaction &c, u32 body, const u64 *coff)
{
    cudaStream_t st = s.stream;
    const u32 n = s.n;
    FastaFrameArgs fa{};
    fa.text = s.d_text; fa.head = s.d_head; fa.seq = s.d_seq; fa.sel = c.sel; fa.n_sel = c.n_sel; fa.n = n; fa.body = body;
    fa.arena = s.d_out; fa.off = s.d_off; fa.coff = coff;
    fa.lens = body == CK_FRAME_COMPACT ? reinterpret_cast<const u32 *>(s.d_hash) : s.d_len;
    fa.flen = s.d_len64; fa.fofs = s.d_fofs; fa.frame = s.d_frame;
    k_fasta_frame_lens<<<(n + 256) / 256, 256, 0, st>>>(fa);
    size_t tb = c.tmp_bytes;
    CK_CUDA(ctx, cub::DeviceScan::ExclusiveSum(c.tmp, tb, s.d_len64, s.d_fofs, (int)n + 1, st));
    k_fasta_frame<<<std::min<u32>((n + 7) / 8, 32u * (u32)ctx->num_sms), 256, 0, st>>>(fa);
    ctx->launches += 3;
    CK_CUDA(ctx, cudaGetLastError());
    CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts + 22, s.d_fofs + n, 8, cudaMemcpyDeviceToHost, st));
    return CK_OK;
}

int ck_fasta_submit(ck_ctx *ctx, int slot, const uint8_t *text, uint64_t text_bytes, uint32_t command, uint32_t flags,
                    uint64_t base_index, const ck_mono_options *mono, uint32_t *out_n_records)
{
    if (!ctx) return CK_ERR_ARG;
    if (out_n_records) *out_n_records = 0;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    if (command < CK_CMD_CANONICALIZE || command > CK_CMD_MONOMERIZE) return fail(ctx, CK_ERR_ARG, "unknown command");
    const bool uniq = command == CK_CMD_UNIQ, is_mono = command == CK_CMD_MONOMERIZE;
    if (flags & ~(uniq ? CK_F_CANONICAL_BODY : 0u)) return fail(ctx, CK_ERR_ARG, "flags must be 0 (CK_F_CANONICAL_BODY: uniq only)");
    if (text_bytes && !text) return fail(ctx, CK_ERR_ARG, "null text");
    if (text_bytes && text[0] != '>') return fail(ctx, CK_ERR_ARG, "text must begin with '>'");
    if (text_bytes > ctx->cfg.max_batch_bytes) return fail(ctx, CK_ERR_ARG, "text exceeds max_batch_bytes");
    Slot &s = ctx->slot[slot];
    if (!s.stream) return fail(ctx, CK_ERR_STATE, "context was created without batch slots");
    if (s.busy) return fail(ctx, CK_ERR_STATE, "slot already holds a batch; call the matching wait first");
    if (uniq && !ctx->table) return fail(ctx, CK_ERR_STATE, "context was created with table_capacity 0");
    if (uniq && ctx->peer.attached) return fail(ctx, CK_ERR_STATE, "text batches do not run in a peer group");
    int rc;
    if (is_mono && (rc = mono_options_check(ctx, mono))) return rc;
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    if ((rc = text_alloc(ctx, s))) return rc;
    s.n = 0; s.total = 0; s.uniq = uniq; s.mono = is_mono; s.text = true; s.defl = false; s.bz = false; s.cmd = command;
    s.flags = CK_F_NORMALIZE | (is_mono ? 0u : CK_F_ALIGNED_OUT) | (uniq && !(flags & CK_F_CANONICAL_BODY) ? CK_F_NO_BYTES : 0u);
    if (text_bytes == 0) return submit_empty(ctx, s, base_index);
    cudaStream_t st = s.stream;
    CK_CUDA(ctx, cudaMemcpyAsync(s.d_text, text, text_bytes, cudaMemcpyHostToDevice, st));
    if ((rc = enqueue_split(ctx, s, text_bytes))) return rc;
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    const u32 n = s.h_counts[24];
    u64 longest;
    memcpy(&longest, s.h_counts + 26, 8);
    if (out_n_records) *out_n_records = n;
    if (n > ctx->cfg.max_batch_records) return fail(ctx, CK_ERR_ARG, "text holds more records than max_batch_records");
    if (is_mono && longest > kMonoMaxRecord) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^32 - 1024 bytes");
    if (!is_mono && longest > (1ull << 30)) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^30 symbols");
    s.n = n; s.longest = longest; s.dbl = longest > 512 ? 1u : 0u;   // as submit_check
    s.rec_mark = 0;
    if (uniq && (rc = table_reserve(ctx, s, n))) return rc;
    Compaction c;
    if ((rc = compaction_carve(ctx, s, c))) return rc;
    // the arena of the seq bytes, as the host-buffer entries receive it
    size_t tb = c.tmp_bytes;
    CK_CUDA(ctx, cub::DeviceScan::ExclusiveSum(c.tmp, tb, s.d_len64, s.d_off, (int)n + 1, st));
    k_fasta_gather<<<std::min<u32>((n + 7) / 8, 32u * (u32)ctx->num_sms), 256, 0, st>>>(s.d_text, s.d_seq, s.d_off, n, s.d_raw);
    ctx->launches += 2;
    if (is_mono) {
        if ((rc = enqueue_mono(ctx, s, c, *mono))) return rc;
        if ((rc = enqueue_frame(ctx, s, c, CK_FRAME_COMPACT, c.coff))) return rc;
    } else {
        if ((rc = enqueue_canon(ctx, s, base_index))) return rc;   // leaves the slot busy
        // the written records: all (canonicalize) or the first occurrences (uniq)
        if (uniq) { k_survivor_flags<<<(n + 255) / 256, 256, 0, st>>>(s.d_first, base_index, n, c.flags); ctx->launches++; }
        else CK_CUDA(ctx, cudaMemsetAsync(c.flags, 1, n, st));
        size_t sb = c.tmp_bytes;
        cub::CountingInputIterator<u32> ids(0);
        CK_CUDA(ctx, cub::DeviceSelect::Flagged(c.tmp, sb, ids, c.flags, c.sel, c.n_sel, (int)n, st));
        CK_CUDA(ctx, cudaMemcpyAsync(s.h_counts + 20, c.n_sel, 4, cudaMemcpyDeviceToHost, st));
        s.sel = c.sel;
        ctx->launches++;
        if ((rc = enqueue_frame(ctx, s, c, (s.flags & CK_F_NO_BYTES) ? CK_FRAME_RAW : CK_FRAME_CANON, nullptr))) return rc;
    }
    s.busy = true;
    return CK_OK;
}

int ck_fasta_wait(ck_ctx *ctx, int slot, uint8_t *out_fasta, uint64_t *out_fasta_bytes, uint32_t *out_n_written,
                  uint32_t *out_index, uint64_t *out_head, uint64_t *out_first_index, uint32_t *out_full_len,
                  uint32_t *out_monomer_len)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    Slot &s = ctx->slot[slot];
    if (!s.busy || !s.text) return fail(ctx, CK_ERR_STATE, "no matching submit on this slot");
    s.busy = false;
    if (out_fasta_bytes) *out_fasta_bytes = 0;
    if (out_n_written) *out_n_written = 0;
    const size_t n = s.n;
    if (n == 0) return CK_OK;
    cudaStream_t st = s.stream;
    if (out_head) CK_CUDA(ctx, cudaMemcpyAsync(out_head, s.d_head, n * 16, cudaMemcpyDeviceToHost, st));
    if (out_first_index && s.uniq) CK_CUDA(ctx, cudaMemcpyAsync(out_first_index, s.d_first, n * 8, cudaMemcpyDeviceToHost, st));
    if (out_full_len && s.mono) CK_CUDA(ctx, cudaMemcpyAsync(out_full_len, s.d_slotof, n * 4, cudaMemcpyDeviceToHost, st));
    if (out_monomer_len && s.mono) CK_CUDA(ctx, cudaMemcpyAsync(out_monomer_len, s.d_hash, n * 4, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    if (s.uniq) note_keys(ctx, s);
    if (!s.mono && s.h_counts[CLS_HUGE]) return fail(ctx, CK_ERR_TOO_LONG, "batch holds a record beyond the staged-length classes");
    if (s.uniq && s.h_counts[16]) return fail(ctx, CK_ERR_TABLE_FULL, "uniq table is full; raise table_capacity");
    const u32 nw = s.h_counts[20];
    u64 bytes;
    memcpy(&bytes, s.h_counts + 22, 8);
    if (out_n_written) *out_n_written = nw;
    if (out_fasta_bytes) *out_fasta_bytes = bytes;
    if (out_index && nw) CK_CUDA(ctx, cudaMemcpyAsync(out_index, s.sel, (size_t)nw * 4, cudaMemcpyDeviceToHost, st));
    if (out_fasta && bytes) CK_CUDA(ctx, cudaMemcpyAsync(out_fasta, s.d_frame, bytes, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    return CK_OK;
}

// ---- DEFLATE (ck_deflate_submit / ck_deflate_wait; csrc/ck_deflate.cuh) ------------------------------------------------
// stored blocks of 65 535 bytes (two per segment), an empty stored block after the last segment, and whole words for the
// pack kernel's edge stores
uint64_t ck_deflate_bound(uint64_t n) { return n + 10 * ((n + CKZ_SEG - 1) / CKZ_SEG) + 16; }

static u64 cap_segs(const Slot::Deflate &z) { return z.cap / CKZ_SEG; }

static int deflate_alloc(ck_ctx *ctx, Slot::Deflate &z, u64 n)
{
    if (!z.stream) CK_CUDA(ctx, cudaStreamCreateWithFlags(&z.stream, cudaStreamNonBlocking));
    if (!z.h_result) CK_CUDA(ctx, cudaMallocHost(&z.h_result, 16));
    if (z.cap >= n) return CK_OK;
    u64 cap = 1ull << 20;
    while (cap < n) cap <<= 1;
    cap = std::min<u64>(cap, CK_DEFLATE_MAX_BYTES);
    CK_CUDA(ctx, cudaStreamSynchronize(z.stream));
    void *zp[] = {z.buf, z.kA, z.kB, z.vA, z.vB, z.prev8, z.prev4, z.seg, z.out, z.result, z.tmp};
    for (void *p : zp) if (p) cudaFree(p);
    cudaStream_t keep_stream = z.stream;
    u32 *keep_result = z.h_result;
    z = Slot::Deflate{};
    z.stream = keep_stream; z.h_result = keep_result;
    const u64 N = cap + CK_DEFLATE_DICT_BYTES, segs = cap / CKZ_SEG;
    CK_CUDA(ctx, cudaMalloc(&z.buf, N + 64));
    for (u32 **p : {&z.kA, &z.kB, &z.vA, &z.vB, &z.prev8, &z.prev4}) CK_CUDA(ctx, cudaMalloc(p, N * 4));
    CK_CUDA(ctx, cudaMalloc(&z.seg, segs * (2 * CKZ_SYMS + CKZ_HDR_WORDS + 8) * 4 + 64));
    CK_CUDA(ctx, cudaMalloc(&z.out, (ck_deflate_bound(cap) + 7) / 4 * 4));
    CK_CUDA(ctx, cudaMalloc(&z.result, 16));
    cub::DoubleBuffer<u32> k(z.kA, z.kB), v(z.vA, z.vB);
    size_t tb = 0;
    CK_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tb, k, v, (int)N, 0, CKZ_HBITS, z.stream));
    CK_CUDA(ctx, cudaMalloc(&z.tmp, tb));
    z.tmp_bytes = tb;
    z.cap = cap;
    return CK_OK;
}

// hash chains of one key width over buf[0, N): keys, stable radix sort, links
static int deflate_chain(ck_ctx *ctx, Slot::Deflate &z, u32 N, u32 width, u32 *prev)
{
    cudaStream_t st = z.stream;
    const u32 g = (N + 255) / 256;
    k_defl_keys<<<g, 256, 0, st>>>(z.buf, N, width, z.kA, z.vA);
    cub::DoubleBuffer<u32> k(z.kA, z.kB), v(z.vA, z.vB);
    size_t tb = z.tmp_bytes;
    CK_CUDA(ctx, cub::DeviceRadixSort::SortPairs(z.tmp, tb, k, v, (int)N, 0, CKZ_HBITS, st));
    k_defl_links<<<g, 256, 0, st>>>(k.Current(), v.Current(), N, prev);
    ctx->launches += 3;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}

int ck_deflate_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, uint64_t n, const uint8_t *dict, uint32_t dict_bytes,
                      uint32_t crc_in)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    if (n == 0 || n > CK_DEFLATE_MAX_BYTES) return fail(ctx, CK_ERR_ARG, "n must be 1 .. CK_DEFLATE_MAX_BYTES");
    if (dict_bytes > CK_DEFLATE_DICT_BYTES) return fail(ctx, CK_ERR_ARG, "dict_bytes exceeds CK_DEFLATE_DICT_BYTES");
    if (!bytes || (dict_bytes && !dict)) return fail(ctx, CK_ERR_ARG, "null argument");
    Slot &s = ctx->slot[slot];
    if (s.busy) return fail(ctx, CK_ERR_STATE, "slot already holds a batch; call the matching wait first");
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot::Deflate &z = s.z;
    int rc;
    if ((rc = deflate_alloc(ctx, z, n))) return rc;
    cudaStream_t st = z.stream;
    const u32 D = dict_bytes, N = (u32)(D + n), nseg = (u32)((n + CKZ_SEG - 1) / CKZ_SEG);
    if (D) CK_CUDA(ctx, cudaMemcpyAsync(z.buf, dict, D, cudaMemcpyHostToDevice, st));
    CK_CUDA(ctx, cudaMemcpyAsync(z.buf + D, bytes, n, cudaMemcpyHostToDevice, st));
    CK_CUDA(ctx, cudaMemsetAsync(z.buf + N, 0, 64, st));
    if ((rc = deflate_chain(ctx, z, N, 8, z.prev8))) return rc;
    if ((rc = deflate_chain(ctx, z, N, 4, z.prev4))) return rc;
    DeflateArgs a{};
    a.buf = z.buf; a.dict = D; a.n = (u32)n; a.nseg = nseg;
    a.prev8 = z.prev8; a.prev4 = z.prev4;
    a.match = z.kA; a.tok = z.kB;                       // the sort buffers are free again
    const u64 S = cap_segs(z);
    a.freq = z.seg; a.table = a.freq + S * CKZ_SYMS; a.hdr = a.table + S * CKZ_SYMS; a.meta = a.hdr + S * CKZ_HDR_WORDS;
    a.seg_crc = a.meta + 4 * S; a.ntok = a.seg_crc + S;
    a.off = reinterpret_cast<u64 *>(a.ntok + S);        // S is even: 8-byte aligned
    a.out = z.out; a.result = z.result; a.crc_in = crc_in;
    k_defl_match<<<nseg, 256, 0, st>>>(a);
    k_defl_parse<<<nseg, 128, 0, st>>>(a);
    k_defl_huff<<<nseg, 256, 0, st>>>(a);
    CK_CUDA(ctx, cudaMemsetAsync(z.out, 0, (ck_deflate_bound(n) + 7) / 4 * 4, st));
    k_defl_place<<<1, 1024, 0, st>>>(a);
    k_defl_pack<<<nseg, 256, 0, st>>>(a);
    ctx->launches += 5;
    CK_CUDA(ctx, cudaGetLastError());
    CK_CUDA(ctx, cudaMemcpyAsync(z.h_result, z.result, 12, cudaMemcpyDeviceToHost, st));
    z.n = n;
    s.busy = true; s.defl = true; s.bz = false; s.uniq = false; s.mono = false; s.text = false;
    return CK_OK;
}

int ck_deflate_wait(ck_ctx *ctx, int slot, uint8_t *out, uint64_t *out_bytes, uint32_t *crc_out)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    Slot &s = ctx->slot[slot];
    if (!s.busy || !s.defl) return fail(ctx, CK_ERR_STATE, "no matching submit on this slot");
    s.busy = false; s.defl = false;
    if (out_bytes) *out_bytes = 0;
    Slot::Deflate &z = s.z;
    CK_CUDA(ctx, cudaStreamSynchronize(z.stream));
    const u64 bytes = (u64)z.h_result[0] | (u64)z.h_result[1] << 32;
    if (bytes > ck_deflate_bound(z.n)) return fail(ctx, CK_ERR_CUDA, "deflate output exceeds its bound");
    if (out && bytes) {
        CK_CUDA(ctx, cudaMemcpyAsync(out, z.out, bytes, cudaMemcpyDeviceToHost, z.stream));
        CK_CUDA(ctx, cudaStreamSynchronize(z.stream));
    }
    if (out_bytes) *out_bytes = bytes;
    if (crc_out) *crc_out = z.h_result[2];
    return CK_OK;
}

// ---- bzip2 (ck_bzip2_submit / ck_bzip2_wait; csrc/ck_bzip2.cuh) --------------------------------------------------------
// at most 17 bits per MTF symbol, at most 5/4 RLE1 bytes per raw byte, and a header per block; every block but the last
// covers >= 4/5 * CKB_BLOCK_MAX raw bytes
uint64_t ck_bzip2_bound(uint64_t n) { return 3 * n + (n / (CKB_BLOCK_MAX * 4 / 5) + 2) * (CKB_HDR_WORDS * 4) + 64; }

// the fixed-size per-block arrays, carved from Slot::Bzip2::small
static size_t bzip2_layout(u8 *p, Bzip2Args *a)
{
    u8 *const p0 = p;
    auto take = [&p](size_t bytes) { u8 *q = p; p += (bytes + 255) / 256 * 256; return q; };
    Bzip2Block *blk = reinterpret_cast<Bzip2Block *>(take(CKB_MAX_BLOCKS * sizeof(Bzip2Block)));
    Bzip2Meta *meta = reinterpret_cast<Bzip2Meta *>(take(sizeof(Bzip2Meta)));
    u32 *freq = reinterpret_cast<u32 *>(take((size_t)CKB_MAX_BLOCKS * CKB_ALPHA * 4));
    u32 *code = reinterpret_cast<u32 *>(take((size_t)CKB_MAX_BLOCKS * CKB_GROUPS * CKB_ALPHA * 4));
    u32 *hdr = reinterpret_cast<u32 *>(take((size_t)CKB_MAX_BLOCKS * CKB_HDR_WORDS * 4));
    int *hb = reinterpret_cast<int *>(take((size_t)CKB_MAX_BLOCKS * CKB_GROUPS * sizeof(BzHeap)));
    u8 *sel = take((size_t)CKB_MAX_BLOCKS * CKB_MAX_SEL);
    if (a) { a->blk = blk; a->meta = meta; a->freq = freq; a->code = code; a->hdr = hdr; a->hb = hb; a->sel = sel; }
    return (size_t)(p - p0);
}

static int bzip2_alloc(ck_ctx *ctx, Slot::Bzip2 &z, u64 n)
{
    if (!z.stream) CK_CUDA(ctx, cudaStreamCreateWithFlags(&z.stream, cudaStreamNonBlocking));
    if (!z.h_host) CK_CUDA(ctx, cudaMallocHost(&z.h_host, 64));
    if (!z.ev[0]) for (cudaEvent_t &e : z.ev) CK_CUDA(ctx, cudaEventCreate(&e));
    if (!z.small) CK_CUDA(ctx, cudaMalloc(&z.small, bzip2_layout(nullptr, nullptr)));
    if (z.cap >= n) return CK_OK;
    u64 cap = 1ull << 20;
    while (cap < n) cap <<= 1;
    cap = std::min<u64>(cap, CK_BZIP2_MAX_BYTES);
    CK_CUDA(ctx, cudaStreamSynchronize(z.stream));
    void *zp[] = {z.in, z.rle, z.bid, z.flag, z.rank, z.sa, z.pos, z.pos2, z.valA, z.valB, z.hp, z.hs, z.keyA, z.keyB,
                  z.out, z.result, z.tmp};
    for (void *p : zp) if (p) cudaFree(p);
    z.in = z.rle = z.bid = z.flag = nullptr;
    z.rank = z.sa = z.pos = z.pos2 = z.valA = z.valB = z.hp = z.hs = nullptr;
    z.keyA = z.keyB = nullptr; z.out = z.result = nullptr; z.tmp = nullptr; z.cap = 0;
    const u64 R = cap + cap / 4 + 64;                   // RLE1 bytes: a run of 4 takes 5
    CK_CUDA(ctx, cudaMalloc(&z.in, cap + 64));
    for (u8 **p : {&z.rle, &z.bid, &z.flag}) CK_CUDA(ctx, cudaMalloc(p, R + 64));
    for (u32 **p : {&z.rank, &z.sa, &z.pos, &z.pos2, &z.valA, &z.valB, &z.hp, &z.hs}) CK_CUDA(ctx, cudaMalloc(p, R * 4));
    for (u64 **p : {&z.keyA, &z.keyB}) CK_CUDA(ctx, cudaMalloc(p, R * 8));
    CK_CUDA(ctx, cudaMalloc(&z.out, (ck_bzip2_bound(cap) + 7) / 4 * 4));
    CK_CUDA(ctx, cudaMalloc(&z.result, 16));
    size_t tb = 0, t1 = 0;
    cub::DoubleBuffer<u64> k(z.keyA, z.keyB);
    cub::DoubleBuffer<u32> v(z.valA, z.valB);
    CK_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, t1, k, v, (int)R, 0, 64, z.stream));
    tb = std::max(tb, t1);
    CK_CUDA(ctx, cub::DeviceScan::InclusiveScan(nullptr, t1, z.hp, z.hs, BzMax(), (int)R, z.stream));
    tb = std::max(tb, t1);
    CK_CUDA(ctx, cub::DeviceScan::InclusiveSum(nullptr, t1, z.pos2, z.valB, (int)R, z.stream));
    tb = std::max(tb, t1);
    CK_CUDA(ctx, cub::DeviceSelect::Flagged(nullptr, t1, z.pos, z.flag, z.pos2, z.result + 3, (int)R, z.stream));
    tb = std::max(tb, t1);
    CK_CUDA(ctx, cudaMalloc(&z.tmp, tb));
    z.tmp_bytes = tb;
    z.cap = cap; z.rcap = R;
    return CK_OK;
}

int ck_bzip2_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, uint64_t n, int final, uint32_t bits_in,
                    uint32_t nbits_in, uint32_t crc_in)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    if (n == 0 || n > CK_BZIP2_MAX_BYTES) return fail(ctx, CK_ERR_ARG, "n must be 1 .. CK_BZIP2_MAX_BYTES");
    if (nbits_in > 7) return fail(ctx, CK_ERR_ARG, "nbits_in must be 0 .. 7");
    if (!bytes) return fail(ctx, CK_ERR_ARG, "null argument");
    Slot &s = ctx->slot[slot];
    if (s.busy) return fail(ctx, CK_ERR_STATE, "slot already holds a batch; call the matching wait first");
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot::Bzip2 &z = s.bz2;
    int rc;
    if ((rc = bzip2_alloc(ctx, z, n))) return rc;
    cudaStream_t st = z.stream;
    Bzip2Args a{};
    bzip2_layout(z.small, &a);
    a.in = z.in; a.n = (u32)n; a.final = final ? 1 : 0;
    a.rs = z.hp; a.runst = z.hs; a.enc = z.pos2; a.cum = z.valB;     // stage 1 only: the sort buffers are free then
    a.rle = z.rle; a.bid = z.bid; a.sa = z.sa; a.rank = z.rank; a.last = z.flag;
    a.mtfv = reinterpret_cast<u16 *>(z.keyA);             // after the sort
    a.out = z.out; a.result = z.result;
    a.bits_in = bits_in & ((1u << nbits_in) - 1); a.nbits_in = nbits_in; a.crc_in = crc_in;
    const u32 n32 = (u32)n, g = (n32 + 255) / 256;
    CK_CUDA(ctx, cudaEventRecord(z.ev[0], st));
    CK_CUDA(ctx, cudaMemcpyAsync(z.in, bytes, n, cudaMemcpyHostToDevice, st));
    k_bz_runs<<<g, 256, 0, st>>>(z.in, n32, a.rs);
    size_t tb = z.tmp_bytes;
    CK_CUDA(ctx, cub::DeviceScan::InclusiveScan(z.tmp, tb, a.rs, a.runst, BzMax(), (int)n32, st));
    k_bz_tok<<<g, 256, 0, st>>>(a);
    tb = z.tmp_bytes;
    CK_CUDA(ctx, cub::DeviceScan::InclusiveSum(z.tmp, tb, a.enc, a.cum, (int)n32, st));
    k_bz_cuts<<<1, 1, 0, st>>>(a);
    ctx->launches += 5;
    CK_CUDA(ctx, cudaGetLastError());
    CK_CUDA(ctx, cudaMemcpyAsync(z.h_host, a.meta, sizeof(Bzip2Meta), cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    Bzip2Meta m;
    memcpy(&m, z.h_host, sizeof m);
    z.n = n; z.nblk = m.nblk; z.consumed = m.consumed; z.rounds = 0;
    z.bits_in = a.bits_in; z.nbits_in = nbits_in; z.crc_in = crc_in;
    if (m.nblk) {
        const u32 N = m.nrle, nb = m.nblk, G = (N + 255) / 256;
        k_bz_gather<<<(m.consumed + 255) / 256, 256, 0, st>>>(a, m.consumed);
        k_bz_crc<<<nb, 1024, 0, st>>>(a);
        CK_CUDA(ctx, cudaEventRecord(z.ev[1], st));
        // BWT: the first sort over (block, 7 bytes), then rounds over the groups not yet split
        u32 rbits = 1, bbits = 1;
        while ((1ull << rbits) < N) rbits++;
        while ((1u << bbits) < nb) bbits++;
        u32 *pos = z.pos, *pos2 = z.pos2;
        k_bz_key0<<<G, 256, 0, st>>>(a, nb, N, z.keyA, z.valA, pos);
        ctx->launches += 3;
        u32 mcount = N, sorted = CKB_KEY0_CHARS;
        for (bool first = true; mcount; first = false) {
            const u32 gm = (mcount + 255) / 256;
            if (!first) { k_bz_key<<<gm, 256, 0, st>>>(a, mcount, pos, sorted, rbits, z.keyA, z.valA); ctx->launches++; }
            const u32 after = first ? sorted : 2 * sorted;     // bytes the rotations are sorted by after this round
            cub::DoubleBuffer<u64> kb(z.keyA, z.keyB);
            cub::DoubleBuffer<u32> vb(z.valA, z.valB);
            tb = z.tmp_bytes;
            CK_CUDA(ctx, cub::DeviceRadixSort::SortPairs(z.tmp, tb, kb, vb, (int)mcount, 0,
                                                         first ? (int)(8 * CKB_KEY0_CHARS + bbits) : (int)(2 * rbits), st));
            k_bz_mark<<<gm, 256, 0, st>>>(a, mcount, kb.Current(), vb.Current(), pos, z.hp);
            tb = z.tmp_bytes;
            CK_CUDA(ctx, cub::DeviceScan::InclusiveScan(z.tmp, tb, z.hp, z.hs, BzMax(), (int)mcount, st));
            k_bz_rank<<<gm, 256, 0, st>>>(a, mcount, kb.Current(), vb.Current(), pos, z.hs, after, z.flag);
            tb = z.tmp_bytes;
            CK_CUDA(ctx, cub::DeviceSelect::Flagged(z.tmp, tb, pos, z.flag, pos2, z.result + 3, (int)mcount, st));
            ctx->launches += 5;
            CK_CUDA(ctx, cudaGetLastError());
            CK_CUDA(ctx, cudaMemcpyAsync(z.h_host + 8, z.result + 3, 4, cudaMemcpyDeviceToHost, st));
            CK_CUDA(ctx, cudaStreamSynchronize(st));
            mcount = z.h_host[8];
            std::swap(pos, pos2);
            sorted = after;
            z.rounds++;
        }
        k_bz_orig<<<G, 256, 0, st>>>(a, N);
        k_bz_periodic<<<nb, 1, 0, st>>>(a, z.hp);
        CK_CUDA(ctx, cudaEventRecord(z.ev[2], st));
        k_bz_mtf<<<nb, 256, 0, st>>>(a);
        CK_CUDA(ctx, cudaEventRecord(z.ev[3], st));
        k_bz_huff<<<nb, 256, 0, st>>>(a);
        CK_CUDA(ctx, cudaEventRecord(z.ev[4], st));
        CK_CUDA(ctx, cudaMemsetAsync(z.out, 0, (ck_bzip2_bound(n) + 7) / 4 * 4, st));
        k_bz_place<<<1, CKB_MAX_BLOCKS, 0, st>>>(a, nb);
        k_bz_pack<<<nb, 256, 0, st>>>(a);
        CK_CUDA(ctx, cudaEventRecord(z.ev[5], st));
        ctx->launches += 7;
        CK_CUDA(ctx, cudaGetLastError());
        CK_CUDA(ctx, cudaMemcpyAsync(z.h_host + 4, z.result, 12, cudaMemcpyDeviceToHost, st));
    }
    s.busy = true; s.bz = true; s.defl = false; s.uniq = false; s.mono = false; s.text = false;
    return CK_OK;
}

int ck_bzip2_wait(ck_ctx *ctx, int slot, uint8_t *out, uint64_t *out_bytes, uint64_t *consumed, uint32_t *bits_out,
                  uint32_t *nbits_out, uint32_t *crc_out)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    Slot &s = ctx->slot[slot];
    if (!s.busy || !s.bz) return fail(ctx, CK_ERR_STATE, "no matching submit on this slot");
    if (!out) return fail(ctx, CK_ERR_ARG, "null argument");
    s.busy = false; s.bz = false;
    Slot::Bzip2 &z = s.bz2;
    CK_CUDA(ctx, cudaStreamSynchronize(z.stream));
    u64 whole = 0, cons = 0;
    u32 bits = z.bits_in, nbits = z.nbits_in, crc = z.crc_in;
    if (z.nblk) {
        const u64 total = (u64)z.h_host[4] | (u64)z.h_host[5] << 32, copy = (total + 7) / 8;
        if (copy > ck_bzip2_bound(z.n)) return fail(ctx, CK_ERR_CUDA, "bzip2 output exceeds its bound");
        CK_CUDA(ctx, cudaMemcpyAsync(out, z.out, copy, cudaMemcpyDeviceToHost, z.stream));
        CK_CUDA(ctx, cudaStreamSynchronize(z.stream));
        whole = total / 8;
        nbits = (u32)(total % 8);
        bits = nbits ? out[whole] >> (8 - nbits) : 0;
        crc = z.h_host[6];
        cons = z.consumed;
    }
    if (out_bytes) *out_bytes = whole;
    if (consumed) *consumed = cons;
    if (bits_out) *bits_out = bits;
    if (nbits_out) *nbits_out = nbits;
    if (crc_out) *crc_out = crc;
    return CK_OK;
}

int ck_bzip2_stats(ck_ctx *ctx, int slot, float *stage_ms, uint32_t *bwt_rounds)
{
    if (!ctx) return CK_ERR_ARG;
    if (slot < 0 || slot > 1) return fail(ctx, CK_ERR_ARG, "slot must be 0 or 1");
    if (!stage_ms) return fail(ctx, CK_ERR_ARG, "null argument");
    Slot &s = ctx->slot[slot];
    if (s.busy && s.bz) return fail(ctx, CK_ERR_STATE, "call ck_bzip2_wait first");
    const Slot::Bzip2 &z = s.bz2;
    for (int k = 0; k < 5; k++) {
        stage_ms[k] = 0.f;
        if (z.nblk) CK_CUDA(ctx, cudaEventElapsedTime(&stage_ms[k], z.ev[k], z.ev[k + 1]));
    }
    if (bwt_rounds) *bwt_rounds = z.rounds;
    return CK_OK;
}

// ---- single-record / library-semantics entry points -------------------------------------------
// Small batches (the single-record calls above all): ONE launch of the generic CTA-per-record kernel on the raw bytes (the
// byte lane is library semantics by construction: bytes as they are, bio's 256-entry complement table), one copy in and
// one copy out through persistent pinned staging on the context's own stream -- no allocation, no default-stream round
// trip.  Larger batches take the full pipeline (k_prepare + lanes) with a workspace that is kept and grown on demand.
static int lib_reserve(ck_ctx *ctx, size_t h_bytes, size_t d_bytes)
{
    if (h_bytes > ctx->lib_h_bytes) {
        if (ctx->lib_h) cudaFreeHost(ctx->lib_h);
        ctx->lib_h = nullptr; ctx->lib_h_bytes = 0;
        const size_t want = std::max<size_t>(h_bytes * 2, 1 << 16);
        CK_CUDA(ctx, cudaMallocHost(&ctx->lib_h, want));
        ctx->lib_h_bytes = want;
    }
    if (d_bytes > ctx->lib_d_bytes) {
        if (ctx->lib_d) cudaFree(ctx->lib_d);
        ctx->lib_d = nullptr; ctx->lib_d_bytes = 0;
        const size_t want = std::max<size_t>(d_bytes * 2, 1 << 16);
        CK_CUDA(ctx, cudaMalloc(&ctx->lib_d, want));
        ctx->lib_d_bytes = want;
    }
    return CK_OK;
}
static int lib_batch(ck_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records, u32 mode,
                     uint8_t *out_bytes, uint32_t *out_start, uint8_t *out_strand)
{
    if (!ctx || !offsets) return ctx ? fail(ctx, CK_ERR_ARG, "null argument") : CK_ERR_ARG;
    if (n_records == 0) return CK_OK;
    const u64 total = offsets[n_records] - offsets[0];
    if (offsets[0] != 0) return fail(ctx, CK_ERR_ARG, "offsets[0] must be 0");
    if (total && !bytes) return fail(ctx, CK_ERR_ARG, "null argument");
    u64 longest = 0;
    for (u32 i = 0; i < n_records; i++) {
        if (offsets[i + 1] < offsets[i]) return fail(ctx, CK_ERR_ARG, "offsets must be non-decreasing");
        longest = std::max<u64>(longest, offsets[i + 1] - offsets[i]);
    }
    if (longest > (1ull << 30)) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^30 symbols");
    std::lock_guard<std::mutex> lock(ctx->lib_mu);
    CK_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = set_attrs(ctx);
    if (rc) return rc;
    cudaStream_t st = ctx->lib_stream;
    const size_t R = n_records;
    const size_t off_bytes = (R + 1) * 8, in_bytes = off_bytes + ((total + 15) & ~15ull);
    const size_t res_bytes = R * 4 + ((R + 15) & ~15ull) + total;             // start | strand | canonical bytes
    const bool small = n_records <= 256 && longest <= cls_max_n(CLS_C8);
    if (small) {
        if ((rc = lib_reserve(ctx, in_bytes + res_bytes + 64, in_bytes + res_bytes + 64))) return rc;
        u8 *h_in = ctx->lib_h, *h_res = ctx->lib_h + in_bytes;
        u8 *d_in = ctx->lib_d, *d_res = ctx->lib_d + in_bytes;
        memcpy(h_in, offsets, off_bytes);
        if (total) memcpy(h_in + off_bytes, bytes, total);
        CK_CUDA(ctx, cudaMemcpyAsync(d_in, h_in, off_bytes + total, cudaMemcpyHostToDevice, st));
        CanonArgs a{};
        a.bytes = d_in + off_bytes; a.offsets = reinterpret_cast<const u64 *>(d_in); a.n_direct = n_records;
        a.out_start = reinterpret_cast<u32 *>(d_res); a.out_strand = d_res + R * 4;
        a.out = out_bytes ? d_res + R * 4 + ((R + 15) & ~15ull) : nullptr;
        a.scratch = ctx->lib_scr.tie[CLS_C8]; a.scratch_stride = cls_tie_words(CLS_C8); a.smem_units = cls_units(CLS_C8);
        a.mode = mode; a.min_n = 1; a.max_n = cls_max_n(CLS_C8);
        const u32 grid = std::min<u32>(n_records, kCls[CLS_C8].ctas_per_sm * (u32)ctx->num_sms);
        k_canon_cta<8, false><<<grid, kCls[CLS_C8].threads, cls_smem_bytes(CLS_C8), st>>>(a);
        ctx->launches++;
        if (longest != offsets[n_records] / std::max<u32>(n_records, 1) || total == 0 || n_records > 1) {   // any empty record?
            bool any_empty = false;
            for (u32 i = 0; i < n_records && !any_empty; i++) any_empty = offsets[i + 1] == offsets[i];
            if (any_empty) { k_canon_empty<<<1, 256, 0, st>>>(a); ctx->launches++; }
        }
        CK_CUDA(ctx, cudaGetLastError());
        CK_CUDA(ctx, cudaMemcpyAsync(h_res, d_res, out_bytes ? res_bytes : R * 4 + R, cudaMemcpyDeviceToHost, st));
        CK_CUDA(ctx, cudaStreamSynchronize(st));
        if (out_start) memcpy(out_start, h_res, R * 4);
        if (out_strand) memcpy(out_strand, h_res + R * 4, R);
        if (out_bytes && total) memcpy(out_bytes, h_res + R * 4 + ((R + 15) & ~15ull), total);
        return CK_OK;
    }
    // the full pipeline; workspace: raw | norm | out | p2 | off | len | lane | start | strand | lists | counts
    size_t o = 0;
    auto take = [&](size_t bytes_) { const size_t at = o; o += (bytes_ + 255) & ~(size_t)255; return at; };
    const size_t o_raw = take(total + 16), o_norm = take(total + 16), o_out = take(total + 16), o_p2 = take(p2_words(total, R) * 8);
    const size_t o_off = take((R + 1) * 8), o_len = take(R * 4), o_lane = take(R), o_start = take(R * 4), o_strand = take(R);
    const size_t o_lists = take(lists_bytes_for(R)), o_counts = take(256);
    if ((rc = lib_reserve(ctx, 64, o))) return rc;
    u8 *d = ctx->lib_d;
    u32 h_counts[16] = {};
    CK_CUDA(ctx, cudaMemcpyAsync(d + o_off, offsets, (R + 1) * 8, cudaMemcpyHostToDevice, st));
    if (total) CK_CUDA(ctx, cudaMemcpyAsync(d + o_raw, bytes, total, cudaMemcpyHostToDevice, st));
    PrepareArgs pa{d + o_raw, (u64 *)(d + o_off), n_records, 1u << 2, (u64 *)(d + o_p2), d + o_norm, (u32 *)(d + o_len), d + o_lane};
    k_prepare<<<ctx->num_sms * 32, 256, 0, st>>>(pa);
    k_extend_packed2<<<extend_grid(ctx, n_records), 256, 0, st>>>((u64 *)(d + o_p2), (u64 *)(d + o_off), (u32 *)(d + o_len), d + o_lane, n_records, nullptr, 1u);
    ctx->launches += 2;
    CanonIO io{};
    io.packed2 = (u64 *)(d + o_p2); io.bytes = d + o_norm; io.offsets = (u64 *)(d + o_off); io.lens = (u32 *)(d + o_len); io.lane = d + o_lane;
    io.n = n_records; io.mode = mode; io.out = out_bytes ? d + o_out : nullptr; io.out_start = (u32 *)(d + o_start); io.out_strand = d + o_strand;
    io.out_hash = nullptr; io.lists = (u32 *)(d + o_lists); io.lists_bytes = lists_bytes_for(R); io.counts = (u32 *)(d + o_counts);
    io.longest = longest;
    rc = run_canon(ctx, st, ctx->lib_scr, io, 0);
    if (rc) return rc;
    CK_CUDA(ctx, cudaMemcpyAsync(h_counts, d + o_counts, 64, cudaMemcpyDeviceToHost, st));
    if (out_bytes && total) CK_CUDA(ctx, cudaMemcpyAsync(out_bytes, d + o_out, total, cudaMemcpyDeviceToHost, st));
    if (out_start) CK_CUDA(ctx, cudaMemcpyAsync(out_start, d + o_start, R * 4, cudaMemcpyDeviceToHost, st));
    if (out_strand) CK_CUDA(ctx, cudaMemcpyAsync(out_strand, d + o_strand, R, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_counts[CLS_HUGE]) return fail(ctx, CK_ERR_TOO_LONG, "record beyond the staged-length classes");
    return CK_OK;
}

int ck_lmsr_index_batch(ck_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records, uint32_t *out_index)
{
    return lib_batch(ctx, bytes, offsets, n_records, 1u, nullptr, out_index, nullptr);
}
int ck_lmsr_index(ck_ctx *ctx, const uint8_t *s, size_t n, size_t *out_index)
{
    if (!out_index) return ctx ? fail(ctx, CK_ERR_ARG, "null argument") : CK_ERR_ARG;
    if (n > (1ull << 30)) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^30 symbols");
    uint64_t off[2] = {0, (uint64_t)n};
    uint32_t idx = 0;
    int rc = lib_batch(ctx, s, off, 1, 1u, nullptr, &idx, nullptr);
    *out_index = idx;
    return rc;
}
int ck_lmsr(ck_ctx *ctx, const uint8_t *s, size_t n, uint8_t *out)
{
    if (n > (1ull << 30)) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^30 symbols");
    uint64_t off[2] = {0, (uint64_t)n};
    return lib_batch(ctx, s, off, 1, 1u, out, nullptr, nullptr);
}
int ck_canonicalize(ck_ctx *ctx, const uint8_t *s, size_t n, uint8_t *out)
{
    if (n > (1ull << 30)) return fail(ctx, CK_ERR_TOO_LONG, "record longer than 2^30 symbols");
    uint64_t off[2] = {0, (uint64_t)n};
    return lib_batch(ctx, s, off, 1, 0u, out, nullptr, nullptr);
}

// ---- device-resident API ---------------------------------------------------------------------
uint64_t ck_dev_workspace_bytes(uint32_t n_records, uint64_t total_bytes)
{
    u64 b = 256 + lists_bytes_for(n_records);
    if (total_bytes) b += p2_words(total_bytes, n_records) * 8 + total_bytes + 64 + ((5ull * (n_records + 16) + 63) & ~63ull) + p4_bytes_total(total_bytes, n_records);
    return (b + 255) & ~255ull;
}
uint64_t ck_out_arena_bytes(uint64_t total_bytes, uint32_t n_records) { return out_bytes_total(total_bytes, n_records); }

int ck_dev_canon_packed2(ck_ctx *ctx, void *stream, const uint64_t *packed2, const uint64_t *offsets, uint32_t n_records,
                         uint32_t flags, uint32_t class_mask, uint8_t *out_bytes, uint32_t *out_start, uint8_t *out_strand,
                         uint64_t *out_hash64, void *workspace, uint64_t workspace_bytes)
{
    if (!ctx) return CK_ERR_ARG;
    if (workspace_bytes < ck_dev_workspace_bytes(n_records, 0)) return fail(ctx, CK_ERR_ARG, "workspace too small");
    CanonIO io{};
    io.packed2 = U(packed2); io.offsets = U(offsets); io.n = n_records; io.dbl = (flags & CK_F_SINGLE_COPY) ? 0u : 1u;
    io.mode = (flags & CK_F_ALIGNED_OUT) ? 2u : 0u;
    io.out = (flags & CK_F_NO_BYTES) ? nullptr : out_bytes; io.out_start = out_start; io.out_strand = out_strand; io.out_hash = U(out_hash64);
    io.counts = (u32 *)workspace; io.lists = (u32 *)((u8 *)workspace + 256); io.lists_bytes = lists_bytes_for(n_records);
    return run_canon(ctx, (cudaStream_t)stream, ctx->dev_scr, io, class_mask);
}
int ck_dev_canon_bytes(ck_ctx *ctx, void *stream, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records,
                       uint64_t total_bytes, uint32_t flags, uint32_t class_mask, uint8_t *out_bytes, uint32_t *out_len,
                       uint32_t *out_start, uint8_t *out_strand, uint64_t *out_hash64, void *workspace,
                       uint64_t workspace_bytes)
{
    if (!ctx) return CK_ERR_ARG;
    if (!n_records) return CK_OK;
    if (!out_len) return fail(ctx, CK_ERR_ARG, "out_len is required");
    if (workspace_bytes < ck_dev_workspace_bytes(n_records, total_bytes)) return fail(ctx, CK_ERR_ARG, "workspace too small");
    if (!total_bytes) {
        // a batch of empty records only is valid (the host path accepts it too): every record goes to the empty class
        cudaStream_t st0 = (cudaStream_t)stream;
        CK_CUDA(ctx, cudaMemsetAsync(out_len, 0, (size_t)n_records * 4, st0));
        CanonIO io0{};
        io0.offsets = U(offsets); io0.lens = out_len; io0.n = n_records; io0.mode = (flags & CK_F_ALIGNED_OUT) ? 2u : 0u;
        io0.out_start = out_start; io0.out_strand = out_strand; io0.out_hash = U(out_hash64);
        io0.counts = (u32 *)workspace; io0.lists = (u32 *)((u8 *)workspace + 256); io0.lists_bytes = lists_bytes_for(n_records);
        return run_canon(ctx, st0, ctx->dev_scr, io0, class_mask);
    }
    u8 *w = (u8 *)workspace;
    u32 *counts = (u32 *)w; w += 256;
    u32 *lists = (u32 *)w; w += lists_bytes_for(n_records);
    u64 *p2 = (u64 *)w; w += p2_words(total_bytes, n_records) * 8;
    u8 *norm = w; w += (total_bytes + 63) & ~63ull;
    u8 *lane = w; w += ((size_t)n_records + 63) & ~63ull;
    u8 *p4 = w;
    cudaStream_t st = (cudaStream_t)stream;
    PrepareArgs pa{bytes, U(offsets), n_records, (flags & CK_F_NORMALIZE) | (1u << 2), p2, norm, out_len, lane};
    cudaEvent_t pe0 = nullptr, pe1 = nullptr;
    if (ctx->timing) { CK_CUDA(ctx, cudaEventCreate(&pe0)); CK_CUDA(ctx, cudaEventCreate(&pe1)); CK_CUDA(ctx, cudaEventRecord(pe0, st)); }
    k_prepare<<<ctx->num_sms * 32, 256, 0, st>>>(pa);
    k_extend_packed2<<<extend_grid(ctx, n_records), 256, 0, st>>>(p2, U(offsets), out_len, lane, n_records, nullptr, 1u);
    if (ctx->timing) { CK_CUDA(ctx, cudaEventRecord(pe1, st)); ctx->ev_pairs[CLS_COUNT + 6].push_back(pe0); ctx->ev_pairs[CLS_COUNT + 6].push_back(pe1); }
    ctx->launches += 2;
    CanonIO io{};
    io.packed2 = p2; io.bytes = norm; io.offsets = U(offsets); io.lens = out_len; io.lane = lane; io.n = n_records; io.p4 = p4;
    io.mode = (flags & CK_F_ALIGNED_OUT) ? 2u : 0u;
    io.out = (flags & CK_F_NO_BYTES) ? nullptr : out_bytes; io.out_start = out_start; io.out_strand = out_strand;
    io.out_hash = U(out_hash64); io.counts = counts; io.lists = lists; io.lists_bytes = lists_bytes_for(n_records);
    return run_canon(ctx, st, ctx->dev_scr, io, class_mask);
}
int ck_dev_check(ck_ctx *ctx, void *stream, const void *workspace)
{
    if (!ctx) return CK_ERR_ARG;
    u32 h[16];
    CK_CUDA(ctx, cudaMemcpyAsync(h, workspace, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK_CUDA(ctx, cudaStreamSynchronize((cudaStream_t)stream));
    if (h[CLS_HUGE]) return fail(ctx, CK_ERR_TOO_LONG, "batch holds a record beyond the staged-length classes");
    return CK_OK;
}

uint64_t ck_dev_table_bytes(uint64_t capacity_keys) { return table_slots_for(capacity_keys) * sizeof(TableSlot) + 64; }
int ck_dev_table_clear(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes)
{
    TableSlot *slots; u64 nslots; u64 *side; u32 *ov;
    if (!ctx || !table_view(table, table_bytes, slots, nslots, side, ov)) return ctx ? fail(ctx, CK_ERR_ARG, "bad table") : CK_ERR_ARG;
    CK_CUDA(ctx, cudaMemsetAsync(table, 0, 64, (cudaStream_t)stream));
    k_table_clear<<<ctx->num_sms * 4, 256, 0, (cudaStream_t)stream>>>(slots, nslots, side);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int ck_dev_table_insert(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *hash64,
                        const uint64_t *index, uint64_t base_index, uint32_t n, uint64_t *slot_scratch)
{
    TableSlot *slots; u64 nslots; u64 *side; u32 *ov;
    if (!ctx || !table_view(table, table_bytes, slots, nslots, side, ov)) return ctx ? fail(ctx, CK_ERR_ARG, "bad table") : CK_ERR_ARG;
    return table_insert(ctx, (cudaStream_t)stream, slots, nslots, side, ov, U(hash64), U(index), base_index, n, U(slot_scratch));
}
int ck_dev_table_first(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *slot_scratch,
                       uint32_t n, uint64_t *out_first_index)
{
    TableSlot *slots; u64 nslots; u64 *side; u32 *ov;
    if (!ctx || !table_view(table, table_bytes, slots, nslots, side, ov)) return ctx ? fail(ctx, CK_ERR_ARG, "bad table") : CK_ERR_ARG;
    return table_first(ctx, (cudaStream_t)stream, slots, nslots, side, U(slot_scratch), n, U(out_first_index));
}
int ck_dev_table_insert_pairs(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *pairs, uint32_t n,
                              uint64_t *slot_scratch)
{
    TableSlot *slots; u64 nslots; u64 *side; u32 *ov;
    if (!ctx || !pairs || !table_view(table, table_bytes, slots, nslots, side, ov)) return ctx ? fail(ctx, CK_ERR_ARG, "bad table") : CK_ERR_ARG;
    return table_insert(ctx, (cudaStream_t)stream, slots, nslots, side, ov, U(pairs), U(pairs) + 1, 0, n, U(slot_scratch), 2);
}
int ck_dev_owner_partition(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index, uint32_t world,
                           uint64_t *send_pairs, uint32_t *pos, uint32_t *counts_dev, uint32_t *counts_host)
{
    if (!ctx || !hash64 || !send_pairs || !pos || !counts_dev || !counts_host || world < 1 || world > 32)
        return ctx ? fail(ctx, CK_ERR_ARG, "bad partition arguments") : CK_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CK_CUDA(ctx, cudaMemsetAsync(counts_dev, 0, 2 * world * sizeof(u32), st));
    OwnerArgs a{U(hash64), n, world, base_index, counts_dev, U(send_pairs), pos};
    if (n) {
        const u32 grid = std::min<u32>((n + 255) / 256, 8u * (u32)ctx->num_sms);
        k_owner_count<<<grid, 256, 0, st>>>(a);
        k_owner_scatter<<<grid, 256, 0, st>>>(a);
        ctx->launches += 2;
    }
    CK_CUDA(ctx, cudaMemcpyAsync(counts_host, counts_dev, world * sizeof(u32), cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    return CK_OK;
}
int ck_dev_owner_partition_padded(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index,
                                  uint32_t world, uint32_t bucket_capacity, uint64_t *send_pairs, uint32_t *pos, uint32_t *cursors_dev)
{
    if (!ctx || !hash64 || !send_pairs || !pos || !cursors_dev || world < 1 || world > 32 || !bucket_capacity ||
        (u64)world * bucket_capacity > 0xffffffffull)
        return ctx ? fail(ctx, CK_ERR_ARG, "bad partition arguments") : CK_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CK_CUDA(ctx, cudaMemsetAsync(cursors_dev, 0, (world + 1) * sizeof(u32), st));
    OwnerPadArgs a{U(hash64), n, world, base_index, bucket_capacity, cursors_dev, U(send_pairs), pos};
    if (n) {
        k_owner_scatter_padded<<<std::min<u32>((n + 255) / 256, 8u * (u32)ctx->num_sms), 256, 0, st>>>(a);
        ctx->launches++;
    }
    k_owner_pad<<<dim3(16, world), 256, 0, st>>>(a);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int ck_dev_owner_scatter_peers(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index,
                               uint32_t world, uint32_t rank, uint32_t bucket_capacity, const uint64_t *peer_recv_ptrs,
                               uint32_t *pos, uint32_t *cursors_dev)
{
    if (!ctx || !hash64 || !peer_recv_ptrs || !pos || !cursors_dev || world < 1 || world > 32 || rank >= world || !bucket_capacity ||
        (u64)world * bucket_capacity > 0xffffffffull)
        return ctx ? fail(ctx, CK_ERR_ARG, "bad partition arguments") : CK_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CK_CUDA(ctx, cudaMemsetAsync(cursors_dev, 0, (world + 1) * sizeof(u32), st));
    OwnerPeerArgs a{};
    a.hash = U(hash64); a.n = n; a.world = world; a.rank = rank; a.base_index = base_index; a.cap = bucket_capacity;
    a.cursors = cursors_dev; a.pos = pos;
    for (u32 o = 0; o < world; o++) {
        if (!peer_recv_ptrs[o]) return fail(ctx, CK_ERR_ARG, "null peer pointer");
        a.recv.p[o] = reinterpret_cast<u64 *>(peer_recv_ptrs[o]);
    }
    if (n) {
        k_owner_scatter_peers<<<std::min<u32>((n + 255) / 256, 8u * (u32)ctx->num_sms), 256, 0, st>>>(a);
        ctx->launches++;
    }
    k_owner_pad_peers<<<dim3(16, world), 256, 0, st>>>(a);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int ck_dev_table_first_peers(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *slot_scratch,
                             uint32_t world, uint32_t rank, uint32_t bucket_capacity, const uint64_t *peer_ret_ptrs)
{
    TableSlot *slots; u64 nslots; u64 *side; u32 *ov;
    if (!ctx || !slot_scratch || !peer_ret_ptrs || world < 1 || world > 32 || rank >= world || !bucket_capacity ||
        !table_view(table, table_bytes, slots, nslots, side, ov))
        return ctx ? fail(ctx, CK_ERR_ARG, "bad table or peer arguments") : CK_ERR_ARG;
    FirstPeerArgs a{};
    a.slots = slots; a.side_first = side; a.slot_of = U(slot_scratch); a.world = world; a.rank = rank; a.cap = bucket_capacity;
    for (u32 s = 0; s < world; s++) {
        if (!peer_ret_ptrs[s]) return fail(ctx, CK_ERR_ARG, "null peer pointer");
        a.ret.p[s] = reinterpret_cast<u64 *>(peer_ret_ptrs[s]);
    }
    const u32 gx = std::max<u32>(1u, std::min<u32>((bucket_capacity + 255) / 256, (8u * (u32)ctx->num_sms + world - 1) / world));
    k_table_first_peers<<<dim3(gx, world), 256, 0, (cudaStream_t)stream>>>(a);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int ck_dev_gather_first(ck_ctx *ctx, void *stream, const uint64_t *ret, const uint32_t *pos, uint32_t n, uint64_t *out_first_index)
{
    if (!ctx || !ret || !pos || !out_first_index) return ctx ? fail(ctx, CK_ERR_ARG, "null argument") : CK_ERR_ARG;
    if (!n) return CK_OK;
    k_gather_first<<<std::min<u32>((n + 255) / 256, 16u * (u32)ctx->num_sms), 256, 0, (cudaStream_t)stream>>>(U(ret), pos, n, U(out_first_index));
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int ck_dev_normalize(ck_ctx *ctx, void *stream, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records,
                     uint8_t *out_bytes, uint32_t *out_len)
{
    if (!ctx) return CK_ERR_ARG;
    if (!n_records) return CK_OK;
    if (!offsets || !out_bytes || !out_len) return fail(ctx, CK_ERR_ARG, "null argument");
    PrepareArgs pa{bytes, U(offsets), n_records, 1u | 2u | 4u, nullptr, out_bytes, out_len, nullptr};
    k_prepare<<<ctx->num_sms * 32, 256, 0, (cudaStream_t)stream>>>(pa);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int ck_dev_monomerize(ck_ctx *ctx, void *stream, const uint8_t *bytes, const uint64_t *offsets, const uint32_t *lens, uint32_t n_records,
                      uint32_t seed_len, uint64_t overlap_dist, double overlap_min_identity, uint32_t flags, uint32_t *out_end_index)
{
    if (!ctx) return CK_ERR_ARG;
    if (seed_len < 1 || seed_len > 63) return fail(ctx, CK_ERR_ARG, "Seed length must be at least 1 and at most 63");
    if (overlap_min_identity >= 0.0 && overlap_dist)
        return fail(ctx, CK_ERR_ARG, "Both overlap_dist and overlap_min_identity are set. They are mutually exclusive");
    if (!n_records) return CK_OK;
    if (!offsets || !out_end_index) return fail(ctx, CK_ERR_ARG, "null argument");
    MonoArgs a{};
    a.bytes = bytes; a.offsets = U(offsets); a.lens = lens; a.n_records = n_records; a.seed_len = seed_len;
    a.use_identity = overlap_min_identity >= 0.0 ? 1u : 0u; a.overlap_dist = overlap_dist;
    a.identity = overlap_min_identity; a.flags = flags; a.out_end = out_end_index;
    const u32 grid = std::min<u32>((n_records + 7) / 8, 16u * (u32)ctx->num_sms);
    k_monomerize<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
uint64_t ck_launch_count(const ck_ctx *ctx) { return ctx ? ctx->launches : 0; }

int ck_kernel_timing(ck_ctx *ctx, int enable)
{
    if (!ctx) return CK_ERR_ARG;
    ctx->timing = enable != 0;
    return CK_OK;
}
int ck_kernel_times(ck_ctx *ctx, double *out_ms, uint32_t *out_launches, uint32_t n_classes)
{
    if (!ctx || !out_ms || !out_launches) return ctx ? fail(ctx, CK_ERR_ARG, "null argument") : CK_ERR_ARG;
    CK_CUDA(ctx, cudaDeviceSynchronize());
    for (u32 c = 0; c < n_classes; c++) { out_ms[c] = 0; out_launches[c] = 0; }
    for (u32 c = 0; c < (u32)CLS_COUNT + 7; c++) {
        std::vector<cudaEvent_t> &v = ctx->ev_pairs[c];
        for (size_t k = 0; k + 1 < v.size(); k += 2) {
            float ms = 0;
            cudaEventElapsedTime(&ms, v[k], v[k + 1]);
            if (c < n_classes) { out_ms[c] += ms; out_launches[c]++; }
            cudaEventDestroy(v[k]); cudaEventDestroy(v[k + 1]);
        }
        v.clear();
    }
    return CK_OK;
}

// ---- synthetic workloads -------------------------------------------------------------------
int ck_synth_offsets(ck_ctx *ctx, void *stream, uint64_t seed, uint64_t first_index, uint32_t n_records, uint32_t kind,
                     uint32_t lo, uint32_t hi, uint32_t dup_permille, uint64_t *offsets_dev, uint64_t *total_out_host)
{
    if (!ctx || !offsets_dev || lo < 1 || hi < lo) return ctx ? fail(ctx, CK_ERR_ARG, "bad synth arguments") : CK_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    u64 *lens = nullptr; void *tmp = nullptr; size_t tmp_bytes = 0;
    CK_CUDA(ctx, cudaMalloc(&lens, ((size_t)n_records + 1) * 8));
    CK_CUDA(ctx, cudaMemsetAsync(lens, 0, ((size_t)n_records + 1) * 8, st));
    SynthArgs a{seed, n_records, kind, lo, hi, dup_permille, 0, first_index};
    if (n_records) k_synth_lens<<<(n_records + 255) / 256, 256, 0, st>>>(a, lens);
    ctx->launches++;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, lens, U(offsets_dev), (int)n_records + 1, st);
    CK_CUDA(ctx, cudaMalloc(&tmp, tmp_bytes ? tmp_bytes : 8));
    cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, lens, U(offsets_dev), (int)n_records + 1, st);
    ctx->launches++;
    u64 total = 0;
    CK_CUDA(ctx, cudaMemcpyAsync(&total, offsets_dev + n_records, 8, cudaMemcpyDeviceToHost, st));
    CK_CUDA(ctx, cudaStreamSynchronize(st));
    cudaFree(lens); cudaFree(tmp);
    if (total_out_host) *total_out_host = total;
    return CK_OK;
}
uint64_t ck_packed2_words(uint64_t total_bytes, uint32_t n_records, uint32_t flags)
{
    return p2_words(total_bytes, n_records, (flags & CK_F_SINGLE_COPY) ? 0u : 1u);
}
int ck_synth_packed2(ck_ctx *ctx, void *stream, uint64_t seed, uint64_t first_index, uint32_t n_records,
                     const uint64_t *offsets_dev, uint32_t dup_permille, uint32_t adversarial_permille, uint64_t *packed2_dev,
                     uint32_t flags)
{
    const u32 dbl = (flags & CK_F_SINGLE_COPY) ? 0u : 1u;
    if (!ctx || !offsets_dev || !packed2_dev) return ctx ? fail(ctx, CK_ERR_ARG, "bad synth arguments") : CK_ERR_ARG;
    SynthArgs a{seed, n_records, 0, 0, 0, dup_permille, adversarial_permille, first_index};
    if (n_records) {
        k_synth_packed2<<<ctx->num_sms * 8, 256, 0, (cudaStream_t)stream>>>(a, U(offsets_dev), U(packed2_dev), dbl);
        k_extend_packed2<<<extend_grid(ctx, n_records), 256, 0, (cudaStream_t)stream>>>(U(packed2_dev), U(offsets_dev), nullptr, nullptr, n_records, nullptr, dbl);
    }
    ctx->launches += 2;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}
int ck_dev_unpack2(ck_ctx *ctx, void *stream, const uint64_t *packed2, const uint64_t *offsets, uint32_t n_records, uint8_t *ascii_out,
                   uint32_t flags)
{
    if (!ctx) return CK_ERR_ARG;
    if (n_records) k_unpack2<<<ctx->num_sms * 8, 256, 0, (cudaStream_t)stream>>>(U(packed2), U(offsets), n_records, ascii_out,
                                                                                 (flags & CK_F_SINGLE_COPY) ? 0u : 1u);
    ctx->launches++;
    CK_CUDA(ctx, cudaGetLastError());
    return CK_OK;
}

}  // extern "C"
