/*
 * circkit_b200.h -- C ABI of the B200 (sm_100a) canonicalize / uniq hot path of circKit.
 *
 * The reference (Benjamin-Lee/circkit, pure Rust) has no FFI of its own; the seam this library
 * replaces is the pair of closures that `seq_io::parallel::parallel_fasta` drives:
 *
 *   worker closure    src/canonicalize.rs:21-30, src/uniq.rs:33-41
 *                     needletail::sequence::normalize(record.seq(), false) -> circkit::canonicalize(..)
 *   consumer closure  src/uniq.rs:42-78
 *                     xxh3_64(canonical) -> HashMap<u64,String> first-occurrence probe
 *
 * and the library entry points lib/src/canonicalize.rs:5 (lmsr_index), :41 (lmsr), :54 (canonicalize).
 * A `circkit-cuda` crate binds exactly these symbols (see INTEGRATION.md for the Rust side).
 *
 * Conventions
 *   - every function returns CK_OK (0) or a negative CK_ERR_* code; ck_last_error() gives the text;
 *     nothing is printed, no exception crosses the ABI (the reference is silent on success:
 *     tests/canon_uniq.rs:74-77);
 *   - the caller owns every buffer; the library keeps no caller pointer past the matching *_wait;
 *   - a batch is `bytes` (concatenated record.seq() bytes) + `offsets[n_records + 1]`; outputs use the
 *     SAME offsets: record i's canonical bytes are out_bytes[offsets[i] .. offsets[i] + out_len[i]);
 *   - one producer thread per context; `slot` (0 or 1) selects one of two in-flight batches, each with
 *     its own CUDA stream and device staging, so copy-in, kernels and copy-out of consecutive batches
 *     overlap (the replacement for parallel_fasta's queue of 64 record sets).
 */
#ifndef CIRCKIT_B200_H
#define CIRCKIT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CK_OK 0
#define CK_ERR_CUDA (-1)       /* a CUDA runtime call failed (no device, out of memory, ...) */
#define CK_ERR_ARG (-2)        /* bad argument */
#define CK_ERR_STATE (-3)      /* wait without submit, slot busy, ... */
#define CK_ERR_TOO_LONG (-4)   /* a record exceeds the supported length (2^30 symbols; ck_mono_submit: 2^32 - 1024 bytes) */
#define CK_ERR_TABLE_FULL (-5) /* first-occurrence table capacity exhausted */

/* flags of ck_canon_submit / ck_uniq_submit */
#define CK_F_NORMALIZE 1u   /* apply needletail::sequence::normalize(seq, false) first (CLI semantics,
                               src/canonicalize.rs:24-27); without it bytes are used as they are, like
                               circkit::canonicalize (lib/src/canonicalize.rs:54) */
#define CK_F_NO_BYTES 2u    /* do not produce canonical bytes (start/strand/hash only) */
#define CK_F_ALIGNED_OUT 4u /* canonical bytes go to a 32-byte-aligned arena: record i starts at byte
                               32 * ((offsets[i] >> 5) + i) of out_bytes (ck_out_arena_bytes() long) instead of
                               offsets[i].  Every device store is then a full 128-bit store; the host writer reads
                               each record from its aligned start (it copies record by record anyway:
                               src/canonicalize.rs:33-37). */

#define CK_F_SURVIVORS 16u  /* uniq: also compact the survivors on the device, for ck_uniq_wait_survivors */
#define CK_F_SINGLE_COPY 32u /* device-resident API: the packed2 arena is in the single-copy layout (batches of records <= 512 bases) */
/* 64u: CK_F_CANONICAL_BODY of ck_fasta_submit (below) */
#define CK_F_PACKED_IN 8u   /* (set by the *_submit_packed entries) the batch came through ck_pack2_host */

typedef struct ck_ctx ck_ctx;

typedef struct ck_config {
    int32_t device;            /* CUDA device ordinal */
    uint64_t max_batch_bytes;  /* largest `bytes` a batch may carry (staging is sized once) */
    uint32_t max_batch_records;
    uint64_t table_capacity;   /* distinct canonical forms the uniq table holds (0: uniq unused); with ck_uniq_grow, the
                                  initial size */
} ck_config;

/* ---- context ------------------------------------------------------------------------------- */
int ck_init(const ck_config *cfg, ck_ctx **out);
void ck_destroy(ck_ctx *ctx);
const char *ck_last_error(const ck_ctx *ctx);   /* ctx may be NULL: error of a failed ck_init */
void *ck_alloc_pinned(ck_ctx *ctx, size_t bytes);
void ck_free_pinned(ck_ctx *ctx, void *p);

/* ---- batch API: the worker closure (normalise + canonicalise) ------------------------------- */
int ck_canon_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, const uint64_t *offsets,
                    uint32_t n_records, uint32_t flags);
/* any out pointer may be NULL.  out_start/out_strand: canonical[j] = s[(start + j) mod n] when strand
 * is 0, complement(s[(start - j) mod n]) when 1 (s = the normalised record).  out_hash64 = XXH3-64. */
int ck_canon_wait(ck_ctx *ctx, int slot, uint8_t *out_bytes, uint32_t *out_len, uint32_t *out_start,
                  uint8_t *out_strand, uint64_t *out_hash64);

/* ---- batch API: worker + consumer closure (uniq) --------------------------------------------
 * base_index = input-order index of the batch's first record.  out_first_index[i] = index of the first
 * record (over everything submitted to this context so far) whose canonical form has record i's hash;
 * record i is written by `circkit uniq` iff out_first_index[i] == base_index + i, otherwise it is the
 * `duplicate_id` row of out_first_index[i] in --table (src/uniq.rs:47-71). */
int ck_uniq_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, const uint64_t *offsets,
                   uint32_t n_records, uint32_t flags, uint64_t base_index);
int ck_uniq_wait(ck_ctx *ctx, int slot, uint8_t *out_bytes, uint32_t *out_len, uint64_t *out_hash64,
                 uint64_t *out_first_index);
/* The consumer closure writes first occurrences only (src/uniq.rs:47-61).  A batch submitted with CK_F_SURVIVORS is
 * compacted on the device (flags -> scan -> gather, input order kept), and this wait copies back what the survivors need and
 * nothing else: *out_n_survivors; out_index[k] = position in the batch of survivor k (increasing); their canonical bytes,
 * survivor k at out_compact_bytes[out_compact_offsets[k]] (16-byte aligned, out_len[out_index[k]] bytes; out_compact_offsets
 * has n_survivors + 1 entries, the last one = bytes to expect; skipped with CK_F_NO_BYTES).  out_len / out_hash64 /
 * out_first_index are per record of the batch as in ck_uniq_wait (the duplicates' rows of --table need them); any may be NULL.
 * Size out_index for n_records entries, out_compact_offsets for n_records + 1 and out_compact_bytes for offsets[n] + 16 n_records. */
int ck_uniq_wait_survivors(ck_ctx *ctx, int slot, uint32_t *out_n_survivors, uint32_t *out_index, uint64_t *out_compact_offsets,
                           uint8_t *out_compact_bytes, uint32_t *out_len, uint64_t *out_hash64, uint64_t *out_first_index);
int ck_uniq_reset(ck_ctx *ctx);   /* forget every key (new input file); a grown table keeps its size */
/* Let the context's first-occurrence table grow as distinct keys arrive: before a uniq batch is enqueued, the table is
 * enlarged (rehashed on the device) whenever the batch could push it past 2/3 load.  max_keys bounds the distinct keys it
 * may hold (UINT64_MAX: as many as device memory allows); 0 turns growth off (the default).  A batch that would need more
 * than max_keys, or whose growth cannot be allocated, is refused by its submit with CK_ERR_TABLE_FULL before anything is
 * enqueued: the table and its contents are unchanged, the slot stays usable.  Not with a peer group (CK_ERR_STATE, either
 * order); needs a context created with table_capacity >= 1.
 * The submit looks at the device's key count only when a host-side bound (the count collected with the last waited batch
 * plus the records submitted since) could pass 2/3 load; it then synchronises both slots, and grows when the exact count
 * plus the batch needs it, to twice the keys plus two batches.  A growth holds the old and the new table (16 bytes per
 * slot, 1.5 slots per key) for the time of the rehash. */
int ck_uniq_grow(ck_ctx *ctx, uint64_t max_keys);
/* distinct keys in the table (exact; synchronises both slots), the keys it can hold at 2/3 load, and how many times it has
 * grown; any output may be NULL */
int ck_uniq_table_info(ck_ctx *ctx, uint64_t *out_keys, uint64_t *out_capacity_keys, uint64_t *out_grows);

/* ---- packed host input: 2 bits per base over PCIe instead of 8 -----------------------------------
 * The host side the reference keeps (FASTA reader threads, src/uniq.rs:29-41) packs while it parses: ck_pack2_host applies
 * needletail's normalisation when flags has CK_F_NORMALIZE (else bytes as they are), decides every record's symbol lane
 * and writes
 *   packed2_dense  the A/C/G/T records, 16 bases per 32-bit unit (first base in the top bits, units in address order), record i
 *                  at 64-bit word (offsets[i] >> 5) + i; ck_pack2_words(total, n) words in all;
 *   lens[i]        normalised length;   lane[i] = 2 (packed), 4 or 8 (bits per symbol of the byte-level lanes);
 *   lane_bytes     the normalised bytes of the records with lane != 2, concatenated in record order; lane_offsets[n + 1]
 *                  = where each starts (all zero when there are none); *lane_bytes_total = their sum.
 * `threads` host threads share the batch (0 = all hardware threads).  Pure host code: no context, no CUDA call.  The
 * result is what ck_canon_submit_packed / ck_uniq_submit_packed take (they copy lens, lane and the dense words -- a
 * quarter of the ASCII bytes -- and spread the records into the device arena themselves); everything else, including the
 * waits and the output layout (same `offsets`), is as for ck_canon_submit / ck_uniq_submit. */
typedef struct ck_packed_batch {
    const uint64_t *packed2;      /* ck_pack2_words(offsets[n_records], n_records) words, pinned for speed */
    const uint64_t *offsets;      /* n_records + 1 raw symbol offsets, offsets[0] == 0 */
    const uint32_t *lens;         /* n_records */
    const uint8_t *lane;          /* n_records */
    const uint8_t *lane_bytes;    /* may be NULL when lane_bytes_total == 0 */
    const uint64_t *lane_offsets; /* n_records + 1; may be NULL when lane_bytes_total == 0 */
    uint64_t lane_bytes_total;
    uint32_t n_records;
} ck_packed_batch;
uint64_t ck_pack2_words(uint64_t total_bytes, uint32_t n_records);
int ck_pack2_host(const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records, uint32_t flags, uint32_t threads,
                  uint64_t *packed2_dense, uint32_t *lens, uint8_t *lane, uint8_t *lane_bytes, uint64_t lane_bytes_capacity,
                  uint64_t *lane_offsets, uint64_t *lane_bytes_total);
int ck_canon_submit_packed(ck_ctx *ctx, int slot, const ck_packed_batch *batch, uint32_t flags);
int ck_uniq_submit_packed(ck_ctx *ctx, int slot, const ck_packed_batch *batch, uint32_t flags, uint64_t base_index);

/* ---- multi-GPU uniq: one `seen` map (src/uniq.rs:27) over several GPUs of one NVLink / NVSwitch node ----------------
 * One process and one context per GPU.  Keys are owned by hash range (owner = floor(hash64 * world / 2^64)); the
 * (hash64, index) pairs of a batch are stored straight into their owners' buffers by the partition kernel, the owners keep
 * the minimum index per key and store the answers straight back -- device-side barriers, no collective, no host
 * synchronisation (DESIGN.md section 6).  Setup, once:
 *   ck_peer_export   allocates this rank's exchange block for batches of up to max_records records and writes its CUDA IPC
 *                    handle (CK_PEER_HANDLE_BYTES bytes) to handle_out;
 *   (the host exchanges the handles by any means: a file, a pipe, MPI, any process group)
 *   ck_peer_attach   all_handles = the world handles in rank order; maps every peer's block.
 * Afterwards ck_uniq_submit / ck_uniq_submit_packed on this context are COLLECTIVE: the ranks submit in rounds -- in round j
 * every rank submits exactly one batch (possibly with 0 records) on the same slot -- and every index of round j must be larger
 * than every index of round j - 1 (e.g. batch k of the input goes to rank k mod world in round k / world, with base_index =
 * the batch's position in the input).  out_first_index then is exact at ck_uniq_wait, as on one GPU: the first occurrence over
 * everything submitted to ANY rank so far.  The table of each context (table_capacity) holds the keys this rank owns.
 * ck_dev_peer_first_index is the same exchange for device-resident hashes (one collective call per rank, any stream). */
#define CK_PEER_HANDLE_BYTES 64
int ck_peer_export(ck_ctx *ctx, uint32_t world, uint32_t rank, uint32_t max_records, void *handle_out);
int ck_peer_attach(ck_ctx *ctx, const void *all_handles);
int ck_dev_peer_first_index(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index, void *table,
                            uint64_t table_bytes, uint64_t *out_first_index);

/* ---- library drop-ins (single record, library semantics: no normalisation) -------------------
 * lib/src/canonicalize.rs:5,41,54.  These run the same device kernels on a batch of one. */
int ck_lmsr_index(ck_ctx *ctx, const uint8_t *s, size_t n, size_t *out_index);
int ck_lmsr(ck_ctx *ctx, const uint8_t *s, size_t n, uint8_t *out);
int ck_canonicalize(ck_ctx *ctx, const uint8_t *s, size_t n, uint8_t *out);
/* batched forms of the same three (library semantics), for callers that hold many records */
int ck_lmsr_index_batch(ck_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records,
                        uint32_t *out_index);

/* ---- device-resident API (buffers already in HBM; used by bench.py and the multi-GPU driver) --
 * All pointers are device pointers, `stream` is a cudaStream_t (0 = default stream).  Nothing is copied
 * and nothing synchronises; call ck_dev_check() once a stream's work matters.
 * packed2: 2-bit arena, A,C,G,T = 0..3, 16 bases per 32-bit unit with the first base in the top bits, units in
 * address order.  Two layouts, a property of the batch (ck_packed2_words() gives the arena size in 64-bit words):
 *   doubled (default)      record i starts at byte 32 * ((offsets[i] >> 6) + 3 i) and is stored twice over: units
 *                          0 .. (2 n + 143) >> 4 (at least (n >> 4) + 5) hold the bases S[b mod n], so every rotation of the
 *                          circular record is a linear window (256-bit loads, no wrap logic);
 *   CK_F_SINGLE_COPY       record i starts at byte 16 * ((offsets[i] >> 6) + 2 i) and is followed by its circular extension
 *                          only (units 0 .. (n >> 4) + 4): less than half the footprint; meant for batches whose records are
 *                          all <= 512 bases (the host-buffer entries choose it by themselves for such batches).
 * class_mask: 0 = any record; else a promise about the batch (bit c set = length/alphabet class c may occur, see
 * CK_CLASS_*), which skips the launches of absent classes; records outside the promise are reported by ck_dev_check(),
 * never silently dropped. */
#define CK_CLASS_2BIT_LE_512 (1u << 0)
#define CK_CLASS_2BIT_LE_2048 (1u << 1)
#define CK_CLASS_2BIT_LE_65536 (1u << 2)
#define CK_CLASS_2BIT_LE_425984 (1u << 3)
#define CK_CLASS_2BIT_LE_4096 (1u << 10)
#define CK_CLASS_2BIT_LE_8192 (1u << 11)
uint64_t ck_dev_workspace_bytes(uint32_t n_records, uint64_t total_bytes /* 0 for the packed2 entry */);
/* bytes of the CK_F_ALIGNED_OUT arena of a batch (host and device entries) */
uint64_t ck_out_arena_bytes(uint64_t total_bytes, uint32_t n_records);
uint64_t ck_packed2_words(uint64_t total_bytes, uint32_t n_records, uint32_t flags /* CK_F_SINGLE_COPY or 0 */);
/* flags: CK_F_NO_BYTES, CK_F_ALIGNED_OUT, CK_F_SINGLE_COPY */
int ck_dev_canon_packed2(ck_ctx *ctx, void *stream, const uint64_t *packed2, const uint64_t *offsets,
                         uint32_t n_records, uint32_t flags, uint32_t class_mask, uint8_t *out_bytes, uint32_t *out_start,
                         uint8_t *out_strand, uint64_t *out_hash64, void *workspace, uint64_t workspace_bytes);
/* raw/normalised bytes -> lane formats (the k_prepare step), then canonicalise; out_len is required.  Records that are not pure
 * ACGT take the byte-level lanes; of those, records over {-, A, C, G, N, T} -- all that needletail's normalisation
 * (src/canonicalize.rs:24-27) leaves of IUPAC input -- with 129..2048 symbols and CK_F_ALIGNED_OUT are packed at 4 bits per
 * symbol, both strands, into a part of the workspace and canonicalised by the lane-per-record kernel of csrc/ck_lane4.cuh;
 * the host-buffer entries (ck_*_submit*) do the same inside the context. */
int ck_dev_canon_bytes(ck_ctx *ctx, void *stream, const uint8_t *bytes, const uint64_t *offsets,
                       uint32_t n_records, uint64_t total_bytes, uint32_t flags, uint32_t class_mask,
                       uint8_t *out_bytes, uint32_t *out_len, uint32_t *out_start, uint8_t *out_strand,
                       uint64_t *out_hash64, void *workspace, uint64_t workspace_bytes);
/* synchronises `stream`; CK_ERR_TOO_LONG if the last call on `workspace` left records unprocessed (the device-resident entries
 * stop at the staged-length classes: 2-bit 425 984, 4-bit 212 992, bytes 106 496 symbols; the host-buffer entries and the library
 * drop-ins process longer records from global memory, up to 2^30 symbols) */
int ck_dev_check(ck_ctx *ctx, void *stream, const void *workspace);
/* first-occurrence table over device arrays; index == NULL means base_index + i */
uint64_t ck_dev_table_bytes(uint64_t capacity_keys);
int ck_dev_table_clear(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes);
int ck_dev_table_insert(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *hash64,
                        const uint64_t *index, uint64_t base_index, uint32_t n, uint64_t *slot_scratch);
int ck_dev_table_first(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *slot_scratch,
                       uint32_t n, uint64_t *out_first_index);
/* Multi-GPU uniq (hash-range owners, replaces the single `seen` map of src/uniq.rs:27 across ranks): bucket the local
 * (hash64, base_index + i) pairs by owner = floor(hash64 * world / 2^64) into per-owner runs of send_pairs (2 u64 per record:
 * the send buffer of one personalised all-to-all); pos[i] = where record i went; counts_host[world] = records per owner
 * (the call synchronises the stream to return them).  counts_dev: 2 * world u32 of device scratch.
 * ck_dev_table_insert_pairs: ck_dev_table_insert over such (hash64, index) pairs as they arrive at the owner. */
int ck_dev_owner_partition(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index, uint32_t world,
                           uint64_t *send_pairs, uint32_t *pos, uint32_t *counts_dev, uint32_t *counts_host);
int ck_dev_table_insert_pairs(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *pairs, uint32_t n,
                              uint64_t *slot_scratch);
/* The same partition into FIXED-capacity buckets, for an equal-split all-to-all with no counts to exchange and no host
 * synchronisation: bucket o = send_pairs[o * bucket_capacity, (o + 1) * bucket_capacity) (2 u64 per entry); unused entries
 * carry index ~0, which ck_dev_table_insert_pairs skips (their first index reads back as ~0); pos[i] = entry of record i
 * (0xffffffff if its bucket was full).  cursors_dev: world + 1 u32 of device scratch; after the call cursors_dev[o] =
 * records sent to owner o and cursors_dev[world] != 0 iff a bucket overflowed -- the caller then repeats the batch with
 * ck_dev_owner_partition.  Nothing is copied to the host and the stream is not synchronised. */
int ck_dev_owner_partition_padded(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index,
                                  uint32_t world, uint32_t bucket_capacity, uint64_t *send_pairs, uint32_t *pos,
                                  uint32_t *cursors_dev);
/* The exchange fused into the kernels around it, over peer-mapped device memory (one process per GPU of one NVLink /
 * NVSwitch node; the caller maps every rank's buffers into every process, e.g. with CUDA IPC handles):
 *   peer_recv_ptrs[o]  device address, in THIS process, of owner o's receive buffer: world regions of bucket_capacity
 *                      (hash64, index) pairs; this rank writes region `rank` of every one of them, padding included;
 *   peer_ret_ptrs[s]   device address of rank s's return buffer: world regions of bucket_capacity first indices;
 *                      the owner writes region `rank` (= itself) with the answers for the pairs rank s sent, in order.
 * Sequence per batch on every rank: ck_dev_owner_scatter_peers; barrier over all ranks; ck_dev_table_insert_pairs over the
 * local receive buffer (world * bucket_capacity entries); ck_dev_table_first_peers; barrier; first_index[i] =
 * own return buffer[pos[i]].  cursors_dev as in ck_dev_owner_partition_padded (overflow flag at [world]).  Neither call
 * synchronises the stream.  Both pointer arrays are host arrays of `world` entries. */
int ck_dev_owner_scatter_peers(ck_ctx *ctx, void *stream, const uint64_t *hash64, uint32_t n, uint64_t base_index,
                               uint32_t world, uint32_t rank, uint32_t bucket_capacity, const uint64_t *peer_recv_ptrs,
                               uint32_t *pos, uint32_t *cursors_dev);
int ck_dev_table_first_peers(ck_ctx *ctx, void *stream, void *table, uint64_t table_bytes, const uint64_t *slot_scratch,
                             uint32_t world, uint32_t rank, uint32_t bucket_capacity, const uint64_t *peer_ret_ptrs);
/* out_first_index[i] = ret[pos[i]] (~0 where pos[i] == 0xffffffff): answers of either fixed-capacity exchange back in input order */
int ck_dev_gather_first(ck_ctx *ctx, void *stream, const uint64_t *ret, const uint32_t *pos, uint32_t n, uint64_t *out_first_index);
/* ---- monomerize (the step that feeds canonicalize / uniq in the author's pipeline, README.md:83) ----
 * For every record of a device-resident batch of raw bytes (record i = bytes[offsets[i], offsets[i+1]) or, with `lens`,
 * its first lens[i] bytes; library semantics: bytes as they are) the end index of its last monomer:
 *   Monomerizer::last_monomer_end_index            lib/src/monomerize.rs:100-125   (flags 0)
 *   Monomerizer::last_monomer_end_index_sensitive  lib/src/monomerize.rs:127-141   (flags CK_MONO_SENSITIVE)
 *   Monomerizer::first_monomer_end_index           lib/src/monomerize.rs:50-99     (flags CK_MONO_FIRST_ONLY)
 * out_end_index[i] = CK_MONO_NONE for None; monomerize(seq) = seq[.. end] (the whole record for None, :144-158).
 * overlap_min_identity < 0 means "not set" (then overlap_dist applies, default 0); the builder's rules hold
 * (lib/src/monomerize.rs:20-40): 1 <= seed_len <= 63, identity and a non-zero distance exclude each other -> CK_ERR_ARG. */
#define CK_MONO_SENSITIVE 1u
#define CK_MONO_FIRST_ONLY 2u
#define CK_MONO_NONE 0xffffffffu
int ck_dev_monomerize(ck_ctx *ctx, void *stream, const uint8_t *bytes, const uint64_t *offsets, const uint32_t *lens,
                      uint32_t n_records, uint32_t seed_len, uint64_t overlap_dist, double overlap_min_identity, uint32_t flags,
                      uint32_t *out_end_index);
/* needletail::sequence::normalize(seq, false) of every record of a resident batch (src/monomerize.rs:86-89,
 * src/canonicalize.rs:24): out_bytes holds record i's normalised bytes at offsets[i], out_len[i] of them (white space is
 * dropped, so out_len[i] <= offsets[i+1] - offsets[i]); feed both to ck_dev_monomerize (`lens`) for the CLI's semantics. */
int ck_dev_normalize(ck_ctx *ctx, void *stream, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records,
                     uint8_t *out_bytes, uint32_t *out_len);
/* Batch API of `circkit monomerize` (host buffers, the two slots of the context, like ck_canon_submit / ck_uniq_submit; a
 * monomerize batch may be in flight on one slot while a canonicalize / uniq batch is on the other).  ck_mono_submit copies
 * the raw record bytes in and, in order on the slot's stream: normalises them (flags CK_F_NORMALIZE: the CLI's semantics,
 * as ck_dev_normalize), runs the monomer search, then the worker and consumer closures' rules (src/monomerize.rs:83-143):
 *   idx      = None when the (normalised) record is shorter than seed_len or min_length, else the monomer search's answer;
 *   ok       = idx is not None and none of idx < min_length, idx > max_length, full_len - idx < min_overlap,
 *              (double)(full_len - idx) / idx < min_overlap_percent holds;
 *   written  = ok or CK_MONO_KEEP_ALL;   monomer_len = ok ? min(idx, full_len) : full_len;
 * full_len = length of seq_io's full_seq (the record without '\n' and without a '\r' that ends a line or the record) with
 * CK_F_NORMALIZE, else the raw length.  The written records' bytes (full_seq[.. monomer_len], or the raw bytes without
 * CK_F_NORMALIZE) are compacted on the device; CK_F_NO_BYTES skips them.  idx counts normalised symbols and is applied to
 * full_seq, which keeps the ' ' / '\t' that normalisation drops: the reference does the same.
 * Every "unset" value below filters nothing, like the reference's None.  seed_len outside 1..63, or identity and a
 * non-zero distance together -> CK_ERR_ARG (the builder's rules, lib/src/monomerize.rs:20-40).  A record may be up to
 * 2^32 - 1024 bytes long (lengths are 32-bit; the 2^30 limit of canonicalize / uniq does not apply); a longer one ->
 * CK_ERR_TOO_LONG. */
#define CK_MONO_KEEP_ALL 4u
typedef struct ck_mono_options {
    uint32_t seed_len;             /* 1..63 */
    uint32_t flags;                /* CK_MONO_SENSITIVE | CK_MONO_FIRST_ONLY | CK_MONO_KEEP_ALL */
    uint64_t overlap_dist;         /* --max-mismatch; 0 = unset */
    double overlap_min_identity;   /* --min-identity; < 0 = unset */
    uint64_t min_length;           /* --min-length (default 0) */
    uint64_t max_length;           /* --max-length; UINT64_MAX = unset */
    uint64_t min_overlap;          /* --min-overlap; 0 = unset */
    double min_overlap_percent;    /* --min-overlap-percent; NaN = unset */
} ck_mono_options;
int ck_mono_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, const uint64_t *offsets, uint32_t n_records,
                   uint32_t flags /* CK_F_NORMALIZE, CK_F_NO_BYTES */, const ck_mono_options *opt);
/* Per record of the batch: out_monomer_len, out_full_len and out_end_index (idx above, before the filters; CK_MONO_NONE =
 * None).  The written records only: *out_n_written; out_index[k] = position in the batch of written record k (increasing);
 * its bytes at out_compact_bytes[out_compact_offsets[k]] (16-byte aligned, out_monomer_len[out_index[k]] bytes;
 * out_compact_offsets has n_written + 1 entries, the last one = bytes to expect).  Any out pointer may be NULL.
 * Size out_index for n_records entries, out_compact_offsets for n_records + 1 and out_compact_bytes for offsets[n] + 16 n_records. */
int ck_mono_wait(ck_ctx *ctx, int slot, uint32_t *out_n_written, uint32_t *out_index, uint64_t *out_compact_offsets,
                 uint8_t *out_compact_bytes, uint32_t *out_monomer_len, uint32_t *out_full_len, uint32_t *out_end_index);

/* ---- FASTA text batches: `circkit canonicalize` / `uniq` / `monomerize` from decompressed text to written bytes ----------
 * ck_fasta_submit takes FASTA text as it comes out of the decompressor, on one of the two slots, and does on the slot's
 * stream everything the CLI's worker and consumer closures do, with seq_io 0.3.2's record split before and the CLI's output
 * framing after:
 *   text         whole records; text[0] must be '>' (leading blank lines are the caller's to strip) -> else CK_ERR_ARG;
 *                a record starts at a '>' at position 0 or after a '\n'; head = the header line without '>' and without
 *                one trailing '\r'; seq = from after the header's '\n' to the record's last '\n' (or the end of the
 *                text), one trailing '\r' trimmed; the last record ends at text_bytes.
 *   command      CK_CMD_CANONICALIZE: every record, '>' head '\n' canonical '\n' (src/canonicalize.rs:33-37);
 *                CK_CMD_UNIQ: the first occurrences only, '>' head '\n' record.seq() '\n' (internal line breaks kept), or
 *                the canonical form with CK_F_CANONICAL_BODY (src/uniq.rs:50-61).  The table is the context's, across
 *                batches, as for ck_uniq_submit; base_index = input-order index of the batch's first record;
 *                CK_CMD_MONOMERIZE: the written records, '>' head '\n' full_seq[.. monomer_len] '\n', with the rules and
 *                options of ck_mono_submit (`mono`).
 * Normalisation is always the CLI's (CK_F_NORMALIZE).  *out_n_records = records in the text (the next batch's base_index
 * follows from it).  Refused before anything is left running on the slot: text_bytes > max_batch_bytes or more records than
 * max_batch_records -> CK_ERR_ARG (the slot stays usable); a seq over 2^30 symbols (canonicalize / uniq) or over
 * 2^32 - 1024 bytes (monomerize) -> CK_ERR_TOO_LONG; uniq on a context with table_capacity 0 or with a peer group attached
 * -> CK_ERR_STATE.  The submit waits for its record count (a small copy after the split); the other slot keeps running.
 * The first text batch of a slot allocates its text and framing buffers (about 2 max_batch_bytes + 2 max_batch_records).
 *
 * ck_fasta_wait: out_fasta (ck_fasta_out_bytes(text_bytes, n_records) bytes) receives exactly the bytes the CLI writes for
 * this batch, *out_fasta_bytes of them; *out_n_written records, out_index[k] = position in the batch of written record k
 * (increasing).  Per record of the batch: out_head[2 i], out_head[2 i + 1] = its head range [lo, hi) in the text;
 * out_first_index (uniq, as ck_uniq_wait); out_full_len / out_monomer_len (monomerize, as ck_mono_wait).  Any out pointer
 * may be NULL. */
#define CK_CMD_CANONICALIZE 1
#define CK_CMD_UNIQ 2
#define CK_CMD_MONOMERIZE 3
#define CK_F_CANONICAL_BODY 64u   /* uniq -c: write the canonical form, not record.seq() */
uint64_t ck_fasta_out_bytes(uint64_t text_bytes, uint32_t n_records);   /* text_bytes + 2 n_records + 64 */
int ck_fasta_submit(ck_ctx *ctx, int slot, const uint8_t *text, uint64_t text_bytes, uint32_t command, uint32_t flags,
                    uint64_t base_index, const ck_mono_options *mono, uint32_t *out_n_records);
int ck_fasta_wait(ck_ctx *ctx, int slot, uint8_t *out_fasta, uint64_t *out_fasta_bytes, uint32_t *out_n_written,
                  uint32_t *out_index, uint64_t *out_head, uint64_t *out_first_index, uint32_t *out_full_len,
                  uint32_t *out_monomer_len);
/* ---- DEFLATE on the device: the `.gz` output of `circkit ... -o out.gz` (src/utils.rs:29-72, flate2 at level 6) ---------
 * ck_deflate_submit compresses n bytes (1 .. CK_DEFLATE_MAX_BYTES) on one of the two slots into raw DEFLATE (RFC 1951):
 * blocks none of which has BFINAL set, ending byte-aligned with an empty stored block (00 00 ff ff, zlib's Z_SYNC_FLUSH).
 * `dict` (dict_bytes <= CK_DEFLATE_DICT_BYTES; may be NULL when 0) is what came before `bytes` in the stream: matches may reach
 * into it, and never further than 32 768 bytes back or before its start, so consecutive calls, each given the last 32 KiB of
 * the input before it, concatenate into one deflate stream (one gzip member: a header, the fragments, 03 00, CRC-32 and
 * ISIZE).  zlib.decompressobj(-15, zdict=dict).decompress(out) == bytes.  The output is a function of (bytes, dict) only.
 * ck_deflate_wait copies *out_bytes (<= ck_deflate_bound(n)) bytes to `out` and gives the CRC-32 of `bytes` continued from
 * crc_in (== zlib.crc32(bytes, crc_in)); out_bytes and crc_out may be NULL.
 * A deflate call occupies its slot like any other batch (CK_ERR_STATE when busy, or for a wait without a submit); it runs on a
 * stream of its own, so it works on a context created with max_batch_bytes = max_batch_records = 0 (no batch staging).  n == 0,
 * n > CK_DEFLATE_MAX_BYTES, dict_bytes > CK_DEFLATE_DICT_BYTES or a NULL pointer -> CK_ERR_ARG, nothing is enqueued and the
 * slot stays usable.  The slot's first deflate call allocates its buffers (about 30 bytes of HBM per input byte of the largest
 * call so far, rounded up to a power of two), so contexts that never deflate use no more device memory.  `bytes` and `dict`
 * may be reused once the submit returns when they are pageable; pinned buffers must stay untouched until the wait. */
#define CK_DEFLATE_MAX_BYTES (64ull << 20)
#define CK_DEFLATE_DICT_BYTES 32768u
uint64_t ck_deflate_bound(uint64_t n);   /* out bytes to provide for n input bytes */
int ck_deflate_submit(ck_ctx *ctx, int slot, const uint8_t *bytes, uint64_t n, const uint8_t *dict, uint32_t dict_bytes,
                      uint32_t crc_in);
int ck_deflate_wait(ck_ctx *ctx, int slot, uint8_t *out, uint64_t *out_bytes, uint32_t *crc_out);

/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t ck_launch_count(const ck_ctx *ctx);
/* per-class kernel timing for the roofline: when enabled, every length/alphabet-class launch is bracketed
 * by CUDA events on its own stream; ck_kernel_times() synchronises, sums the elapsed ms and launch counts
 * per class (index = class bit position of CK_CLASS_*) and clears the record. */
int ck_kernel_timing(ck_ctx *ctx, int enable);
int ck_kernel_times(ck_ctx *ctx, double *out_ms, uint32_t *out_launches, uint32_t n_classes);

/* ---- synthetic workloads of BASELINE.json (device generators, bench + tests) ------------------
 * Record g = first_index + i is a pure function of (seed, g): any shard can be generated on any rank.
 * lengths: kind 0 = uniform integer [lo, hi], 1 = log-uniform [lo, hi]; dup_permille/1000 of the records
 * are duplicates (random rotation, reverse complement w.p. 1/2) of an earlier original and share its
 * length.  Writes n_records + 1 offsets; synchronises `stream` to return the total. */
int ck_synth_offsets(ck_ctx *ctx, void *stream, uint64_t seed, uint64_t first_index, uint32_t n_records,
                     uint32_t kind, uint32_t lo, uint32_t hi, uint32_t dup_permille, uint64_t *offsets_dev,
                     uint64_t *total_out_host);
/* content in the packed2 layout; adversarial_permille/1000 of the originals are tandem repeats
 * (period 1, 2, 3, 7, 171, n/2) or carry >= 1 kb poly-A runs (config 4) */
int ck_synth_packed2(ck_ctx *ctx, void *stream, uint64_t seed, uint64_t first_index, uint32_t n_records,
                     const uint64_t *offsets_dev, uint32_t dup_permille, uint32_t adversarial_permille,
                     uint64_t *packed2_dev, uint32_t flags /* CK_F_SINGLE_COPY or 0 */);
/* 2-bit arena -> ASCII arena (record i at offsets[i]) */
int ck_dev_unpack2(ck_ctx *ctx, void *stream, const uint64_t *packed2, const uint64_t *offsets, uint32_t n_records,
                   uint8_t *ascii_out, uint32_t flags /* CK_F_SINGLE_COPY or 0 */);

#ifdef __cplusplus
}
#endif
#endif /* CIRCKIT_B200_H */
