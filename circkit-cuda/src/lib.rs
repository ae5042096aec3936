//! circkit-cuda: the device side of `circkit canonicalize` / `circkit uniq` / `circkit monomerize` on B200 (sm_100a).
//!
//! * [`ffi`] mirrors `include/circkit_b200.h` one to one.
//! * [`Context`] owns a `ck_ctx` (one device, two in-flight batch slots, the first-occurrence table).
//! * [`Pump`] is the replacement for `seq_io::parallel::parallel_fasta` as circKit uses it
//!   (`src/canonicalize.rs:17-45`, `src/uniq.rs:29-79`): the reader thread appends `record.seq()` to a pinned batch, full
//!   batches are packed to 2 bits per base on the host (`ck_pack2_host`), shipped and processed on alternating slots, and the
//!   caller's consumer closure sees every record in input order with its canonical bytes / survival decision.  For
//!   `circkit monomerize` (`src/monomerize.rs:16-160`) the raw bytes go to the device as they are (`ck_mono_submit`), and the
//!   closure gets the written records' monomers and the lengths of the `--table` row.
//! * [`canonicalize`], [`lmsr`], [`lmsr_index`] are the drop-ins for `circkit::canonicalize` (`lib/src/canonicalize.rs:54`),
//!   `circkit::canonicalize::lmsr` (`:41`) and `lmsr_index` (`:5`): same signatures, same results, a process-wide context.
//!
//! Errors: every negative return code becomes an `anyhow::Error` carrying `ck_last_error` (the CLI already propagates
//! `anyhow`, `src/main.rs:22-38`); the library drop-ins panic instead, like the reference's `unwrap()`s.

use anyhow::{anyhow, Result};
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};
use std::ptr::{null, null_mut};
use std::sync::{Mutex, OnceLock};

pub mod ffi {
    use super::*;
    #[repr(C)]
    pub struct CkCtx {
        _p: [u8; 0],
    }
    #[repr(C)]
    #[derive(Clone, Copy)]
    pub struct CkConfig {
        pub device: i32,
        pub max_batch_bytes: u64,
        pub max_batch_records: u32,
        pub table_capacity: u64,
    }
    #[repr(C)]
    pub struct CkPackedBatch {
        pub packed2: *const u64,
        pub offsets: *const u64,
        pub lens: *const u32,
        pub lane: *const u8,
        pub lane_bytes: *const u8,
        pub lane_offsets: *const u64,
        pub lane_bytes_total: u64,
        pub n_records: u32,
    }
    /// `ck_mono_options`: the consumer-closure options of `circkit monomerize` (`src/commands.rs:19-90`); every "unset"
    /// value filters nothing, like the reference's `None`.
    #[repr(C)]
    #[derive(Clone, Copy, PartialEq, Debug)]
    pub struct MonoOptions {
        pub seed_len: u32,              // 1..63
        pub flags: u32,                 // CK_MONO_SENSITIVE | CK_MONO_FIRST_ONLY | CK_MONO_KEEP_ALL
        pub overlap_dist: u64,          // --max-mismatch; 0 = unset
        pub overlap_min_identity: f64,  // --min-identity; < 0 = unset
        pub min_length: u64,            // --min-length (default 0)
        pub max_length: u64,            // --max-length; u64::MAX = unset
        pub min_overlap: u64,           // --min-overlap; 0 = unset
        pub min_overlap_percent: f64,   // --min-overlap-percent; NaN = unset
    }
    pub const CK_OK: c_int = 0;
    pub const CK_F_NORMALIZE: u32 = 1;
    pub const CK_F_NO_BYTES: u32 = 2;
    pub const CK_F_ALIGNED_OUT: u32 = 4;
    pub const CK_F_PACKED_IN: u32 = 8;
    pub const CK_F_SURVIVORS: u32 = 16;
    pub const CK_PEER_HANDLE_BYTES: usize = 64;
    pub const CK_MONO_SENSITIVE: u32 = 1;
    pub const CK_MONO_FIRST_ONLY: u32 = 2;
    pub const CK_MONO_KEEP_ALL: u32 = 4;
    pub const CK_MONO_NONE: u32 = 0xffff_ffff;
    // FASTA text batches (ck_fasta_submit / ck_fasta_wait): the commands, and uniq -c's body
    pub const CK_CMD_CANONICALIZE: u32 = 1;
    pub const CK_CMD_UNIQ: u32 = 2;
    pub const CK_CMD_MONOMERIZE: u32 = 3;
    pub const CK_F_CANONICAL_BODY: u32 = 64;
    /// ck_deflate_submit: largest input of one call, largest dictionary
    pub const CK_DEFLATE_MAX_BYTES: u64 = 64 << 20;
    pub const CK_DEFLATE_DICT_BYTES: u32 = 32768;
    extern "C" {
        pub fn ck_init(cfg: *const CkConfig, out: *mut *mut CkCtx) -> c_int;
        pub fn ck_destroy(ctx: *mut CkCtx);
        pub fn ck_last_error(ctx: *const CkCtx) -> *const c_char;
        pub fn ck_alloc_pinned(ctx: *mut CkCtx, bytes: usize) -> *mut c_void;
        pub fn ck_free_pinned(ctx: *mut CkCtx, p: *mut c_void);
        pub fn ck_out_arena_bytes(total_bytes: u64, n_records: u32) -> u64;
        pub fn ck_canon_submit(ctx: *mut CkCtx, slot: c_int, bytes: *const u8, offsets: *const u64, n: u32, flags: u32) -> c_int;
        pub fn ck_canon_wait(ctx: *mut CkCtx, slot: c_int, out_bytes: *mut u8, out_len: *mut u32, out_start: *mut u32,
                             out_strand: *mut u8, out_hash64: *mut u64) -> c_int;
        pub fn ck_uniq_submit(ctx: *mut CkCtx, slot: c_int, bytes: *const u8, offsets: *const u64, n: u32, flags: u32,
                              base_index: u64) -> c_int;
        pub fn ck_uniq_wait(ctx: *mut CkCtx, slot: c_int, out_bytes: *mut u8, out_len: *mut u32, out_hash64: *mut u64,
                            out_first_index: *mut u64) -> c_int;
        pub fn ck_uniq_wait_survivors(ctx: *mut CkCtx, slot: c_int, out_n_survivors: *mut u32, out_index: *mut u32,
                                      out_compact_offsets: *mut u64, out_compact_bytes: *mut u8, out_len: *mut u32,
                                      out_hash64: *mut u64, out_first_index: *mut u64) -> c_int;
        pub fn ck_uniq_reset(ctx: *mut CkCtx) -> c_int;
        pub fn ck_uniq_grow(ctx: *mut CkCtx, max_keys: u64) -> c_int;
        pub fn ck_uniq_table_info(ctx: *mut CkCtx, out_keys: *mut u64, out_capacity_keys: *mut u64, out_grows: *mut u64) -> c_int;
        pub fn ck_pack2_words(total_bytes: u64, n_records: u32) -> u64;
        pub fn ck_pack2_host(bytes: *const u8, offsets: *const u64, n_records: u32, flags: u32, threads: u32,
                             packed2_dense: *mut u64, lens: *mut u32, lane: *mut u8, lane_bytes: *mut u8,
                             lane_bytes_capacity: u64, lane_offsets: *mut u64, lane_bytes_total: *mut u64) -> c_int;
        pub fn ck_canon_submit_packed(ctx: *mut CkCtx, slot: c_int, batch: *const CkPackedBatch, flags: u32) -> c_int;
        pub fn ck_uniq_submit_packed(ctx: *mut CkCtx, slot: c_int, batch: *const CkPackedBatch, flags: u32, base_index: u64) -> c_int;
        pub fn ck_mono_submit(ctx: *mut CkCtx, slot: c_int, bytes: *const u8, offsets: *const u64, n: u32, flags: u32,
                              opt: *const MonoOptions) -> c_int;
        pub fn ck_mono_wait(ctx: *mut CkCtx, slot: c_int, out_n_written: *mut u32, out_index: *mut u32, out_compact_offsets: *mut u64,
                            out_compact_bytes: *mut u8, out_monomer_len: *mut u32, out_full_len: *mut u32,
                            out_end_index: *mut u32) -> c_int;
        // FASTA text in, the CLI's output bytes out; `mono` may be null except for CK_CMD_MONOMERIZE, any out pointer may be
        // null.  Declared from the header; this crate has no Pump over them (callers drive the two slots themselves).
        pub fn ck_fasta_out_bytes(text_bytes: u64, n_records: u32) -> u64;
        pub fn ck_fasta_submit(ctx: *mut CkCtx, slot: c_int, text: *const u8, text_bytes: u64, command: u32, flags: u32,
                               base_index: u64, mono: *const MonoOptions, out_n_records: *mut u32) -> c_int;
        pub fn ck_fasta_wait(ctx: *mut CkCtx, slot: c_int, out_fasta: *mut u8, out_fasta_bytes: *mut u64, out_n_written: *mut u32,
                             out_index: *mut u32, out_head: *mut u64, out_first_index: *mut u64, out_full_len: *mut u32,
                             out_monomer_len: *mut u32) -> c_int;
        pub fn ck_deflate_bound(n: u64) -> u64;
        pub fn ck_deflate_submit(ctx: *mut CkCtx, slot: c_int, bytes: *const u8, n: u64, dict: *const u8, dict_bytes: u32,
                                 crc_in: u32) -> c_int;
        pub fn ck_deflate_wait(ctx: *mut CkCtx, slot: c_int, out: *mut u8, out_bytes: *mut u64, crc_out: *mut u32) -> c_int;
        pub fn ck_peer_export(ctx: *mut CkCtx, world: u32, rank: u32, max_records: u32, handle_out: *mut c_void) -> c_int;
        pub fn ck_peer_attach(ctx: *mut CkCtx, all_handles: *const c_void) -> c_int;
        pub fn ck_lmsr_index(ctx: *mut CkCtx, s: *const u8, n: usize, out_index: *mut usize) -> c_int;
        pub fn ck_lmsr(ctx: *mut CkCtx, s: *const u8, n: usize, out: *mut u8) -> c_int;
        pub fn ck_canonicalize(ctx: *mut CkCtx, s: *const u8, n: usize, out: *mut u8) -> c_int;
    }
}

/// One `ck_ctx`.  `Send` (a context may move to the reader thread) but not `Sync`: one producer thread per context;
/// the three library drop-ins are the exception (the library serialises them itself).
pub struct Context {
    raw: *mut ffi::CkCtx,
    pub cfg: ffi::CkConfig,
}
unsafe impl Send for Context {}

impl Context {
    pub fn new(device: i32, max_batch_bytes: u64, max_batch_records: u32, table_capacity: u64) -> Result<Self> {
        let cfg = ffi::CkConfig { device, max_batch_bytes, max_batch_records, table_capacity };
        let mut raw = null_mut();
        let rc = unsafe { ffi::ck_init(&cfg, &mut raw) };
        if rc != ffi::CK_OK {
            let msg = unsafe { CStr::from_ptr(ffi::ck_last_error(null())) }.to_string_lossy().into_owned();
            return Err(anyhow!("circkit-cuda: ck_init failed ({rc}): {msg}"));
        }
        Ok(Context { raw, cfg })
    }
    fn check(&self, rc: c_int) -> Result<()> {
        if rc == ffi::CK_OK {
            return Ok(());
        }
        let msg = unsafe { CStr::from_ptr(ffi::ck_last_error(self.raw)) }.to_string_lossy().into_owned();
        Err(anyhow!("circkit-cuda error {rc}: {msg}"))
    }
    /// Forget every key (a new input file).
    pub fn uniq_reset(&self) -> Result<()> {
        self.check(unsafe { ffi::ck_uniq_reset(self.raw) })
    }
    /// Let the uniq table grow on the device as distinct keys arrive, up to `max_keys` keys (None: as many as device
    /// memory allows).  Not with a peer group.
    pub fn uniq_grow(&self, max_keys: Option<u64>) -> Result<()> {
        self.check(unsafe { ffi::ck_uniq_grow(self.raw, max_keys.unwrap_or(u64::MAX)) })
    }
    /// (distinct keys in the uniq table, keys it holds at 2/3 load, growths so far); synchronises both slots.
    pub fn uniq_table_info(&self) -> Result<(u64, u64, u64)> {
        let (mut keys, mut cap, mut grows) = (0u64, 0u64, 0u64);
        self.check(unsafe { ffi::ck_uniq_table_info(self.raw, &mut keys, &mut cap, &mut grows) })?;
        Ok((keys, cap, grows))
    }
    /// Multi-GPU uniq, step 1: this rank's exchange block as a CUDA IPC handle (send it to every rank).
    pub fn peer_export(&self, world: u32, rank: u32, max_records: u32) -> Result<[u8; ffi::CK_PEER_HANDLE_BYTES]> {
        let mut h = [0u8; ffi::CK_PEER_HANDLE_BYTES];
        self.check(unsafe { ffi::ck_peer_export(self.raw, world, rank, max_records, h.as_mut_ptr() as *mut c_void) })?;
        Ok(h)
    }
    /// Multi-GPU uniq, step 2: the handles of all ranks, in rank order.  Afterwards uniq submits are collective rounds.
    pub fn peer_attach(&self, all_handles: &[[u8; ffi::CK_PEER_HANDLE_BYTES]]) -> Result<()> {
        let flat: Vec<u8> = all_handles.iter().flat_map(|h| h.iter().copied()).collect();
        self.check(unsafe { ffi::ck_peer_attach(self.raw, flat.as_ptr() as *const c_void) })
    }
}
impl Drop for Context {
    fn drop(&mut self) {
        unsafe { ffi::ck_destroy(self.raw) }
    }
}

/// A pinned host buffer of `T` (page-locked through the library, so copies run at full PCIe speed and asynchronously).
pub struct Pinned<T> {
    ctx: *mut ffi::CkCtx,
    ptr: *mut T,
    len: usize,
}
impl<T: Copy> Pinned<T> {
    fn new(ctx: &Context, len: usize) -> Result<Self> {
        let p = unsafe { ffi::ck_alloc_pinned(ctx.raw, len.max(1) * std::mem::size_of::<T>()) } as *mut T;
        if p.is_null() {
            return Err(anyhow!("circkit-cuda: cudaMallocHost of {} bytes failed", len * std::mem::size_of::<T>()));
        }
        Ok(Pinned { ctx: ctx.raw, ptr: p, len })
    }
    pub fn as_slice(&self) -> &[T] {
        unsafe { std::slice::from_raw_parts(self.ptr, self.len) }
    }
    pub fn as_mut_slice(&mut self) -> &mut [T] {
        unsafe { std::slice::from_raw_parts_mut(self.ptr, self.len) }
    }
}
impl<T> Drop for Pinned<T> {
    fn drop(&mut self) {
        unsafe { ffi::ck_free_pinned(self.ctx, self.ptr as *mut c_void) }
    }
}

/// One batch under construction / in flight: what the reader thread fills, what the packer leaves, what comes back.
struct Batch {
    bytes: Pinned<u8>,          // record.seq() bytes, raw (line breaks included)
    offsets: Pinned<u64>,       // n + 1
    heads: Vec<Vec<u8>>,        // header line of every record (src/canonicalize.rs:34), ids for --table come from it
    n: usize,
    used: usize,
    base_index: u64,
    // packed form (ck_pack2_host)
    dense: Pinned<u64>,
    lens: Pinned<u32>,
    lane: Pinned<u8>,
    lane_bytes: Pinned<u8>,
    lane_offsets: Pinned<u64>,
    // results
    out: Pinned<u8>,            // canonicalize: aligned arena; uniq / monomerize: the survivors' / written records' compact arena
    out_len: Pinned<u32>,       // monomerize: monomer_length
    full_len: Pinned<u32>,      // monomerize: original_length (length of full_seq)
    end: Pinned<u32>,           // monomerize: the worker's end index (CK_MONO_NONE = None)
    first: Pinned<u64>,
    sel: Pinned<u32>,
    sel_off: Pinned<u64>,
}

/// What the consumer closure gets per record, in input order (the `F` closure of `parallel_fasta`).
pub struct Done<'a> {
    pub head: &'a [u8],
    /// the raw `record.seq()` bytes the reader appended (uniq without `-c` echoes them, `src/uniq.rs:57-59`)
    pub raw_seq: &'a [u8],
    /// canonical form (None for uniq duplicates, and for `uniq` without `canonical_bytes`)
    pub canonical: Option<&'a [u8]>,
    /// global input index of this record and of the first record with the same canonical form (`uniq` only)
    pub index: u64,
    pub first_index: u64,
    /// `monomerize`: full_seq[..monomer_length] of a record the consumer closure writes (`src/monomerize.rs:139-143`), None
    /// for a record it drops; None in the other modes
    pub monomer: Option<&'a [u8]>,
    /// `monomerize`: the `original_length` / `monomer_length` columns of `--table` (`:145-154`); 0 in the other modes
    pub original_length: u64,
    pub monomer_length: u64,
}

#[derive(Clone, Copy, PartialEq)]
pub enum Mode {
    /// `circkit canonicalize`: every record comes back with its canonical form
    Canonicalize,
    /// `circkit uniq`: `first_index == index` marks the survivors; `canonical_bytes` = the `-c` flag
    Uniq { canonical_bytes: bool },
    /// `circkit monomerize`: normalisation, the monomer search, the filters and the extraction of the written monomers run
    /// on the device (`ck_mono_submit`); `Done::monomer` is Some for the records the CLI writes
    Monomerize(ffi::MonoOptions),
}

/// The record pump: replacement for `parallel_fasta(reader, threads, 64, W, F)`.
pub struct Pump {
    ctx: Context,
    mode: Mode,
    threads: u32,
    batches: [Batch; 2],
    cur: usize,                 // batch being filled
    in_flight: [bool; 2],
    next_index: u64,
}

impl Pump {
    /// `threads` = the CLI's `--threads` (`src/commands.rs:122,147`): host packer threads (monomerize does not pack).
    /// `table_capacity` = the initial size of `uniq`'s table in distinct canonical forms; it grows on the device as they
    /// arrive (ignored for canonicalize / monomerize).
    pub fn new(device: i32, mode: Mode, threads: u32, table_capacity: u64) -> Result<Self> {
        const MAX_BYTES: u64 = 256 << 20;
        const MAX_RECORDS: u32 = 1 << 20;
        let uniq = matches!(mode, Mode::Uniq { .. });
        let ctx = Context::new(device, MAX_BYTES, MAX_RECORDS, if uniq { table_capacity.max(1) } else { 0 })?;
        if uniq {
            ctx.uniq_grow(None)?;
        }
        let mk = |ctx: &Context| -> Result<Batch> {
            let r = MAX_RECORDS as usize;
            let b = MAX_BYTES as usize;
            Ok(Batch {
                bytes: Pinned::new(ctx, b + 64)?,
                offsets: Pinned::new(ctx, r + 1)?,
                heads: Vec::new(),
                n: 0,
                used: 0,
                base_index: 0,
                dense: Pinned::new(ctx, unsafe { ffi::ck_pack2_words(MAX_BYTES, MAX_RECORDS) } as usize)?,
                lens: Pinned::new(ctx, r)?,
                lane: Pinned::new(ctx, r)?,
                lane_bytes: Pinned::new(ctx, b + 64)?,
                lane_offsets: Pinned::new(ctx, r + 1)?,
                out: Pinned::new(ctx, unsafe { ffi::ck_out_arena_bytes(MAX_BYTES, MAX_RECORDS) } as usize)?,
                out_len: Pinned::new(ctx, r)?,
                full_len: Pinned::new(ctx, r)?,
                end: Pinned::new(ctx, r)?,
                first: Pinned::new(ctx, r)?,
                sel: Pinned::new(ctx, r)?,
                sel_off: Pinned::new(ctx, r + 1)?,
            })
        };
        let batches = [mk(&ctx)?, mk(&ctx)?];
        Ok(Pump { ctx, mode, threads, batches, cur: 0, in_flight: [false, false], next_index: 0 })
    }

    /// The reader side: one record (`record.head()`, `record.seq()` of seq_io).  Submits the batch when it is full and
    /// drains the other slot through `consume`.
    pub fn push<F: FnMut(Done) -> Result<()>>(&mut self, head: &[u8], seq: &[u8], consume: &mut F) -> Result<()> {
        let cap_b = self.ctx.cfg.max_batch_bytes as usize;
        let cap_r = self.ctx.cfg.max_batch_records as usize;
        if seq.len() > cap_b {
            return Err(anyhow!("circkit-cuda: a record of {} bytes exceeds the batch size", seq.len()));
        }
        if self.batches[self.cur].used + seq.len() > cap_b || self.batches[self.cur].n == cap_r {
            self.flush_current(consume)?;
        }
        let b = &mut self.batches[self.cur];
        if b.n == 0 {
            b.base_index = self.next_index;
            b.offsets.as_mut_slice()[0] = 0;
        }
        b.bytes.as_mut_slice()[b.used..b.used + seq.len()].copy_from_slice(seq);
        b.used += seq.len();
        b.n += 1;
        b.offsets.as_mut_slice()[b.n] = b.used as u64;
        b.heads.push(head.to_vec());
        self.next_index += 1;
        Ok(())
    }

    /// End of input: submit what is left and drain both slots in order.
    pub fn finish<F: FnMut(Done) -> Result<()>>(&mut self, consume: &mut F) -> Result<()> {
        self.flush_current(consume)?;
        let other = self.cur;           // flush_current switched: `cur` is the older batch (if still in flight)
        self.drain(other, consume)?;
        self.drain(other ^ 1, consume)
    }

    fn flush_current<F: FnMut(Done) -> Result<()>>(&mut self, consume: &mut F) -> Result<()> {
        let slot = self.cur;
        if self.batches[slot].n > 0 {
            self.submit(slot)?;
        }
        // the other slot holds the previous batch: its results are due now, and it becomes the batch to fill
        self.drain(slot ^ 1, consume)?;
        self.cur = slot ^ 1;
        Ok(())
    }

    fn submit(&mut self, slot: usize) -> Result<()> {
        let threads = self.threads;
        let mode = self.mode;
        let b = &mut self.batches[slot];
        if let Mode::Monomerize(opt) = mode {
            // the raw bytes as the reader appended them: the device normalises them and needs the raw form for full_seq
            let rc = unsafe {
                ffi::ck_mono_submit(self.ctx.raw, slot as c_int, b.bytes.as_slice().as_ptr(), b.offsets.as_slice().as_ptr(), b.n as u32,
                                    ffi::CK_F_NORMALIZE, &opt)
            };
            self.ctx.check(rc)?;
            self.in_flight[slot] = true;
            return Ok(());
        }
        let mut lane_total = 0u64;
        // pack on the host: needletail normalisation + symbol lanes + 2 bits per base (a quarter of the bytes cross PCIe)
        let rc = unsafe {
            ffi::ck_pack2_host(b.bytes.as_slice().as_ptr(), b.offsets.as_slice().as_ptr(), b.n as u32, ffi::CK_F_NORMALIZE, threads,
                               b.dense.as_mut_slice().as_mut_ptr(), b.lens.as_mut_slice().as_mut_ptr(), b.lane.as_mut_slice().as_mut_ptr(),
                               b.lane_bytes.as_mut_slice().as_mut_ptr(), b.lane_bytes.len as u64,
                               b.lane_offsets.as_mut_slice().as_mut_ptr(), &mut lane_total)
        };
        if rc != ffi::CK_OK {
            return Err(anyhow!("circkit-cuda: ck_pack2_host failed ({rc})"));
        }
        let pb = ffi::CkPackedBatch {
            packed2: b.dense.as_slice().as_ptr(),
            offsets: b.offsets.as_slice().as_ptr(),
            lens: b.lens.as_slice().as_ptr(),
            lane: b.lane.as_slice().as_ptr(),
            lane_bytes: if lane_total > 0 { b.lane_bytes.as_slice().as_ptr() } else { null() },
            lane_offsets: if lane_total > 0 { b.lane_offsets.as_slice().as_ptr() } else { null() },
            lane_bytes_total: lane_total,
            n_records: b.n as u32,
        };
        let rc = match mode {
            Mode::Canonicalize => unsafe { ffi::ck_canon_submit_packed(self.ctx.raw, slot as c_int, &pb, ffi::CK_F_ALIGNED_OUT) },
            Mode::Monomerize(_) => unreachable!(),
            Mode::Uniq { canonical_bytes } => {
                let flags = ffi::CK_F_SURVIVORS | ffi::CK_F_ALIGNED_OUT | if canonical_bytes { 0 } else { ffi::CK_F_NO_BYTES };
                unsafe { ffi::ck_uniq_submit_packed(self.ctx.raw, slot as c_int, &pb, flags, b.base_index) }
            }
        };
        self.ctx.check(rc)?;
        self.in_flight[slot] = true;
        Ok(())
    }

    fn drain<F: FnMut(Done) -> Result<()>>(&mut self, slot: usize, consume: &mut F) -> Result<()> {
        if !self.in_flight[slot] {
            return Ok(());
        }
        self.in_flight[slot] = false;
        let mode = self.mode;
        let raw = self.ctx.raw;
        let b = &mut self.batches[slot];
        let n = b.n;
        match mode {
            Mode::Canonicalize => {
                let rc = unsafe {
                    ffi::ck_canon_wait(raw, slot as c_int, b.out.as_mut_slice().as_mut_ptr(), b.out_len.as_mut_slice().as_mut_ptr(),
                                       null_mut(), null_mut(), null_mut())
                };
                self.ctx.check(rc)?;
                let b = &self.batches[slot];
                let (off, out, len) = (b.offsets.as_slice(), b.out.as_slice(), b.out_len.as_slice());
                for i in 0..n {
                    let at = 32 * ((off[i] >> 5) as usize + i);           // CK_F_ALIGNED_OUT layout
                    consume(Done {
                        head: &b.heads[i],
                        raw_seq: &b.bytes.as_slice()[off[i] as usize..off[i + 1] as usize],
                        canonical: Some(&out[at..at + len[i] as usize]),
                        index: b.base_index + i as u64,
                        first_index: b.base_index + i as u64,
                        monomer: None,
                        original_length: 0,
                        monomer_length: 0,
                    })?;
                }
            }
            Mode::Uniq { canonical_bytes } => {
                let mut ns = 0u32;
                let rc = unsafe {
                    ffi::ck_uniq_wait_survivors(raw, slot as c_int, &mut ns, b.sel.as_mut_slice().as_mut_ptr(),
                                                b.sel_off.as_mut_slice().as_mut_ptr(), b.out.as_mut_slice().as_mut_ptr(),
                                                b.out_len.as_mut_slice().as_mut_ptr(), null_mut(), b.first.as_mut_slice().as_mut_ptr())
                };
                self.ctx.check(rc)?;
                let b = &self.batches[slot];
                let (off, out, len, first) = (b.offsets.as_slice(), b.out.as_slice(), b.out_len.as_slice(), b.first.as_slice());
                let (sel, sel_off) = (b.sel.as_slice(), b.sel_off.as_slice());
                let mut k = 0usize;                                       // next survivor
                for i in 0..n {
                    let survivor = k < ns as usize && sel[k] as usize == i;
                    let canonical = if survivor && canonical_bytes {
                        let at = sel_off[k] as usize;
                        Some(&out[at..at + len[i] as usize])
                    } else {
                        None
                    };
                    if survivor {
                        k += 1;
                    }
                    consume(Done {
                        head: &b.heads[i],
                        raw_seq: &b.bytes.as_slice()[off[i] as usize..off[i + 1] as usize],
                        canonical,
                        index: b.base_index + i as u64,
                        first_index: first[i],
                        monomer: None,
                        original_length: 0,
                        monomer_length: 0,
                    })?;
                }
            }
            Mode::Monomerize(_) => {
                let mut nw = 0u32;
                let rc = unsafe {
                    ffi::ck_mono_wait(raw, slot as c_int, &mut nw, b.sel.as_mut_slice().as_mut_ptr(), b.sel_off.as_mut_slice().as_mut_ptr(),
                                      b.out.as_mut_slice().as_mut_ptr(), b.out_len.as_mut_slice().as_mut_ptr(),
                                      b.full_len.as_mut_slice().as_mut_ptr(), b.end.as_mut_slice().as_mut_ptr())
                };
                self.ctx.check(rc)?;
                let b = &self.batches[slot];
                let (off, out, len, full) = (b.offsets.as_slice(), b.out.as_slice(), b.out_len.as_slice(), b.full_len.as_slice());
                let (sel, sel_off) = (b.sel.as_slice(), b.sel_off.as_slice());
                let mut k = 0usize;                                       // next written record
                for i in 0..n {
                    let monomer = if k < nw as usize && sel[k] as usize == i {
                        let at = sel_off[k] as usize;
                        k += 1;
                        Some(&out[at..at + len[i] as usize])
                    } else {
                        None
                    };
                    consume(Done {
                        head: &b.heads[i],
                        raw_seq: &b.bytes.as_slice()[off[i] as usize..off[i + 1] as usize],
                        canonical: None,
                        index: b.base_index + i as u64,
                        first_index: b.base_index + i as u64,
                        monomer,
                        original_length: full[i] as u64,
                        monomer_length: len[i] as u64,
                    })?;
                }
            }
        }
        let b = &mut self.batches[slot];
        b.n = 0;
        b.used = 0;
        b.heads.clear();
        Ok(())
    }
}

// ---- library drop-ins (lib/src/canonicalize.rs:5,41,54): a lazily created process-wide context ------------------------
static DEFAULT: OnceLock<Mutex<Context>> = OnceLock::new();
fn default_ctx() -> &'static Mutex<Context> {
    DEFAULT.get_or_init(|| Mutex::new(Context::new(0, 1 << 20, 1 << 12, 0).expect("circkit-cuda: no usable CUDA device")))
}

/// `circkit::canonicalize::lmsr_index` (lib/src/canonicalize.rs:5): start of the lexicographically minimal rotation, the
/// smallest one on ties.
pub fn lmsr_index(s: &[u8]) -> usize {
    let ctx = default_ctx().lock().unwrap();
    let mut idx = 0usize;
    let rc = unsafe { ffi::ck_lmsr_index(ctx.raw, s.as_ptr(), s.len(), &mut idx) };
    ctx.check(rc).expect("ck_lmsr_index");
    idx
}
/// `circkit::canonicalize::lmsr` (lib/src/canonicalize.rs:41).
pub fn lmsr(s: &[u8]) -> Vec<u8> {
    let ctx = default_ctx().lock().unwrap();
    let mut out = vec![0u8; s.len()];
    let rc = unsafe { ffi::ck_lmsr(ctx.raw, s.as_ptr(), s.len(), out.as_mut_ptr()) };
    ctx.check(rc).expect("ck_lmsr");
    out
}
/// `circkit::canonicalize` (lib/src/canonicalize.rs:54): min(lmsr(s), lmsr(revcomp(s))), ties keep the reverse complement.
pub fn canonicalize(s: &[u8]) -> Vec<u8> {
    let ctx = default_ctx().lock().unwrap();
    let mut out = vec![0u8; s.len()];
    let rc = unsafe { ffi::ck_canonicalize(ctx.raw, s.as_ptr(), s.len(), out.as_mut_ptr()) };
    ctx.check(rc).expect("ck_canonicalize");
    out
}
