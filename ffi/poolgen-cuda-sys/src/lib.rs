//! Raw bindings of `include/poolgen_cuda.h` (libpoolgen_cuda.so, CUDA C++ for sm_100a) and a thin safe layer for the
//! call sequence poolgen's chunk workers need.  Every function returns `PG_OK` (0) or a negative error class; the text
//! is available from `pg_last_error`.  Nothing here falls back to the CPU.
#![allow(non_camel_case_types)]
use std::ffi::{c_char, c_int, c_void, CStr};

pub const PG_OK: c_int = 0;
pub const PG_ERR_ARG: c_int = -1;
pub const PG_ERR_CUDA: c_int = -2;
pub const PG_ERR_STATE: c_int = -3;
pub const PG_ERR_UNSUPPORTED: c_int = -4;
pub const PG_ERR_NCCL: c_int = -5;

/// the per-locus callbacks (`fn(&mut LocusCountsAndPhenotypes, &FilterStats) -> Option<String>`)
pub const PG_KIND_OLS: c_int = 0; // gwas::ols_iterate, src/gwas/ols.rs:201-276
pub const PG_KIND_CORR: c_int = 1; // gwas::correlation, src/gwas/correlation_test.rs:73-129
pub const PG_KIND_CHISQ: c_int = 2; // tables::chisq, src/tables/chisq_test.rs:5-47
pub const PG_KIND_FISHER: c_int = 3; // tables::fisher, src/tables/fisher_exact_test.rs:32-130
pub const PG_KIND_OLS_KINSHIP: c_int = 4; // header selector of the writer only

pub const PG_LOCUS_FILTERED: u64 = 0; // the callback returned None (filter)
pub const PG_LOCUS_OK: u64 = 1; // Some(line)
pub const PG_LOCUS_FAILED: u64 = 2; // None (regression failed)
pub const PG_LOCUS_UNSUPPORTED: u64 = 3;
pub const PG_LOCUS_PANIC: u64 = 4; // the reference would panic on this locus
pub const PG_STREAM_DEPTH: usize = 3;

#[repr(C)]
pub struct pg_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct pg_scan {
    _private: [u8; 0],
}
#[repr(C)]
pub struct pg_batch {
    _private: [u8; 0],
}
#[repr(C)]
pub struct pg_kin {
    _private: [u8; 0],
}
#[repr(C)]
pub struct pg_comm {
    _private: [u8; 0],
}
pub const PG_COMM_ID_BYTES: usize = 128;

/// FilterStats (src/base/structs_and_traits.rs:69-78), sync-path fields
#[repr(C)]
pub struct pg_filter {
    pub remove_ns: i32,
    pub min_coverage_depth: u64,
    pub min_allele_frequency: f64,
    pub max_missingness_rate: f64,
    pub n_pool_sizes: i32,
    pub pool_sizes: *const f64,
}

#[repr(C)]
pub struct pg_results {
    pub n_loci: i64,
    pub n_slots: i32,
    pub n_phen: i32,
    pub meta: *const u64,
    pub freq_mean: *const f64,
    pub stats: *const f64,
}

#[repr(C)]
pub struct pg_row_labels {
    pub positions: *const u64,
    pub text: *const c_char,
    pub line_offsets: *const u64,
    pub chr_names: *const *const c_char,
    pub chr_index: *const u32,
}

extern "C" {
    // ---- context
    pub fn pg_abi_version() -> c_int;
    pub fn pg_init(device: c_int, out: *mut *mut pg_ctx) -> c_int;
    pub fn pg_destroy(ctx: *mut pg_ctx);
    pub fn pg_last_error(ctx: *const pg_ctx) -> *const c_char;
    pub fn pg_device_info(ctx: *mut pg_ctx, sm_count: *mut c_int, cc_major: *mut c_int, cc_minor: *mut c_int, total_mem: *mut usize) -> c_int;
    /// free and total device memory now (cudaMemGetInfo): size device blocks from what is free on a shared GPU
    pub fn pg_device_mem_info(ctx: *mut pg_ctx, free_bytes: *mut usize, total_bytes: *mut usize) -> c_int;
    pub fn pg_pinned_alloc(ctx: *mut pg_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn pg_pinned_free(ctx: *mut pg_ctx, p: *mut c_void) -> c_int;
    // ---- scan configuration
    pub fn pg_scan_open(ctx: *mut pg_ctx, kind: c_int, filter: *const pg_filter, n_pools: c_int, n_alleles: c_int, allele_codes: *const u8, phen: *const f64, k: c_int, out: *mut *mut pg_scan) -> c_int;
    pub fn pg_scan_close(scan: *mut pg_scan) -> c_int;
    // ---- resident batches
    pub fn pg_batch_create(scan: *mut pg_scan, capacity_loci: i64, out: *mut *mut pg_batch) -> c_int;
    pub fn pg_batch_destroy(b: *mut pg_batch) -> c_int;
    pub fn pg_batch_upload_counts(b: *mut pg_batch, counts: *const u32, n_loci: i64) -> c_int;
    pub fn pg_batch_upload_counts_u16(b: *mut pg_batch, counts: *const u16, n_loci: i64) -> c_int;
    pub fn pg_batch_upload_counts_u8(b: *mut pg_batch, counts: *const u8, n_loci: i64) -> c_int;
    pub fn pg_batch_upload_freq(b: *mut pg_batch, freq: *const f64, depth: *const u32, n_loci: i64) -> c_int;
    pub fn pg_batch_upload_sync_text(b: *mut pg_batch, text: *const c_char, n_bytes: usize, n_loci: *mut i64) -> c_int;
    pub fn pg_batch_text_labels(b: *mut pg_batch, line_offsets: *mut *const u64, positions: *mut *const u64) -> c_int;
    pub fn pg_batch_synth(b: *mut pg_batch, seed: u64, first_locus: i64, n_loci: i64) -> c_int;
    pub fn pg_batch_run(b: *mut pg_batch) -> c_int;
    pub fn pg_batch_download(b: *mut pg_batch) -> c_int;
    pub fn pg_batch_sync(b: *mut pg_batch) -> c_int;
    pub fn pg_batch_results(b: *mut pg_batch, out: *mut pg_results) -> c_int;
    pub fn pg_batch_time_runs(b: *mut pg_batch, iters: c_int, ms_total: *mut f32, n_launches: *mut c_int) -> c_int;
    pub fn pg_batch_bytes(b: *mut pg_batch, input_bytes: *mut usize, result_bytes: *mut usize) -> c_int;
    // ---- streaming (one scan handle per reader thread)
    pub fn pg_scan_stream_begin(scan: *mut pg_scan, max_loci_per_slab: i64) -> c_int;
    pub fn pg_scan_submit_counts(scan: *mut pg_scan, counts: *const u32, n_loci: i64, ticket: *mut c_int) -> c_int;
    pub fn pg_scan_submit_counts_u16(scan: *mut pg_scan, counts: *const u16, n_loci: i64, ticket: *mut c_int) -> c_int;
    pub fn pg_scan_submit_counts_u8(scan: *mut pg_scan, counts: *const u8, n_loci: i64, ticket: *mut c_int) -> c_int;
    pub fn pg_scan_submit_freq(scan: *mut pg_scan, freq: *const f64, depth: *const u32, n_loci: i64, ticket: *mut c_int) -> c_int;
    pub fn pg_scan_submit_sync_text(scan: *mut pg_scan, text: *const c_char, n_bytes: usize, ticket: *mut c_int, n_loci: *mut i64) -> c_int;
    pub fn pg_scan_collect(scan: *mut pg_scan, ticket: c_int, out: *mut pg_results) -> c_int;
    pub fn pg_scan_text_labels(scan: *mut pg_scan, ticket: c_int, line_offsets: *mut *const u64, positions: *mut *const u64) -> c_int;
    // ---- ols_iter_with_kinship
    pub fn pg_kin_open(ctx: *mut pg_ctx, n_pools: c_int, max_columns: i64, out: *mut *mut pg_kin) -> c_int;
    pub fn pg_kin_close(kin: *mut pg_kin) -> c_int;
    pub fn pg_kin_reset(kin: *mut pg_kin) -> c_int;
    pub fn pg_kin_columns(kin: *mut pg_kin) -> i64;
    pub fn pg_kin_append_columns(kin: *mut pg_kin, cols: *const f64, p_add: i64) -> c_int;
    pub fn pg_kin_append_counts(kin: *mut pg_kin, filter: *const pg_filter, n_alleles: c_int, allele_codes: *const u8, counts: *const u32, n_loci: i64, keep_p_minus_1: c_int, n_cols_added: *mut i64) -> c_int;
    pub fn pg_kin_last_labels(kin: *mut pg_kin, n_cols: i64, col_locus: *mut i64, col_allele: *mut u8) -> c_int;
    pub fn pg_kin_append_sync_text(kin: *mut pg_kin, filter: *const pg_filter, text: *const c_char, n_bytes: usize, max_loci: i64, keep_p_minus_1: c_int, n_loci: *mut i64, n_cols_added: *mut i64) -> c_int;
    pub fn pg_kin_text_labels(kin: *mut pg_kin, line_offsets: *mut *const u64, positions: *mut *const u64) -> c_int;
    /// sync2csv rows of columns [first, first + count) of the last text append, formatted on the device; stops at
    /// the last whole row that fits `capacity` (see pg_kin_format_frequency_rows in poolgen_cuda.h)
    pub fn pg_kin_format_frequency_rows(kin: *mut pg_kin, first: i64, count: i64, out: *mut c_char, capacity: usize, n_bytes: *mut usize, n_rows: *mut i64) -> c_int;
    pub fn pg_kin_synth(kin: *mut pg_kin, seed: u64, first_locus: i64, n_loci: i64) -> c_int;
    pub fn pg_kin_get_columns(kin: *mut pg_kin, first: i64, count: i64, out: *mut f64) -> c_int;
    pub fn pg_kin_gram(kin: *mut pg_kin) -> c_int;
    /// K += G G' of the resident columns (blocks 2..B of a column set larger than the device; pg_kin_reset keeps K)
    pub fn pg_kin_gram_accumulate(kin: *mut pg_kin) -> c_int;
    pub fn pg_kin_gram_time(kin: *mut pg_kin, iters: c_int, ms_total: *mut f32) -> c_int;
    pub fn pg_kin_partial(kin: *mut pg_kin, device_ptr: *mut *mut f64, n_elems: *mut usize) -> c_int;
    pub fn pg_kin_partial_get(kin: *mut pg_kin, out_host: *mut f64) -> c_int;
    pub fn pg_kin_partial_set(kin: *mut pg_kin, in_host: *const f64) -> c_int;
    pub fn pg_kin_eig_select(kin: *mut pg_kin, p_total: i64, variance_explained: f64, n_eigenvecs: *mut c_int) -> c_int;
    pub fn pg_kin_eigvals(kin: *mut pg_kin, out: *mut f64, count: c_int) -> c_int;
    pub fn pg_kin_set_covariates(kin: *mut pg_kin, cov: *const f64, m: c_int) -> c_int;
    pub fn pg_kin_covar_scan(kin: *mut pg_kin, phen: *const f64, k: c_int, iters: c_int, ms_total: *mut f32, beta: *mut *const f64, var: *mut *const f64, pval: *mut *const f64) -> c_int;
    /// mle_iter_with_kinship: gwas::mle_with_covariate (src/gwas/mle.rs:307-463) over the same columns and covariates
    pub fn pg_kin_mle_scan(kin: *mut pg_kin, phen: *const f64, k: c_int, ms: *mut f32, beta: *mut *const f64, var: *mut *const f64, pval: *mut *const f64) -> c_int;
    // ---- the reference's CSV rows
    pub fn pg_format_header(kind: c_int, out: *mut c_char, capacity: usize, n_bytes: *mut usize) -> c_int;
    pub fn pg_format_rows(kind: c_int, res: *const pg_results, labels: *const pg_row_labels, n_threads: c_int, out: *mut c_char, capacity: usize, n_bytes: *mut usize) -> c_int;
    pub fn pg_format_rows_ex(kind: c_int, res: *const pg_results, labels: *const pg_row_labels, flags: c_int, n_pools: c_int, n_threads: c_int, out: *mut c_char, capacity: usize, n_bytes: *mut usize) -> c_int;
    pub fn pg_format_kinship_rows(n_columns: i64, k: c_int, chromosome: *const *const c_char, position: *const u64, allele: *const *const c_char, beta: *const f64, pval: *const f64, n_threads: c_int, out: *mut c_char, capacity: usize, n_bytes: *mut usize) -> c_int;
    pub fn pg_sort_loci(labels: *const pg_row_labels, n_loci: i64, order_out: *mut i64) -> c_int;
    pub fn pg_format_frequency_header(pool_names: *const *const c_char, n_pools: c_int, out: *mut c_char, capacity: usize, n_bytes: *mut usize) -> c_int;
    pub fn pg_format_frequency_rows(n_columns: i64, n_pools: c_int, columns: *const f64, col_locus: *const i64, col_allele: *const u8, labels: *const pg_row_labels, locus_order: *const i64, n_order: i64, n_threads: c_int, out: *mut c_char, capacity: usize, n_bytes: *mut usize) -> c_int;
    pub fn pg_format_f64(x: f64, n_digits: c_int, out: *mut c_char, capacity: usize) -> c_int;
    // ---- several GPUs: shard ranges, the library's NCCL communicator, the kinship exchange step
    pub fn pg_shard_range(total: i64, rank: c_int, world: c_int, begin: *mut i64, end: *mut i64) -> c_int;
    pub fn pg_nccl_version(version: *mut c_int) -> c_int;
    pub fn pg_init_multi(devices: *const c_int, n: c_int, ctxs_out: *mut *mut pg_ctx, comm_out: *mut *mut pg_comm) -> c_int;
    pub fn pg_comm_unique_id(id: *mut u8) -> c_int;
    pub fn pg_comm_init_rank(ctx: *mut pg_ctx, id: *const u8, rank: c_int, world: c_int, out: *mut *mut pg_comm) -> c_int;
    pub fn pg_comm_info(comm: *const pg_comm, world: *mut c_int, n_local: *mut c_int, first_rank: *mut c_int) -> c_int;
    pub fn pg_comm_destroy(comm: *mut pg_comm) -> c_int;
    pub fn pg_kin_allreduce(comm: *mut pg_comm, kins: *const *mut pg_kin, n_local: c_int, p_total: *mut i64, ms: *mut f32) -> c_int;
    pub fn pg_kin_copy_covariates(dst: *mut pg_kin, src: *const pg_kin) -> c_int;
}

/// `Err(message)` for a negative return code
pub fn check(ctx: *const pg_ctx, rc: c_int) -> Result<(), String> {
    if rc == PG_OK {
        return Ok(());
    }
    let msg = unsafe {
        let p = pg_last_error(ctx);
        if p.is_null() { String::new() } else { CStr::from_ptr(p).to_string_lossy().into_owned() }
    };
    Err(format!("libpoolgen_cuda error {rc}: {msg}"))
}

/// One reader thread's scan: text blocks in, the reference's CSV rows out -- what the body of
/// `FileSyncPhen::read_analyse_write`'s per-chunk worker (src/base/sync.rs:794-870) becomes.  `blocks` yields
/// line-aligned byte blocks of the thread's chunk (pinned memory for an asynchronous copy; each block must stay alive
/// until its rows have been written, which the ring of PG_STREAM_DEPTH blocks below guarantees).
pub struct TextScan {
    pub ctx: *mut pg_ctx,
    pub scan: *mut pg_scan,
    pub kind: c_int,
    pending: Vec<(c_int, *const c_char)>,
    rows: Vec<u8>,
}

impl TextScan {
    pub fn new(ctx: *mut pg_ctx, scan: *mut pg_scan, kind: c_int, max_loci_per_block: i64) -> Result<Self, String> {
        check(ctx, unsafe { pg_scan_stream_begin(scan, max_loci_per_block) })?;
        Ok(TextScan { ctx, scan, kind, pending: Vec::new(), rows: vec![0u8; 1 << 20] })
    }

    fn finish_oldest(&mut self, n_threads: c_int, sink: &mut dyn std::io::Write) -> Result<(), String> {
        let (ticket, text) = self.pending.remove(0);
        let mut res = pg_results { n_loci: 0, n_slots: 0, n_phen: 0, meta: std::ptr::null(), freq_mean: std::ptr::null(), stats: std::ptr::null() };
        check(self.ctx, unsafe { pg_scan_collect(self.scan, ticket, &mut res) })?;
        let (mut off, mut pos) = (std::ptr::null(), std::ptr::null());
        check(self.ctx, unsafe { pg_scan_text_labels(self.scan, ticket, &mut off, &mut pos) })?;
        let lab = pg_row_labels { positions: pos, text, line_offsets: off, chr_names: std::ptr::null(), chr_index: std::ptr::null() };
        let mut need: usize = 0;
        let mut rc = unsafe { pg_format_rows(self.kind, &res, &lab, n_threads, self.rows.as_mut_ptr() as *mut c_char, self.rows.len(), &mut need) };
        if rc != PG_OK && need > self.rows.len() {
            self.rows.resize(need, 0);
            rc = unsafe { pg_format_rows(self.kind, &res, &lab, n_threads, self.rows.as_mut_ptr() as *mut c_char, self.rows.len(), &mut need) };
        }
        check(self.ctx, rc)?;
        sink.write_all(&self.rows[..need]).map_err(|e| e.to_string())
    }

    /// submit one block; rows of the oldest block are written once PG_STREAM_DEPTH blocks are in flight
    pub fn push(&mut self, block: &[u8], n_threads: c_int, sink: &mut dyn std::io::Write) -> Result<(), String> {
        let mut ticket: c_int = 0;
        check(self.ctx, unsafe { pg_scan_submit_sync_text(self.scan, block.as_ptr() as *const c_char, block.len(), &mut ticket, std::ptr::null_mut()) })?;
        self.pending.push((ticket, block.as_ptr() as *const c_char));
        if self.pending.len() == PG_STREAM_DEPTH {
            self.finish_oldest(n_threads, sink)?;
        }
        Ok(())
    }

    pub fn finish(&mut self, n_threads: c_int, sink: &mut dyn std::io::Write) -> Result<(), String> {
        while !self.pending.is_empty() {
            self.finish_oldest(n_threads, sink)?;
        }
        Ok(())
    }
}
