// pg_kin.h -- the handle of the ols_iter_with_kinship path (shared by pg_kinship.cu and pg_comm.cu; not part of the ABI)
#pragma once
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "pg_internal.h"

struct pg_kin {
    pg_ctx *ctx = nullptr;
    int n = 0, ldg = 0;
    int64_t cap = 0, P = 0;
    int64_t P_total = 0;      // columns over all shards (pg_kin_allreduce); 0 = this handle holds them all
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    pg::DeviceBuffer<double> d_G;
    pg::DeviceBuffer<double> d_K;   // [n][n] partial Gram matrix (sum over the resident columns)
    pg::DeviceBuffer<double> d_ws;  // split-K workspace
    int nt = 0, n_slices = 0;
    // covariates
    int m = -1;
    bool minnorm = false;         // m == n: the reference's n < p branch (pg_kin_eig_select)
    std::vector<double> eigvals;  // descending
    std::vector<double> Q;        // [1+m][ldg] orthonormal basis of [1 | PCs] (host)
    std::vector<double> C;        // [m][ldg] the covariates themselves (pg_kin_mle_scan: the simplex search is not basis-invariant)
    pg::DeviceBuffer<double> d_mle;  // pg_kin_mle_scan: centred covariates and phenotypes, then the fixed moments
    pg::DeviceBuffer<double> d_V;    // [(1+m) + k][ldg]
    pg::DeviceBuffer<double> d_ptab;
    double ptab_isd = 0, ptab_bits = 0, ptab_t1 = 0, ptab_t0 = 0;
    int ptab_M = 0;
    // results
    int k = 0;
    pg::DeviceBuffer<double> d_res;  // [3][k][P]
    pg::PinnedBuffer<double> h_res;
    pg::DeviceBuffer<int64_t> d_defer;  // covariate scan: [count | columns left to the two-pass kernel]
    pg::DeviceBuffer<double> d_part;    // covariate scan (DMMA form in pool passes): partial sums per column block
    // loader scratch
    pg::DeviceBuffer<uint32_t> d_sel;
    pg::DeviceBuffer<int64_t> d_off;
    pg::DeviceBuffer<int64_t> d_col_locus;
    pg::DeviceBuffer<uint8_t> d_col_allele;
    pg::DeviceBuffer<uint8_t> d_scan_tmp;
    pg::DeviceBuffer<uint32_t> d_counts;
    pg::DeviceBuffer<double> d_w;
    pg::TextScratch text;  // sync text parsed on the device (pg_kin_append_sync_text)
    // the columns the last append took from sync text: [text_first, text_first + text_cols); text_cols = -1 when the
    // last append (or reset) was anything else
    int64_t text_first = 0, text_cols = -1;
    // sync2csv rows formatted on the device (pg_fmt.cu)
    pg::DeviceBuffer<uint64_t> d_fmt_off;   // [rows + 1] row lengths, then their exclusive scan
    pg::DeviceBuffer<uint32_t> d_fmt_chr;   // [rows] chromosome bytes
    pg::DeviceBuffer<uint8_t> d_fmt_tmp;    // scan scratch
    pg::DeviceBuffer<unsigned long long> d_fmt_info;
    pg::PinnedBuffer<unsigned long long> h_fmt_info;
    pg::DeviceBuffer<char> d_fmt_text;      // the rows of one call
    // eigen step: cuSOLVER is mapped and its handle created by a background thread started in pg_kin_open and joined
    // by pg_kin_eig_select / the destructor
    std::thread warm;
    void *solver = nullptr;  // cusolverDnHandle_t
    ~pg_kin();
};
