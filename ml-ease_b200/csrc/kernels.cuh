// kernels.cuh -- launcher declarations shared by the translation units of libmlease_b200.so
#pragma once
#include "common.cuh"

namespace mlease {

// K1 (k1_score_grad.cu)
bool k1_dense_plan(int ldx, int* R_out, int* S_out, int* G_out, size_t* smem_out, int* ctas_per_sm);
int k1_csr_window(int ldx);
cudaError_t k1_launch(const Problem* d_probs, int nprob, bool csr, int ldx, int has_bias, int ctas_per_problem,
                      int force_emit, cudaStream_t stream, int* launches, int csr_fx = 0, int nprob_dyn = 0);

// fused multi-lambda CSR K1 (k1_csr_fused.cu)
bool k1f_plan(long long n, int ldx, int L, int num_sms, int* S_out, int* rows_out, int* LP_out, size_t* smem_out);
cudaError_t k1f_build(long long n, int Dg, long long nnz, const long long* rowptr, const int* colidx, const float* vals, int S, int sg_rows, int* ngrp_out,
                      int** perm_out, int** depth_out, long long** goff_out, unsigned short** row16_out, float** val_out, long long* total_out,
                      cudaStream_t st);
cudaError_t k1f_launch(const Problem* d_probs, int ngroups, int L, int S, int LP, size_t smem, int has_bias, int force_emit, cudaStream_t st, int* launches);

// Newton state machine (newton.cu)
cudaError_t newton_begin(const Problem* d_probs, int nprob, double xtol, int max_newton, int hess_policy,
                         int invalidate_hess, int rebuild_is_expensive, cudaStream_t st, int* launches);
cudaError_t k1_reduce_decide(const Problem* d_probs, int nprob, int Dt, cudaStream_t st, int* launches, int spec = 0);
cudaError_t newton_solve(const Problem* d_probs, int nprob, int ldh, cudaStream_t st, int* launches, int group_L = 1);

// K2 (k2_gram.cu)
int gram_make_tensor_map(void* out_map_host, const void* xt, long long n, int Dp);
int gram_tile_list(int Dp, short* bi_bj_pairs, int max_tiles, int pair_tiles = 0);
cudaError_t gram_launch_tcgen05(const Problem* d_probs, int nprob, const void* d_tmaps, const void* d_tiles, int ntiles,
                                int nslices, int force, cudaStream_t st, int* launches, int share = 0);
cudaError_t gram_launch_csr_tcgen05(const Problem* d_probs, int nprob, const void* d_tiles, int ntiles, int nslices, int force,
                                    int bias_col, cudaStream_t st, int* launches, int share = 0);
cudaError_t csr_bm_offsets(long long n, const long long* rowptr, const int* colidx, int nblk, long long ngroups, long long* offs, cudaStream_t st);
cudaError_t csr_bm_fill(long long n, const long long* rowptr, const int* colidx, const float* vals, int nblk, long long ngroups,
                        const long long* offs, unsigned short* keys, float* bvals, cudaStream_t st);
cudaError_t gram_launch_simt(const Problem* d_probs, int nprob, int Dp, int force, cudaStream_t st, int* launches);

// K3 (k3_cholesky.cu)
cudaError_t cholesky_launch(const Problem* d_probs, int nprob, int ldh, cudaStream_t st, int* launches, int share = 0, int skip_prep = 0,
                            int want_hinv = 0);
bool cholesky_factored_direction(int ldh);   // wide systems: Ysym holds Y = L^-1 (bf16, symmetric storage), the direction is Y^T (Y q)
cudaError_t cholesky_share_begin(const Problem* d_probs, int nprob, int share, cudaStream_t st, int* launches);
cudaError_t cholesky_share_end(const Problem* d_probs, int nprob, int share, cudaStream_t st, int* launches);

// K4 (k4_consensus.cu)
cudaError_t admm_reset(const Problem* d_probs, int nprob, int L, double* d_z, int ldv, const double* d_rho_eff,
                       cudaStream_t st, int* launches);
cudaError_t admm_init(const Problem* d_probs, int nprob, const double* d_z, int ldv, cudaStream_t st, int* launches);
cudaError_t admm_pack(const Problem* d_probs, int nlocal_parts, int L, int Dt, double* d_exchange, cudaStream_t st,
                      int* launches);
cudaError_t admm_consensus(const Problem* d_probs, int nlocal_parts, int L, int Dt, int ldv, int P, const double* d_exchange_sum,
                           double* d_z, const double* d_wz, const double* d_rho_eff_next, double* d_diff, cudaStream_t st,
                           int* launches, const double* d_l1_thr = nullptr);

// posterior variance (k6_postvar.cu): exact fp64 Hessian diagonal / full Hessian into Lc
cudaError_t postvar_rowweights(const Problem* d_prob, const double* d_w, int has_bias, double* d_dvec, cudaStream_t st, int* launches);
cudaError_t postvar_diag(const Problem* d_prob, const double* d_dvec, int has_bias, double* d_H, cudaStream_t st, int* launches);
cudaError_t postvar_hessian(const Problem* d_prob, bool csr, int ldh, const double* d_dvec, const double* d_q, int has_bias, cudaStream_t st,
                            int* launches);

// K5 (k5_score.cu)
cudaError_t score_launch(int Dg, long long nrows, const long long* rowptr, const int* colidx, const float* vals, long long ldx,
                         const float* offset, const double* d_model, double intercept_term, int binary_feature, float* pred,
                         cudaStream_t st);
cudaError_t loglik_launch(long long nrows, const int* response, const float* pred, const float* weight, long long combiner_block,
                          float* d_ll, double* d_block_sum, double* d_block_cnt, int* d_bad, cudaStream_t st);

// upload helpers (session.cu)
}  // namespace mlease
