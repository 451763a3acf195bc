// common.cuh -- shared device structures and sm_100a PTX wrappers (mbarrier, bulk-copy TMA,
// tensor-map TMA, tcgen05/TMEM).  B200 only: compile with -gencode arch=compute_100a,code=sm_100a.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mlease {

// secant pairs kept on top of the (possibly stale) explicit inverse Hessian.  Measured at 1M x 10k x 1 %: 12 / 16 pairs save
// 2-4 % of the K1 passes and cost 45-60 % more two-loop time
constexpr int BFGS_M = 6;

// ------------------------------------------------------------------------------------------
// Per-problem control block, device resident.  A "problem" is one (local partition, lambda)
// x-update = one AdmmReducer.reduce call (jobs/RegressionAdmmTrain.java:642-718).
// Every kernel of the Newton slot reads these flags and exits early when it has nothing to
// do, so the host launches a fixed kernel sequence per slot and never branches on device data.
// ------------------------------------------------------------------------------------------
struct Ctrl {
  int done;          // x-update finished (converged or gave up)
  int have_dir;      // a Newton direction exists for the accepted point
  int need_solve;    // accepted a point this slot -> compute a new direction
  int need_hess;     // ... and rebuild Gram + Cholesky first
  int emit;          // K1 must write the sqrt(d)-scaled bf16 copy (a Hessian rebuild may follow)
  int hess_valid;    // a Cholesky factor exists (possibly stale -> chord Newton)
  int fail;          // 1 = not SPD, 2 = line search gave up, 3 = max_newton hit
  int newton_steps;  // accepted steps in this x-update
  int evals;         // K1 passes in this x-update
  int rejects;       // rejected trial points in this x-update
  int hess_builds;   // Gram+Cholesky rebuilds in this x-update
  int stall;         // consecutive poor contractions
  int bfgs_count;    // secant pairs stored so far (ring of BFGS_M), reset when the Hessian is rebuilt
  double h0_scale;   // self-scaling factor applied to the explicit inverse inside the L-BFGS two-loop (rebuild_is_expensive only; 1 after a rebuild)
  int k1_chunks;     // number of per-CTA partials the last K1 pass wrote for this problem (gpart / fpart rows)
  int refresh_next;  // rebuild the Hessian at the first point of the NEXT x-update (chord steps contracted slowly)
  int skip_eval;     // 1: the gradient at the start point of this x-update is already in g_t (data term) -- see admm_consensus_kernel:
                     //    slot 0 runs no K1 pass for this problem, the decide kernel accepts the start point on that gradient
  int warm_used;     // this x-update started from the estimated gradient (skip_eval was consumed): its first exact evaluation is accepted
                     // unconditionally (the estimate is not good enough to police a line search; the secant pair of that step is
                     // kept whenever s.y > 0: it carries most of the curvature information of the update)
  int build_step;    // newton_steps at the last rebuild of this x-update (0 if none yet): steps taken on the current factor = newton_steps - build_step
  double worst_ratio;// largest |g_new|/|g_old| seen over the chord steps of this x-update
  double alpha;      // current step length along dir
  double phi0;       // g_acc . dir  (< 0)
  double f_acc, f_t; // objective at accepted / trial point
  double gnorm;      // |g_acc|_inf
  double gnorm_prev;
  double dirnorm;    // |dir|_inf
  double dirnorm_prev;
  double xtol;
  int max_newton;
  int hess_policy;   // 0 adaptive chord, 1 every step
  int rebuild_is_expensive;  // a Gram+Cholesky rebuild costs more than ~8 passes over X: never rebuild mid-update, lean on L-BFGS
  // cumulative counters (never reset by begin-of-iteration)
  long long tot_evals, tot_newton, tot_rejects, tot_hess;
  // factored inverse the direction kernels read: this problem's own Ysym after its own factorisation, the group leader's after a
  // shared cold-start factorisation (the lambdas of a partition then stream ONE copy of Y for all their directions)
  const void* ysym_use;
};

// One problem's device pointers.  Vectors have length ldv (= ldx, multiple of 4, >= Dt) and are
// zero in [Dt, ldv).  The bias column is PHYSICAL: column Dt-1 of X is 1.0f for every row when the
// problem has an intercept (llf/LibLinearDataset.java:592-614), so no kernel special-cases it.
struct Problem {
  // data (shared by the L problems of one partition)
  const float* X;          // dense [n][ldx] fp32, or nullptr for CSR
  long long n;             // rows
  int ldx;                 // leading dim in floats (multiple of 4)
  int Dt;                  // columns incl. bias
  const signed char* y;    // +1 / -1
  const float* w;          // weight
  const float* o;          // offset
  const long long* rowptr; // CSR (bias NOT stored; handled by the kernels)
  const int* colidx;
  const float* vals;
  long long nnz_hint;      // CSR nnz (host-side accounting only)
  int csr_unique;          // every CSR row has strictly increasing column ids (parallel bf16 emit is exact)
  const long long* bm_offs;       // block-major entry list for the CSR Gram: run offsets [nblk128][bm_groups] (+1 total)
  const unsigned short* bm_keys;  // per entry: byte offset inside the swizzled [32 rows][128 cols] operand block
  const float* bm_vals;           // per entry: the stored value
  long long bm_groups;            // number of 32-row groups
  float vmax, wmax;               // max |stored value| and max record weight of the partition (fixed-point scale of the CSR K1)
  int nblk128;             // number of 128-column blocks (Dp / 128)
  // fused multi-lambda CSR K1 (k1_csr_fused.cu): the partition's rows cut into sg_S segments of sg_rows rows; per segment the
  // stored values regrouped by column: 32 columns (lanes) per group, groups of columns of similar length, entries [k][lane]
  int sg_S, sg_rows, sg_ngrp;
  const int* sg_perm;               // [sg_S][sg_ngrp*32] column id of each lane slot, -1 = unused slot
  const int* sg_depth;              // [sg_S][sg_ngrp] entries per lane of the group
  const long long* sg_goff;         // [sg_S][sg_ngrp] first 32-lane row of the group in sg_row16 / sg_val
  const unsigned short* sg_row16;   // [..][32] row inside the segment
  const float* sg_val;              // [..][32] value (0 in padding slots)
  float* gpart_f;                   // [sg_S][ldx] per-segment partial gradients when the fused K1 runs (else NULL; gpart is used)
  float* sdvec;            // [n] sqrt(d_i) written by K1 when the Gram is assembled straight from CSR (no Xt)
  float* rvec;             // [n] row residuals r_i, only for CSR partitions wider than one K1 column window (else NULL)
  int gram_from_csr;       // 1: gram_csr_tcgen05_kernel builds the operand tiles in shared memory from the sparse rows
  float gram_scale;        // CSR Gram operands are e4m3: sqrt(d) x is multiplied by this power of two before rounding ...
  float gram_unscale;      // ... and the Gram sums by 1 / gram_scale^2 in chol_prep (1 for the bf16 dense-operand path)
  __nv_bfloat16* Xt;       // [n][Dp] bf16 = sqrt(d_i) * x_ij  (Gram operand), zero in [ldx, Dp)
  int Dp;                  // multiple of 128
  // solver state
  double* beta;            // accepted iterate
  double* beta_t;          // trial iterate
  float* beta_tf;          // float copy of the trial iterate (what K1 reads)
  double* m;               // prior mean  (z - u)
  double* q;               // prior precision 1/priorVar (rho for ADMM)
  double* g_t;             // gradient at trial
  double* g_acc;           // gradient at accepted
  double* dir;             // Newton direction
  double* gpart;           // [k1_ctas][ldx] per-CTA partial X^T r
  double* fpart;           // [k1_ctas] per-CTA partial loss
  int k1_ctas;
  float* Hpart;            // [gram_slices][Dp][Dp] split-K partial Gram (lower tiles)
  int gram_slices;
  double* Lc;              // [ldh][ldh] Cholesky factor (lower), ldh multiple of 32
  double* Ldiag;           // [ldh][32] factorised diagonal blocks (side buffer, see k3_cholesky.cu)
  double* Ldinv;           // [ldh][32] inverses of the diagonal blocks (lower triangular)
  double* Yinv;            // [ldh][ldh] L^-1 (lower)
  double* Hinv;            // [ldh][ldh] (L L^T)^-1, full symmetric: a Newton direction is one GEMV
  __nv_bfloat16* Ysym;    // wide systems (ldh > 2048; NULL otherwise): operand of the direction product.  It holds Y = L^-1 as bf16 in
                          // symmetric storage M[i][j] = Y[max(i,j)][min(i,j)] (k3_cholesky.cu ysym_kernel): H^-1 q ~ Y^T (Y q) is two
                          // row-wise triangular GEMVs over it, HBM-bound on D'^2 2-byte entries in total.  The product form is
                          // symmetric positive definite for ANY rounding of Y, so the low precision can never turn the preconditioner
                          // indefinite (a rounded explicit H^-1 could)
  float* qf;              // [ldx] fp32 copy of the two-loop vector q (written by the decide kernel when Ysym is in use)
  float* tf;              // [ldx] t = Y q in fp32 (between the two phases)
  int ldh;
  Ctrl* ctrl;
  // ADMM per-problem vectors (float, as the reference's avro files hold them)
  float* u_f;              // u used by this iteration
  float* uplusx_f;         // float(u + x)
  float* x_f;              // float(x)
  double* bfgs_S;          // [BFGS_M][ldx] steps  s_k = beta_{k+1} - beta_k
  double* bfgs_Y;          // [BFGS_M][ldx] gradient differences y_k
  double* bfgs_rho;        // [BFGS_M] 1/(s.y)
  double* bfgs_alpha;      // [BFGS_M] two-loop scratch
  double* x_d;             // x of the last x-update (the ADMM consensus overwrites beta with the next init)
  int lambda_idx;
  int self_idx;            // index of this problem in its batch (tensor-map slot), valid also in compacted copies
  int part_local;
};

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// Byte store to a 32-bit shared-space address.  A pointer derived from the dynamic shared array by integer alignment loses its
// address space: the compiler then emits GENERIC stores and rebuilds the 64-bit window base (S2UR CgaCtaId / SWINHI, ~10
// instructions) at every store -- the Gram producers' scatter stores spent more instructions on that than on the data.
__device__ __forceinline__ void sts_u8(uint32_t saddr, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(saddr), "r"(v) : "memory"); }
// 1-D bulk copy global -> shared (TMA engine, no tensor map): SASS UBLKCP.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// 2-D tensor-map TMA load: SASS UTMALDG.
__device__ __forceinline__ void tma_load_2d(void* dst_smem, const void* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst_smem)),
      "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}

// tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (bf16/fp16 inputs, fp32 accumulate): SASS UTCHMMA.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// ---- CTA pair (cta_group::2): two CTAs of a cluster, on the two SMs of a TPC, run one M=256 MMA; each supplies its 128 rows of A
// and its half of B's N columns from its own shared memory at the SAME offsets; only the leader (cluster rank 0) issues.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared-memory object of this CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa_u32(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// Arrive on a barrier of another CTA of the cluster.  Default semantics (.release.cta), as CUTLASS's ClusterBarrier::arrive(cta_id):
// the .release.cluster form compiles to MEMBAR.ALL.GPU + ERRBAR, which waits for EVERY outstanding global load of the warp (the
// producers' prefetches) -- 26 % of all stall samples in the first CTA-pair Gram.  The data handed over is shared memory this warp
// wrote and already fenced for the async proxy (fence.proxy.async) before the arrive.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc] over the pair, kind::f8f6f4 (e4m3 / e5m2 inputs, fp32 accumulate, K = 32 per instruction)
__device__ __forceinline__ void umma_f8_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at this offset in BOTH CTAs of the pair when the leader's previously issued MMAs have completed
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  const unsigned short mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (SASS LDTM).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// warp / block reductions
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace mlease
