// k3_cholesky.cu -- K3: H = sum of split-K Gram partials + diag(q), blocked right-looking Cholesky
// in fp64, batched over problems (blockIdx.y / z).  The triangular solves live in newton.cu.
//
// No direct reference equivalent on the ADMM path (TRON is matrix-free, bw/Tron.java:126-179);
// the only Cholesky in the reference is commons-math's at llf/LibLinear.java:321-325 (posterior
// covariance).  H itself is LogisticRegressionL2.hessian (llf/LogisticRegressionL2.java:258-297).
//
// fp64 on purpose: the Gram comes from bf16 tensor-core products, but the factorisation must not
// break down when cond(H) approaches 1/eps_fp32; 3.3e8 flop at D'=1001 is latency- not
// throughput-bound on B200's fp64 pipe.
#include <algorithm>

#include "kernels.cuh"

namespace mlease {

constexpr int NB = 32;   // panel width
constexpr int TB = 64;   // trailing-update tile

// Hd (lower incl. diagonal) = sum_s Hpart[s] + diag(q); padded rows/cols (>= Dt) = identity.
__global__ void chol_prep_kernel(const Problem* __restrict__ probs, int share) {
  const Problem& pb = probs[blockIdx.z];
  // share = L > 1: the Gram partials of the group's first problem stand for the whole group (see gram_tcgen05_kernel)
  const float* __restrict__ hpart = share > 1 ? probs[blockIdx.z - blockIdx.z % share].Hpart : pb.Hpart;
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  const int ldh = pb.ldh, Dt = pb.Dt, Dp = pb.Dp, S = pb.gram_slices;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ldh || j >= ldh || j > i) return;
  double v;
  if (i < Dt) {
    double s = 0.0;
    const size_t off = (size_t)i * Dp + j;
    for (int t = 0; t < S; t++) s += (double)hpart[(size_t)t * Dp * Dp + off];
    s *= (double)pb.gram_unscale;   // e4m3 operands of the CSR Gram carry a power-of-two scale
    if (i == j) s += pb.q[i];
    v = s;
  } else {
    v = (i == j) ? 1.0 : 0.0;
  }
  pb.Lc[(size_t)i * ldh + j] = v;
}

// Panel step k, part 1: ONE warp per problem factorises the NBxNB diagonal block in registers and inverts it.
// lane i holds row i; column j is scaled by lane-j's pivot and every L[kk][j] reaches the other rows by shuffle: ~500 double
// shuffles + FMAs (a few microseconds) instead of 32 rounds of block-wide barriers.  This kernel and the two below are one link
// of a chain of ldh/32 dependent steps: latency is what counts.  The factor and its inverse go to the side buffers Ldiag / Ldinv
// (chol_finish_kernel copies the diagonal blocks back into Lc).
constexpr int RB = 64;
__global__ void __launch_bounds__(32) chol_diag_kernel(const Problem* __restrict__ probs, int k) {
  const Problem& pb = probs[blockIdx.x];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  __shared__ double A[NB][NB + 1];
  const int ldh = pb.ldh;
  const int c0 = k * NB;
  const double* H = pb.Lc;
  const int lane = threadIdx.x;
  double a[NB];
#pragma unroll
  for (int kk = 0; kk < NB; kk++) a[kk] = (kk <= lane) ? H[(size_t)(c0 + lane) * ldh + c0 + kk] : 0.0;
  int bad = 0;
  double dinv[NB];   // 1 / L[j][j]: one rsqrt per pivot serves the column scaling here and the substitution below (no divisions)
#pragma unroll
  for (int j = 0; j < NB; j++) {
    double djj = __shfl_sync(0xffffffffu, a[j], j);
    if (!(djj > 0.0)) { bad = 1; djj = 1.0; }
    const double r = rsqrt(djj);
    dinv[j] = r;
    if (lane == j) a[j] = djj * r;
    else if (lane > j) a[j] = a[j] * r;
#pragma unroll
    for (int kk = j + 1; kk < NB; kk++) {
      const double lkj = __shfl_sync(0xffffffffu, a[j], kk);
      if (lane >= kk) a[kk] -= a[j] * lkj;
    }
  }
#pragma unroll
  for (int kk = 0; kk < NB; kk++) {
    A[lane][kk] = (kk <= lane) ? a[kk] : 0.0;
    pb.Ldiag[(size_t)(c0 + lane) * NB + kk] = (kk <= lane) ? a[kk] : 0.0;
  }
  __syncwarp();
  // inverse of the lower-triangular factor: lane cc solves column cc by forward substitution (A is read as a broadcast)
  {
    const int cc = lane;
    double li[NB];
#pragma unroll
    for (int i = 0; i < NB; i++) {
      double sacc = 0.0;
#pragma unroll
      for (int kk = 0; kk < NB; kk++)
        if (kk < i) sacc += A[i][kk] * li[kk];     // li[kk] = 0 for kk < cc
      li[i] = i < cc ? 0.0 : (i == cc ? dinv[i] : -sacc * dinv[i]);
    }
#pragma unroll
    for (int i = 0; i < NB; i++) pb.Ldinv[(size_t)(c0 + i) * NB + cc] = li[i];
  }
  if (lane == 0 && bad) c->fail = 1;
}

// Panel step k, part 2: rows of L21 = A21 * L11^-T, RB rows per CTA, with the inverse of the diagonal block from Ldinv.
__global__ void __launch_bounds__(256) chol_panel_kernel(const Problem* __restrict__ probs, int k) {
  const Problem& pb = probs[blockIdx.y];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  __shared__ double Li[NB][NB + 1];
  __shared__ double P[RB][NB + 1];
  const int ldh = pb.ldh;
  const int c0 = k * NB;
  double* H = pb.Lc;
  const int tid = threadIdx.x;
  const int r0 = c0 + NB + blockIdx.x * RB;
  if (r0 >= ldh) return;
  const int rows = min(RB, ldh - r0);
  for (int e = tid; e < NB * NB; e += 256) Li[e / NB][e % NB] = pb.Ldinv[(size_t)(c0 + e / NB) * NB + e % NB];
  for (int e = tid; e < rows * NB; e += 256) {
    const int i = e / NB, j = e % NB;
    P[i][j] = H[(size_t)(r0 + i) * ldh + c0 + j];
  }
  __syncthreads();
  for (int e = tid; e < rows * NB; e += 256) {
    const int i = e / NB, j = e % NB;
    double sacc = 0.0;
    for (int kk = 0; kk <= j; kk++) sacc += P[i][kk] * Li[j][kk];   // (A21 * L11^-T)[i][j]
    H[(size_t)(r0 + i) * ldh + c0 + j] = sacc;
  }
}

// Trailing update A22 -= L21 L21^T on lower-triangular TBxTB tiles.
__global__ void __launch_bounds__(256) chol_update_kernel(const Problem* __restrict__ probs, int k, int jlimit) {
  const Problem& pb = probs[blockIdx.z];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  if (blockIdx.x > blockIdx.y) return;  // lower tiles only (x = tile col, y = tile row)
  const int ldh = pb.ldh;
  const int base = (k + 1) * NB;
  const int i0 = base + blockIdx.y * TB, j0 = base + blockIdx.x * TB;
  if (i0 >= ldh || j0 >= ldh || j0 >= jlimit) return;   // jlimit: the wide path only updates inside its outer panel
  __shared__ double Ai[NB][TB + 2];   // [k][row]: a thread's 4 rows are contiguous -> conflict-light vector reads
  __shared__ double Aj[NB][TB + 2];
  double* H = pb.Lc;
  const int c0 = k * NB;
  const int tid = threadIdx.x;
  for (int e = tid; e < TB * NB; e += 256) {
    const int i = e / NB, kk = e % NB;
    Ai[kk][i] = (i0 + i < ldh) ? H[(size_t)(i0 + i) * ldh + c0 + kk] : 0.0;
    Aj[kk][i] = (j0 + i < ldh) ? H[(size_t)(j0 + i) * ldh + c0 + kk] : 0.0;
  }
  __syncthreads();
  const int ti = (tid / 16) * 4, tj = (tid % 16) * 4;
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
#pragma unroll 4
  for (int kk = 0; kk < NB; kk++) {
    double x[4], y[4];
#pragma unroll
    for (int a = 0; a < 4; a++) { x[a] = Ai[kk][ti + a]; y[a] = Aj[kk][tj + a]; }
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) acc[a][b] += x[a] * y[b];
  }
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++) {
      const int i = i0 + ti + a, j = j0 + tj + b;
      if (i < ldh && j <= i && j < jlimit) H[(size_t)i * ldh + j] -= acc[a][b];
    }
}

__global__ void chol_finish_kernel(const Problem* __restrict__ probs) {
  const Problem& pb = probs[blockIdx.y];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  const int c0 = blockIdx.x * NB;
  for (int e = threadIdx.x; e < NB * NB; e += blockDim.x) {
    const int i = e / NB, j = e % NB;
    if (j <= i) pb.Lc[(size_t)(c0 + i) * pb.ldh + c0 + j] = pb.Ldiag[(size_t)(c0 + i) * NB + j];
  }
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (c->fail == 1) { c->done = 1; c->hess_valid = 0; }
    else { c->hess_valid = 1; c->hess_builds++; c->tot_hess++; c->bfgs_count = 0; c->h0_scale = 1.0; c->build_step = c->newton_steps; c->ysym_use = pb.Ysym; }
  }
}

// ------------------------------------------------------------------------------------------
// Explicit inverse, built once per factorisation so that every chord-Newton direction afterwards is a
// single multi-CTA GEMV instead of two latency-bound triangular solves:
//   Y = L^-1    : forward substitution with 64 right-hand sides (columns of I) per CTA, tiles staged through shared
//                 memory, diagonal blocks applied through their stored inverses
//   Hinv = Y^T Y: 64x64 tiles, both triangles written
// ------------------------------------------------------------------------------------------
// Y = L^-1 by blocked forward substitution, one CTA per NR columns of Y.  Row block kb of those columns is
//   Y[kb] = Ldinv[kb] * ( I[kb] - sum_{jb<kb} L[kb][jb] * Y[jb] )
// with 32x32 tiles of L and 32xNR tiles of the already computed Y (read back from global memory / L2, so the column
// count per CTA is not bounded by shared memory: D' = 10k works the same way as D' = 1k).  The next pair of tiles is
// prefetched into registers while the current pair is multiplied.  Thread (ti, tq) owns row ti and the NR/8 columns
// tq, tq+8, tq+16, ... : for a fixed k the 8 lanes of a row read 8 consecutive doubles (no bank conflicts).
template <int NR>
__global__ void __launch_bounds__(256) trinv_kernel(const Problem* __restrict__ probs, int leaf) {
  const Problem& pb = probs[blockIdx.y];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  constexpr int CPT = NR / 8;   // columns per thread
  __shared__ double Lt[NB][NB + 1];
  __shared__ double Yt[NB][NR + 2];
  __shared__ double Rb[NB][NR + 2];
  const int ldh = pb.ldh;
  const int c0 = blockIdx.x * NR;
  if (c0 >= ldh) return;
  // leaf > 0: invert only the diagonal leaf x leaf block this column group lies in (the wide path merges leaves with GEMMs)
  const int nb = leaf > 0 ? min(ldh, (c0 / leaf + 1) * leaf) / NB : ldh / NB;
  const int ncols = min(NR, ldh - c0);
  const int kb0 = c0 / NB;
  const int tid = threadIdx.x;
  const int ti = tid >> 3, tq = tid & 7;
  const double* __restrict__ L = pb.Lc;
  double* __restrict__ Y = pb.Yinv;
  const int lr = tid >> 3, lc = (tid & 7) * 4;   // Lt 32x32: 4 consecutive doubles per thread
  for (int kb = kb0; kb < nb; kb++) {
    const int r0 = kb * NB;
    double acc[CPT];
#pragma unroll
    for (int q = 0; q < CPT; q++) acc[q] = (r0 + ti == c0 + tq + 8 * q) ? 1.0 : 0.0;
    double pl[4], py[CPT];
    auto prefetch = [&](int jb) {
#pragma unroll
      for (int q = 0; q < 4; q++) pl[q] = L[(size_t)(r0 + lr) * ldh + jb * NB + lc + q];
#pragma unroll
      for (int q = 0; q < CPT; q++) py[q] = (tq + 8 * q < ncols) ? Y[(size_t)(jb * NB + ti) * ldh + c0 + tq + 8 * q] : 0.0;
    };
    if (kb > kb0) prefetch(kb0);
    for (int jb = kb0; jb < kb; jb++) {
#pragma unroll
      for (int q = 0; q < 4; q++) Lt[lr][lc + q] = pl[q];
#pragma unroll
      for (int q = 0; q < CPT; q++) Yt[ti][tq + 8 * q] = py[q];
      __syncthreads();
      if (jb + 1 < kb) prefetch(jb + 1);
#pragma unroll 8
      for (int kk = 0; kk < NB; kk++) {
        const double l = Lt[ti][kk];
#pragma unroll
        for (int q = 0; q < CPT; q++) acc[q] -= l * Yt[kk][tq + 8 * q];
      }
      __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < CPT; q++) Rb[ti][tq + 8 * q] = acc[q];
#pragma unroll
    for (int q = 0; q < 4; q++) Lt[lr][lc + q] = pb.Ldinv[(size_t)(r0 + lr) * NB + lc + q];
    __syncthreads();
    double yv[CPT];
#pragma unroll
    for (int q = 0; q < CPT; q++) yv[q] = 0.0;
    for (int kk = 0; kk <= ti; kk++) {
      const double l = Lt[ti][kk];
#pragma unroll
      for (int q = 0; q < CPT; q++) yv[q] += l * Rb[kk][tq + 8 * q];
    }
#pragma unroll
    for (int q = 0; q < CPT; q++)
      if (tq + 8 * q < ncols) Y[(size_t)(r0 + ti) * ldh + c0 + tq + 8 * q] = yv[q];
    __syncthreads();   // the Y block just written is read back (by other threads of this CTA) for the next row blocks
  }
}

__global__ void __launch_bounds__(256) hinv_syrk_kernel(const Problem* __restrict__ probs) {
  const Problem& pb = probs[blockIdx.z];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  if (blockIdx.x > blockIdx.y) return;
  const int ldh = pb.ldh;
  const int i0 = blockIdx.y * TB, j0 = blockIdx.x * TB;   // i0 >= j0
  if (i0 >= ldh) return;
  __shared__ double Yi[NB][TB + 1];
  __shared__ double Yj[NB][TB + 1];
  const double* Y = pb.Yinv;
  const int tid = threadIdx.x;
  const int ti = (tid / 16) * 4, tj = (tid % 16) * 4;
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
  // Y is lower triangular: Y[k][i] != 0 only for k >= i, so start at the row block of i0 (>= j0)
  for (int k0 = (i0 / NB) * NB; k0 < ldh; k0 += NB) {
    for (int e = tid; e < NB * TB; e += 256) {
      const int kk = e / TB, cc = e % TB;
      const int k = k0 + kk;
      Yi[kk][cc] = (i0 + cc < ldh && i0 + cc <= k) ? Y[(size_t)k * ldh + i0 + cc] : 0.0;
      Yj[kk][cc] = (j0 + cc < ldh && j0 + cc <= k) ? Y[(size_t)k * ldh + j0 + cc] : 0.0;
    }
    __syncthreads();
#pragma unroll 4
    for (int kk = 0; kk < NB; kk++) {
      double x[4], y[4];
#pragma unroll
      for (int a = 0; a < 4; a++) { x[a] = Yi[kk][ti + a]; y[a] = Yj[kk][tj + a]; }
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] += x[a] * y[b];
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++) {
      const int i = i0 + ti + a, j = j0 + tj + b;
      if (i < ldh && j < ldh) {
        pb.Hinv[(size_t)i * ldh + j] = acc[a][b];
        pb.Hinv[(size_t)j * ldh + i] = acc[a][b];
      }
    }
}


// ------------------------------------------------------------------------------------------
// Wide systems (ldh > 1000): the same factorisation / inverse / product, restructured so that almost all flops are
// fp64 tensor-core GEMMs (DMMA m8n8k4) on 128x64 tiles with K chunks of 16 staged through shared memory:
//   Cholesky : outer panels of WNB columns; inside a panel the NB=32 steps above (panel kernel + K=32 updates limited
//              to the panel's columns), then one K=WNB trailing update             C -= A A^T      (mode 0)
//   Y = L^-1 : leaves of WLEAF columns by trinv_kernel, then pairwise merges bottom-up
//              T = L21 * Y11 (mode 1, T in the Hinv buffer), Y21 = -Y22 * T          (mode 2)
//   Hinv     : Y^T Y over k >= max(i, j)                                            (mode 3)
// Operand tiles live in shared memory either [row][k] (stride 20) or [k][row] (stride tile+4), whichever matches the
// contiguous direction in global memory; both strides are = 4 mod 16 doubles, which makes the DMMA fragment loads
// (thread t: row t/4, k t%4) bank-conflict free.
// ------------------------------------------------------------------------------------------
constexpr int WNB = 256;     // outer panel width of the wide Cholesky
constexpr int WLEAF = 256;   // leaf size of the recursive inverse
constexpr int DM = 128, DN = 64, DK = 16;
constexpr int DA_SZ = DM * 20 > DK * (DM + 4) ? DM * 20 : DK * (DM + 4);   // doubles per A stage
constexpr int DB_SZ = DN * 20 > DK * (DN + 4) ? DN * 20 : DK * (DN + 4);
constexpr size_t DGEMM_SMEM = (size_t)2 * (DA_SZ + DB_SZ) * sizeof(double);

__device__ __forceinline__ void dmma_8x8x4(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(256, 2) dgemm_kernel(const Problem* __restrict__ probs, int mode, int p0, int p1) {
  const Problem& pb = probs[blockIdx.z];
  Ctrl* ctl = pb.ctrl;
  if (ctl->done || !ctl->need_hess) return;
  const int ldh = pb.ldh;
  const double* A; const double* B; double* C;
  int M, N, K;
  if (mode == 0) {            // trailing update after the outer panel at column p0 of width p1
    const int c = p0, w = p1;
    M = N = ldh - c - w; K = w;
    A = B = pb.Lc + (size_t)(c + w) * ldh + c;
    C = pb.Lc + (size_t)(c + w) * ldh + (c + w);
  } else if (mode == 1 || mode == 2) {   // merge of the diagonal blocks [r0, r0+m) and [r0+m, r0+m+m2)
    const int m = p0, r0 = 2 * blockIdx.y * m;
    const int m2 = min(m, ldh - r0 - m);
    if (m2 <= 0) return;
    M = m2; N = m;
    if (mode == 1) {
      K = m;
      A = pb.Lc + (size_t)(r0 + m) * ldh + r0;
      B = pb.Yinv + (size_t)r0 * ldh + r0;
      C = pb.Hinv + (size_t)(r0 + m) * ldh + r0;
    } else {
      K = m2;
      A = pb.Yinv + (size_t)(r0 + m) * ldh + (r0 + m);
      B = pb.Hinv + (size_t)(r0 + m) * ldh + r0;
      C = pb.Yinv + (size_t)(r0 + m) * ldh + r0;
    }
  } else {
    M = N = K = ldh;
    A = B = pb.Yinv;
    C = pb.Hinv;
  }
  const int tiles_n = (N + DN - 1) / DN;
  const int i0 = (blockIdx.x / tiles_n) * DM, j0 = (blockIdx.x % tiles_n) * DN;
  if (i0 >= M) return;
  if ((mode == 0 || mode == 3) && j0 >= i0 + DM) return;   // strictly upper tile of a symmetric result
  int klo = 0, khi = K;
  if (mode == 1) klo = j0;                      // Y11 is lower triangular: Y11[k][j] = 0 for k < j
  if (mode == 2) khi = min(K, i0 + DM);         // Y22 is lower triangular: Y22[i][k] = 0 for k > i
  if (mode == 3) klo = max(i0, j0);             // Y[k][i] = 0 for k < i

  extern __shared__ double dg_smem[];
  double* As = dg_smem;                 // [2][DA_SZ]
  double* Bs = dg_smem + 2 * DA_SZ;     // [2][DB_SZ]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, tg = lane & 3;
  const int wm = (warp & 3) * 32, wn = (warp >> 2) * 32;

  double2 ra[4], rb[2];
  auto gload = [&](int k0) {
#pragma unroll
    for (int q = 0; q < 4; q++) {
      if (A_KC) {
        const int row = (tid >> 3) + 32 * q, kk = (tid & 7) * 2;
        ra[q] = (i0 + row < M) ? *reinterpret_cast<const double2*>(A + (size_t)(i0 + row) * ldh + k0 + kk) : make_double2(0.0, 0.0);
      } else {
        const int kk = (tid >> 6) + 4 * q, ii = (tid & 63) * 2;
        ra[q] = (i0 + ii < M) ? *reinterpret_cast<const double2*>(A + (size_t)(k0 + kk) * ldh + i0 + ii) : make_double2(0.0, 0.0);
      }
    }
#pragma unroll
    for (int q = 0; q < 2; q++) {
      if (B_KC) {
        const int col = (tid >> 3) + 32 * q, kk = (tid & 7) * 2;
        rb[q] = (j0 + col < N) ? *reinterpret_cast<const double2*>(B + (size_t)(j0 + col) * ldh + k0 + kk) : make_double2(0.0, 0.0);
      } else {
        const int kk = (tid >> 5) + 8 * q, jj = (tid & 31) * 2;
        rb[q] = (j0 + jj < N) ? *reinterpret_cast<const double2*>(B + (size_t)(k0 + kk) * ldh + j0 + jj) : make_double2(0.0, 0.0);
      }
    }
  };
  auto sstore = [&](int buf) {
    double* a = As + buf * DA_SZ;
    double* b = Bs + buf * DB_SZ;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      if (A_KC) *reinterpret_cast<double2*>(a + ((tid >> 3) + 32 * q) * 20 + (tid & 7) * 2) = ra[q];
      else *reinterpret_cast<double2*>(a + ((tid >> 6) + 4 * q) * (DM + 4) + (tid & 63) * 2) = ra[q];
    }
#pragma unroll
    for (int q = 0; q < 2; q++) {
      if (B_KC) *reinterpret_cast<double2*>(b + ((tid >> 3) + 32 * q) * 20 + (tid & 7) * 2) = rb[q];
      else *reinterpret_cast<double2*>(b + ((tid >> 5) + 8 * q) * (DN + 4) + (tid & 31) * 2) = rb[q];
    }
  };

  double acc[4][4][2];
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;

  if (klo < khi) {
    gload(klo);
    sstore(0);
    __syncthreads();
    int buf = 0;
    for (int k0 = klo; k0 < khi; k0 += DK) {
      const bool more = k0 + DK < khi;
      if (more) gload(k0 + DK);
      const double* a = As + buf * DA_SZ;
      const double* b = Bs + buf * DB_SZ;
#pragma unroll
      for (int k4 = 0; k4 < DK; k4 += 4) {
        double fa[4], fb[4];
#pragma unroll
        for (int f = 0; f < 4; f++) {
          fa[f] = A_KC ? a[(wm + f * 8 + g) * 20 + k4 + tg] : a[(k4 + tg) * (DM + 4) + wm + f * 8 + g];
          fb[f] = B_KC ? b[(wn + f * 8 + g) * 20 + k4 + tg] : b[(k4 + tg) * (DN + 4) + wn + f * 8 + g];
        }
#pragma unroll
        for (int fm = 0; fm < 4; fm++)
#pragma unroll
          for (int fn = 0; fn < 4; fn++) dmma_8x8x4(acc[fm][fn][0], acc[fm][fn][1], fa[fm], fb[fn]);
      }
      if (more) sstore(buf ^ 1);
      __syncthreads();
      buf ^= 1;
    }
  }

#pragma unroll
  for (int fm = 0; fm < 4; fm++) {
    const int i = i0 + wm + fm * 8 + g;
    if (i >= M) continue;
#pragma unroll
    for (int fn = 0; fn < 4; fn++) {
      const int j = j0 + wn + fn * 8 + 2 * tg;
      if (j >= N) continue;
      const double v0 = acc[fm][fn][0], v1 = acc[fm][fn][1];
      if (mode == 0) {
        double* d = C + (size_t)i * ldh + j;
        if (j + 1 <= i) { double2 o = *reinterpret_cast<double2*>(d); o.x -= v0; o.y -= v1; *reinterpret_cast<double2*>(d) = o; }
        else if (j <= i) d[0] -= v0;
      } else if (mode == 1) {
        *reinterpret_cast<double2*>(C + (size_t)i * ldh + j) = make_double2(v0, v1);
      } else if (mode == 2) {
        *reinterpret_cast<double2*>(C + (size_t)i * ldh + j) = make_double2(-v0, -v1);
      } else {
        if (j <= i) { C[(size_t)i * ldh + j] = v0; C[(size_t)j * ldh + i] = v0; }
        if (j + 1 <= i) { C[(size_t)i * ldh + j + 1] = v1; C[(size_t)(j + 1) * ldh + i] = v1; }
      }
    }
  }
}

template <bool A_KC, bool B_KC>
static cudaError_t dgemm_launch(const Problem* d_probs, int nprob, int mode, int p0, int p1, int M, int N, int nmerge, cudaStream_t st,
                                int* launches) {
  {
    // the attribute is per device: set it once for every device this process launches on
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
      cudaError_t e = cudaFuncSetAttribute(dgemm_kernel<A_KC, B_KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DGEMM_SMEM);
      if (e != cudaSuccess) return e;
      if (dev >= 0 && dev < 64) configured[dev] = true;
    }
  }
  const int tiles = ((M + DM - 1) / DM) * ((N + DN - 1) / DN);
  if (tiles <= 0 || nmerge <= 0) return cudaSuccess;
  dgemm_kernel<A_KC, B_KC><<<dim3(tiles, nmerge, nprob), 256, DGEMM_SMEM, st>>>(d_probs, mode, p0, p1);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Merges of the inverse in TF32 (wide systems whose direction runs on the factored form, ysym_kernel below).
// There Y = L^-1 is only ever read after rounding to bf16, and Y^T Y is SPD for ANY Y, so an inexact inverse cannot turn the
// preconditioner indefinite (the factorisation itself -- pivots -- stays in fp64).  The two GEMMs of a merge,
//   T = L21 * Y11 (mode 1)   and   Y21 = -Y22 * T (mode 2),
// are half of the D'^3 flops of a 10k-wide factorisation and run at ~25 TFLOP/s on the fp64 pipe; here the fp64 operands
// are rounded to tf32 on their way into shared memory (cvt.rna) and multiplied by mma.sync.m16n8k8 with fp32 accumulation:
// operand rounding 2^-11, against 2^-8 of the bf16 storage the result ends up in.  128x128 tiles, K chunks of 16, the same
// register-staged double buffer as dgemm_kernel; both operands are row-major (A[i][k], B[k][j]) as in dgemm_kernel<true,false>.
// Shared-memory strides: A rows of 20 words (fragment loads (row g, k tg): bank 20 g + tg, all distinct), B rows of 136
// words (fragment loads (k tg, col g): bank 8 tg + g, all distinct).
// ------------------------------------------------------------------------------------------
constexpr int TM = 128, TN = 128, TK = 16;
constexpr int TA_LD = TK + 4, TB_LD = TN + 8;
constexpr int TA_SZ = TM * TA_LD, TB_SZ = TK * TB_LD;   // 32-bit words per stage

__device__ __forceinline__ uint32_t to_tf32(double x) {
  uint32_t r;
  const float f = (float)x;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(f));
  return r;
}
__device__ __forceinline__ void mma_tf32_16x8x8(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__global__ void __launch_bounds__(256, 2) merge_tf32_kernel(const Problem* __restrict__ probs, int mode, int m) {
  const Problem& pb = probs[blockIdx.z];
  Ctrl* ctl = pb.ctrl;
  if (ctl->done || !ctl->need_hess) return;
  const int ldh = pb.ldh;
  // merge of the diagonal blocks [r0, r0+m) and [r0+m, r0+m+m2), exactly as dgemm_kernel modes 1 / 2
  const int r0 = 2 * blockIdx.y * m;
  const int m2 = min(m, ldh - r0 - m);
  if (m2 <= 0) return;
  const int M = m2, N = m;
  const double* __restrict__ A; const double* __restrict__ B; double* __restrict__ C;
  int K;
  if (mode == 1) {
    K = m;
    A = pb.Lc + (size_t)(r0 + m) * ldh + r0;
    B = pb.Yinv + (size_t)r0 * ldh + r0;
    C = pb.Hinv + (size_t)(r0 + m) * ldh + r0;
  } else {
    K = m2;
    A = pb.Yinv + (size_t)(r0 + m) * ldh + (r0 + m);
    B = pb.Hinv + (size_t)(r0 + m) * ldh + r0;
    C = pb.Yinv + (size_t)(r0 + m) * ldh + r0;
  }
  const int tiles_n = (N + TN - 1) / TN;
  const int i0 = (blockIdx.x / tiles_n) * TM, j0 = (blockIdx.x % tiles_n) * TN;
  if (i0 >= M) return;
  int klo = 0, khi = K;
  if (mode == 1) klo = j0;                 // Y11 is lower triangular: Y11[k][j] = 0 for k < j
  else khi = min(K, i0 + TM);              // Y22 is lower triangular: Y22[i][k] = 0 for k > i

  __shared__ __align__(16) uint32_t As[2][TA_SZ];
  __shared__ __align__(16) uint32_t Bs[2][TB_SZ];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, tg = lane & 3;
  const int wm = (warp & 1) * 64, wn = (warp >> 1) * 32;   // 2 x 4 warps, 64 x 32 per warp

  // global -> register staging: thread t fetches rows (t >> 3) + 32 q of A (two consecutive k) and k-rows (t >> 6) + 4 q of B
  // (two consecutive columns); the pointers walk along k, the row guards are loop-invariant.  Neither operand is written by
  // this launch (C is a different block of the buffers), so the read-only path is safe.
  const double* pa = A + (size_t)(i0 + (tid >> 3)) * ldh + klo + (tid & 7) * 2;
  const double* pbk = B + (size_t)(klo + (tid >> 6)) * ldh + j0 + (tid & 63) * 2;
  const size_t a_step = (size_t)32 * ldh, b_step = (size_t)4 * ldh, b_adv = (size_t)TK * ldh;
  unsigned a_ok = 0;
#pragma unroll
  for (int q = 0; q < 4; q++) a_ok |= (i0 + (tid >> 3) + 32 * q < M ? 1u : 0u) << q;
  const bool b_ok = j0 + (tid & 63) * 2 < N;
  double2 ra[4], rb[4];
  auto gload = [&]() {   // the next K chunk
#pragma unroll
    for (int q = 0; q < 4; q++)
      ra[q] = ((a_ok >> q) & 1u) ? __ldg(reinterpret_cast<const double2*>(pa + q * a_step)) : make_double2(0.0, 0.0);
#pragma unroll
    for (int q = 0; q < 4; q++)
      rb[q] = b_ok ? __ldg(reinterpret_cast<const double2*>(pbk + q * b_step)) : make_double2(0.0, 0.0);
    pa += TK;
    pbk += b_adv;
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int row = (tid >> 3) + 32 * q, kk = (tid & 7) * 2;
      *reinterpret_cast<uint2*>(&As[buf][row * TA_LD + kk]) = make_uint2(to_tf32(ra[q].x), to_tf32(ra[q].y));
    }
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int kk = (tid >> 6) + 4 * q, jj = (tid & 63) * 2;
      *reinterpret_cast<uint2*>(&Bs[buf][kk * TB_LD + jj]) = make_uint2(to_tf32(rb[q].x), to_tf32(rb[q].y));
    }
  };

  float acc[4][4][4];
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++)
#pragma unroll
      for (int e = 0; e < 4; e++) acc[a][b][e] = 0.f;

  if (klo < khi) {
    gload();
    sstore(0);
    __syncthreads();
    int buf = 0;
    for (int k0 = klo; k0 < khi; k0 += TK) {
      const bool more = k0 + TK < khi;
      if (more) gload();
      const uint32_t* a = As[buf];
      const uint32_t* b = Bs[buf];
#pragma unroll
      for (int k8 = 0; k8 < TK; k8 += 8) {
        uint32_t fa[4][4], fb[4][2];
#pragma unroll
        for (int f = 0; f < 4; f++) {
          const uint32_t* pa = a + (wm + f * 16 + g) * TA_LD + k8 + tg;
          fa[f][0] = pa[0];                 // (row g,     k tg)
          fa[f][1] = pa[8 * TA_LD];         // (row g + 8, k tg)
          fa[f][2] = pa[4];                 // (row g,     k tg + 4)
          fa[f][3] = pa[8 * TA_LD + 4];     // (row g + 8, k tg + 4)
          const uint32_t* pbk = b + (k8 + tg) * TB_LD + wn + f * 8 + g;
          fb[f][0] = pbk[0];                // (k tg,     col g)
          fb[f][1] = pbk[4 * TB_LD];        // (k tg + 4, col g)
        }
#pragma unroll
        for (int fm = 0; fm < 4; fm++)
#pragma unroll
          for (int fn = 0; fn < 4; fn++) mma_tf32_16x8x8(acc[fm][fn], fa[fm], fb[fn]);
      }
      if (more) sstore(buf ^ 1);
      __syncthreads();
      buf ^= 1;
    }
  }

  const double sgn = mode == 1 ? 1.0 : -1.0;
#pragma unroll
  for (int fm = 0; fm < 4; fm++)
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int i = i0 + wm + fm * 16 + g + 8 * h;    // accumulator rows g (c0, c1) and g + 8 (c2, c3)
      if (i >= M) continue;
#pragma unroll
      for (int fn = 0; fn < 4; fn++) {
        const int j = j0 + wn + fn * 8 + 2 * tg;      // accumulator columns 2 tg, 2 tg + 1
        if (j >= N) continue;
        *reinterpret_cast<double2*>(C + (size_t)i * ldh + j) =
            make_double2(sgn * (double)acc[fm][fn][2 * h], sgn * (double)acc[fm][fn][2 * h + 1]);
      }
    }
}

static cudaError_t merge_tf32_launch(const Problem* d_probs, int nprob, int mode, int m, int nmerge, cudaStream_t st, int* launches) {
  const int t = (m + TM - 1) / TM;
  if (t <= 0 || nmerge <= 0) return cudaSuccess;
  merge_tf32_kernel<<<dim3(t * ((m + TN - 1) / TN), nmerge, nprob), 256, 0, st>>>(d_probs, mode, m);
  if (launches) *launches += 1;
  return cudaGetLastError();
}
// Systems wider than this take the GEMM-rich path.
// Measured on B200: D'=1001 (ldh 1024) rebuilds take 4.9 ms (8 problems) / 2.0 ms (1) wide vs 8.1 / 2.75 ms narrow.
constexpr int WIDE_MIN = 1000;

// Wide systems (Ysym != NULL, ldh > 2048): the solver never needs H^-1 itself, only the
// product H^-1 q = Y^T (Y q) with Y = L^-1.  Ysym receives Y (bf16) in SYMMETRIC storage, M[i][j] = Y[max(i,j)][min(i,j)]: row r of
// the lower part is row r of Y, row c of the upper part is column c of Y, so both triangular GEMVs of the direction read rows
// (coalesced) and together touch each element once -- the same bytes as one GEMV with a full H^-1, without the D'^3/3-flop
// Y^T Y product (10 ms of DMMA per 10k-wide factorisation).
__global__ void __launch_bounds__(256) ysym_kernel(const Problem* __restrict__ probs) {
  const Problem& pb = probs[blockIdx.z];
  const Ctrl* c = pb.ctrl;
  if (c->done || !c->need_hess) return;
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj > bi) return;
  __shared__ float t[32][33];
  const int ldh = pb.ldh;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int i = bi * 32 + r, j = bj * 32 + tx;
    const float v = j <= i ? (float)pb.Yinv[(size_t)i * ldh + j] : 0.f;
    t[r][tx] = v;
    if (j <= i) pb.Ysym[(size_t)i * ldh + j] = __float2bfloat16_rn(v);
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int j = bj * 32 + r, i = bi * 32 + tx;     // element (j, i) of the upper part = Y[i][j]
    if (j < i) pb.Ysym[(size_t)j * ldh + i] = __float2bfloat16_rn(t[tx][r]);
  }
}

bool cholesky_factored_direction(int ldh) { return ldh > 2048; }   // = the problems that carry Ysym (batch_alloc)

static cudaError_t cholesky_launch_wide(const Problem* d_probs, int nprob, int ldh, cudaStream_t st, int* launches, bool factored_direction) {
  cudaError_t e;
  // ---- factorisation
  for (int c = 0; c < ldh; c += WNB) {
    const int w = std::min(WNB, ldh - c);
    for (int k = c / NB; k < (c + w) / NB; k++) {
      const int below = ldh - (k + 1) * NB;
      const int gx = below > 0 ? (below + RB - 1) / RB : 1;
      chol_diag_kernel<<<nprob, 32, 0, st>>>(d_probs, k);
      if (below > 0) chol_panel_kernel<<<dim3(gx, nprob), 256, 0, st>>>(d_probs, k);
      if (launches) *launches += 2;
      const int inner = c + w - (k + 1) * NB;   // panel columns still to be updated
      if (inner > 0) {
        chol_update_kernel<<<dim3((inner + TB - 1) / TB, (below + TB - 1) / TB, nprob), 256, 0, st>>>(d_probs, k, c + w);
        if (launches) *launches += 1;
      }
    }
    const int rest = ldh - c - w;
    if (rest > 0 && (e = dgemm_launch<true, true>(d_probs, nprob, 0, c, w, rest, rest, 1, st, launches)) != cudaSuccess) return e;
  }
  // ---- inverse: leaves, then merges
  trinv_kernel<64><<<dim3((ldh + 63) / 64, nprob), 256, 0, st>>>(d_probs, WLEAF);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (launches) *launches += 1;
  // the factored direction reads Y only as bf16 (ysym_kernel): its merges run in TF32; an explicit H^-1 (posterior variance,
  // systems up to 2048 columns) keeps the fp64 merges
  for (int m = WLEAF; m < ldh; m *= 2) {
    const int nmerge = (ldh + 2 * m - 1) / (2 * m);
    if (factored_direction) {
      if ((e = merge_tf32_launch(d_probs, nprob, 1, m, nmerge, st, launches)) != cudaSuccess) return e;
      if ((e = merge_tf32_launch(d_probs, nprob, 2, m, nmerge, st, launches)) != cudaSuccess) return e;
      continue;
    }
    if ((e = dgemm_launch<true, false>(d_probs, nprob, 1, m, 0, m, m, nmerge, st, launches)) != cudaSuccess) return e;
    if ((e = dgemm_launch<true, false>(d_probs, nprob, 2, m, 0, m, m, nmerge, st, launches)) != cudaSuccess) return e;
  }
  if (factored_direction) {
    ysym_kernel<<<dim3(ldh / 32, ldh / 32, nprob), 256, 0, st>>>(d_probs);
    if (launches) *launches += 1;
    return cudaGetLastError();
  }
  // ---- Hinv = Y^T Y
  return dgemm_launch<false, false>(d_probs, nprob, 3, 0, 0, ldh, ldh, 1, st, launches);
}

// Cold start of a multi-lambda run with equal rho: the L problems of a partition have the same H = G + rho I, so only
// the group's first problem is factorised and inverted; the host then copies its inverse to the others.
// begin: park the followers (need_hess = 0 makes every factorisation kernel skip them); end: give them the leader's outcome.
__global__ void chol_share_begin_kernel(const Problem* __restrict__ probs, int nprob, int share) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nprob && b % share != 0) probs[b].ctrl->need_hess = 0;
}
__global__ void chol_share_end_kernel(const Problem* __restrict__ probs, int nprob, int share) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nprob || b % share == 0) return;
  Ctrl* c = probs[b].ctrl;
  const Ctrl* lead = probs[b - b % share].ctrl;
  c->need_hess = 1;
  if (lead->fail == 1) { c->fail = 1; c->done = 1; c->hess_valid = 0; }
  else {
    c->hess_valid = 1; c->hess_builds++; c->tot_hess++; c->bfgs_count = 0; c->h0_scale = 1.0; c->build_step = c->newton_steps;
    c->ysym_use = probs[b - b % share].Ysym;   // wide systems: no copy of the factored inverse, the group streams the leader's
  }
}
cudaError_t cholesky_share_begin(const Problem* d_probs, int nprob, int share, cudaStream_t st, int* launches) {
  chol_share_begin_kernel<<<(nprob + 127) / 128, 128, 0, st>>>(d_probs, nprob, share);
  if (launches) *launches += 1;
  return cudaGetLastError();
}
cudaError_t cholesky_share_end(const Problem* d_probs, int nprob, int share, cudaStream_t st, int* launches) {
  chol_share_end_kernel<<<(nprob + 127) / 128, 128, 0, st>>>(d_probs, nprob, share);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// skip_prep: Lc already holds H (lower triangle + diag(q) + identity padding), e.g. the exact fp64 Hessian of k6_postvar.cu
// want_hinv: the caller reads the explicit H^-1 afterwards (posterior variance, the inverse parity test): wide systems then run
// the Y^T Y product even where the solver's direction works on the factored form (see ysym_kernel).
cudaError_t cholesky_launch(const Problem* d_probs, int nprob, int ldh, cudaStream_t st, int* launches, int share, int skip_prep, int want_hinv) {
  if (!skip_prep) {
    dim3 blk(32, 8);
    dim3 grd((ldh + 31) / 32, (ldh + 7) / 8, nprob);
    chol_prep_kernel<<<grd, blk, 0, st>>>(d_probs, share);
    if (launches) *launches += 1;
  }
  const int nb = ldh / NB;
  if (ldh > WIDE_MIN) {
    cudaError_t e = cholesky_launch_wide(d_probs, nprob, ldh, st, launches, cholesky_factored_direction(ldh) && !want_hinv);
    if (e != cudaSuccess) return e;
  } else {
    for (int k = 0; k < nb; k++) {
      const int below = ldh - (k + 1) * NB;
      const int gx = below > 0 ? (below + RB - 1) / RB : 1;
      chol_diag_kernel<<<nprob, 32, 0, st>>>(d_probs, k);
      if (below > 0) chol_panel_kernel<<<dim3(gx, nprob), 256, 0, st>>>(d_probs, k);
      if (launches) *launches += 2;
      if (below > 0) {
        const int T = (below + TB - 1) / TB;
        chol_update_kernel<<<dim3(T, T, nprob), 256, 0, st>>>(d_probs, k, ldh);
        if (launches) *launches += 1;
      }
    }
    // explicit inverse (reads the panel blocks below the diagonal from Lc and the diagonal inverses from Ldinv)
    trinv_kernel<32><<<dim3((ldh + 31) / 32, nprob), 256, 0, st>>>(d_probs, 0);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (launches) *launches += 1;
    const int T = (ldh + TB - 1) / TB;
    hinv_syrk_kernel<<<dim3(T, T, nprob), 256, 0, st>>>(d_probs);
    if (launches) *launches += 1;
  }
  chol_finish_kernel<<<dim3(nb, nprob), 256, 0, st>>>(d_probs);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

}  // namespace mlease
