// session.cu -- host side of libmlease_b200.so: the C ABI of include/mlease_b200.h, device memory
// management, partition upload, the Newton slot loop and the ADMM iteration driver.
// No CPU fallback anywhere: every compute entry point needs a CUDA device and fails loudly without one.
#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/mlease_b200.h"
#include "kernels.cuh"

using namespace mlease;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
}  // namespace
// comm.cu reports through the same thread-local error string
extern "C" int mlease_internal_set_error(int code, const char* msg) { return fail(code, msg ? msg : ""); }
extern "C" int mlease_internal_allreduce(mlease_comm* c, double* buf, size_t count, void* stream);
namespace {
#define CK(call)                                                                                                  \
  do {                                                                                                            \
    cudaError_t e__ = (call);                                                                                     \
    if (e__ != cudaSuccess)                                                                                       \
      return fail(MLEASE_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + \
                                       std::to_string(__LINE__) + ")");                                           \
  } while (0)

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// ------------------------------------------------------------------------------------------
// upload helpers
// ------------------------------------------------------------------------------------------
__global__ void fill_bias_pad_kernel(float* X, long long n, int ldx, int Dg, int has_bias) {
  const int npad = ldx - Dg;
  const long long total = n * npad;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / npad;
    const int c = Dg + (int)(e % npad);
    X[i * ldx + c] = (c == Dg && has_bias) ? 1.0f : 0.0f;
  }
}
// response {1,0,-1} -> int8 {+1,-1,-1} (llf/LibLinearDataset.java:419-422); weight >= 0 (:428-429)
__global__ void convert_labels_kernel(long long n, const int* resp, const float* w_in, const float* o_in, signed char* y, float* w,
                                      float* o, int* bad) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int r = resp[i];
    if (r != 1 && r != 0 && r != -1) atomicOr(bad, 1);
    y[i] = (r == 1) ? 1 : -1;
    const float ww = w_in ? w_in[i] : 1.0f;
    if (!(ww >= 0.f)) atomicOr(bad, 2);
    w[i] = ww;
    o[i] = o_in ? o_in[i] : 0.0f;
  }
}
__global__ void check_rows_sorted_kernel(long long n, const long long* rowptr, const int* colidx, int* bad) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    for (long long j = rowptr[i] + 1; j < rowptr[i + 1]; j++)
      if (colidx[j] <= colidx[j - 1]) { atomicOr(bad, 8); break; }
}
// max |a[i]| as the bit pattern of a non-negative float (order preserving), NaN ignored
__global__ void absmax_kernel(long long n, const float* __restrict__ a, unsigned* __restrict__ out) {
  float m = 0.f;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(a[j]));
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));
}
__global__ void check_csr_kernel(long long nnz, const int* colidx, float* vals, int Dg, int binary, int* bad) {
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += (long long)gridDim.x * blockDim.x) {
    const int c = colidx[j];
    if (c < 0 || c >= Dg) atomicOr(bad, 4);
    if (binary) vals[j] = 1.0f;
  }
}
__global__ void repack_rows_kernel(float* dst, int ldx, const float* src, long long ld_in, long long rows, int Dg) {
  const long long total = rows * Dg;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / Dg;
    const int c = (int)(e - i * Dg);
    dst[i * ldx + c] = src[i * ld_in + c];
  }
}
// End-of-slot poll for large batches (one CTA): flag_out[0] = running | emit << 1; and, for the Gram / Cholesky launches of
// the NEXT slot, the problems that may rebuild there (running and emit set) are copied, as Problem structs, into `compact`
// and counted in flag_out[1]: a rebuild slot then launches grids over those only instead of over thousands of finished fits.
__global__ void poll2_kernel(const Problem* probs, int nprob, int* flag_out, Problem* compact) {
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  int running = 0, emit = 0;
  for (int b = threadIdx.x; b < nprob; b += blockDim.x) {
    const Ctrl* c = probs[b].ctrl;
    if (!c->done) {
      running = 1;
      if (c->emit) { emit = 1; compact[atomicAdd(&s_cnt, 1)] = probs[b]; }   // order is irrelevant: the problems are independent
    }
  }
  running = __syncthreads_or(running);
  emit = __syncthreads_or(emit);
  if (threadIdx.x == 0) { flag_out[0] = running | (emit << 1); flag_out[1] = s_cnt; }
}

struct PartData {
  int pid = -1;
  long long n = 0;
  bool csr = false;
  float* X = nullptr;
  signed char* y = nullptr;
  float* w = nullptr;
  float* o = nullptr;
  long long* rowptr = nullptr;
  int* colidx = nullptr;
  float* vals = nullptr;
  long long nnz = 0;
  int csr_unique = 0;
  float vmax = 0.f, wmax = 1.f;
  long long* bm_offs = nullptr;    // block-major entry list for the CSR Gram (built at upload when rows are sorted & unique)
  unsigned short* bm_keys = nullptr;
  float* bm_vals = nullptr;
  long long bm_groups = 0;
  int nblk128 = 0;
  // segment lists of the fused multi-lambda CSR K1 (k1_csr_fused.cu), built at upload for rows with unique sorted columns
  int sg_S = 0, sg_rows = 0, sg_ngrp = 0;
  int* sg_perm = nullptr; int* sg_depth = nullptr; long long* sg_goff = nullptr; unsigned short* sg_row16 = nullptr; float* sg_val = nullptr;
  long long sg_total = 0;   // 32-lane rows stored (padding included)
};

// A batch of problems with identical shape that advance in lockstep through the Newton slots.
struct Batch {
  int nprob = 0, Dt = 0, ldx = 0, Dp = 0, ldh = 0;
  bool csr = false;
  int has_bias = 1;
  int k1_grid = 1, gram_slices = 1, ntiles = 0;
  int gram_from_csr = 0;          // every problem of the batch assembles its Gram tiles from CSR (no dense bf16 operand) on CTA
                                  // pairs (cta_group::2, 256 x 256 tiles); d_tiles then holds pair tiles
  int group_L = 1;                // problems b = g * group_L + l share the data of partition g (the lambdas of one partition)
  int k1_fused = 0;               // the fused multi-lambda CSR K1 runs (segment lists present): one launch, grid (sg_S, nprob / group_L)
  int k1f_LP = 1;                 // lambdas padded to 1 / 2 / 4 in the interleaved shared-memory vectors
  size_t k1f_smem = 0;
  int k1_dyn = 0;                 // > 0: K1 CTAs are dealt to the running problems at run time (value = nprob, <= 32); k1_grid = whole grid
  int rebuild_is_expensive = 0;   // cost model: Gram + Cholesky + inverse vs one K1 pass (set in batch_alloc); also turns on the
                                  // self-scaling of the stale inverse from the secant pairs
  std::vector<Problem> h;
  Problem* d = nullptr;
  Problem* d_compact = nullptr;   // large batches: Problem structs of the problems that may rebuild in the next slot
  Ctrl* d_ctrl = nullptr;
  void* d_tmaps = nullptr;
  void* d_tiles = nullptr;
  std::vector<Ctrl> mirror;   // host copy of the control blocks as of the last read-back
  Ctrl* h_ctrl[2] = {nullptr, nullptr};   // pinned read-back buffers of the slot pipeline (small batches)
  cudaEvent_t slot_ev[2] = {nullptr, nullptr};
  std::vector<void*> owned;
  ~Batch() {
    for (void* p : owned) cudaFree(p);
    for (int i = 0; i < 2; i++) { if (h_ctrl[i]) cudaFreeHost(h_ctrl[i]); if (slot_ev[i]) cudaEventDestroy(slot_ev[i]); }
  }
};

struct Counters {
  long long k1_passes = 0, gram_builds = 0, newton_steps = 0, rejected = 0, launches = 0;
  int not_converged = 0, last_slots = 0;
  double k1_bytes = 0;     // algorithmic bytes of all K1 passes (SURVEY 8d): dense n*(4*ldx+9), CSR 8*nnz+8*n+9*n
  double k1_emit_bytes = 0;// extra bytes written by passes that emitted the scaled bf16 copy (n*Dp*2)
  double gram_flops = 0;   // algorithmic flops of all Gram builds: n*Dt*(Dt+1) (lower triangle, 2 flop/MAC)
  double k1_shared_bytes = 0;  // CSR: bytes of the K1 passes when the lambdas of a partition are counted as ONE read of its rows:
                               // per (partition, slot) with A active lambdas 8*nnz + 9*n + 8*n*A (rows once, r/d out per lambda)
};

// Optional per-kernel device timing (CUDA events on the launching stream) for bench.py's roofline.
struct Profiler {
  bool on = false;
  struct Rec { int cat; cudaEvent_t a, b; };
  std::vector<Rec> recs;
  std::vector<cudaEvent_t> pool;
  double ms[4] = {0, 0, 0, 0};
  long long n[4] = {0, 0, 0, 0};
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
  void begin(int cat, cudaStream_t st) {
    if (!on) return;
    Rec r; r.cat = cat; r.a = get(); r.b = get();
    cudaEventRecord(r.a, st);
    recs.push_back(r);
  }
  void end(cudaStream_t st) {
    if (!on) return;
    cudaEventRecord(recs.back().b, st);
  }
  void resolve() {   // call after a stream synchronize
    for (auto& r : recs) {
      float t = 0;
      if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms[r.cat] += t; n[r.cat]++; }
      pool.push_back(r.a); pool.push_back(r.b);
    }
    recs.clear();
  }
  ~Profiler() { for (auto& r : recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); } for (auto e : pool) cudaEventDestroy(e); }
};

int dev_alloc(Batch& B, void** p, size_t bytes, bool zero = true) {
  CK(cudaMalloc(p, bytes ? bytes : 16));
  B.owned.push_back(*p);
  if (zero) CK(cudaMemset(*p, 0, bytes ? bytes : 16));
  return 0;
}

// Allocate the per-problem solver state.  Data pointers (X, y, ...) and n must be filled in h[] first.
int batch_alloc(Batch& B, int num_sms) {
  const int nprob = B.nprob, ldx = B.ldx;
  B.Dp = round_up(B.ldx, 128);
  B.ldh = round_up(B.Dt, 32);
  long long maxn = 1;
  for (auto& p : B.h) maxn = std::max(maxn, p.n);
  if (B.csr) {
    const int cps = 1;   // 1024-thread CTAs at 64 registers: one per SM
    B.k1_dyn = (nprob > 1 && nprob <= 32) ? nprob : 0;
    if (B.k1_dyn) B.k1_grid = (int)std::max(1LL, std::min((long long)num_sms * cps, (long long)nprob * ((maxn + 63) / 64)));
    else B.k1_grid = std::max(1, std::min((int)((maxn + 63) / 64), (num_sms * cps) / std::max(1, nprob)));
  } else {
    int R, S, G, cps = 1;
    size_t smem;
    if (!k1_dense_plan(ldx, &R, &S, &G, &smem, &cps))
      return fail(MLEASE_ERR_INVALID, "dense partitions support at most 4095 features (+intercept); use CSR input beyond that");
    const long long row_tiles = (maxn + R - 1) / R;
    B.k1_dyn = (nprob > 1 && nprob <= 32) ? nprob : 0;
    if (B.k1_dyn) B.k1_grid = (int)std::max(1LL, std::min((long long)num_sms * cps, (long long)nprob * row_tiles));
    else B.k1_grid = (int)std::max(1LL, std::min(row_tiles, (long long)std::max(1, (num_sms * cps) / std::max(1, nprob))));
  }
  B.gram_from_csr = B.csr ? 1 : 0;
  for (auto& p : B.h) if (!p.bm_offs) B.gram_from_csr = 0;
  // fused multi-lambda CSR K1: every problem has segment lists, the groups are whole, and the shared-memory vectors fit
  B.k1_fused = 0;
  if (B.csr && B.gram_from_csr && B.group_L >= 1 && B.group_L <= 4 && nprob % B.group_L == 0) {
    bool ok = true;
    for (auto& p : B.h) if (!p.sg_perm || p.sg_S != B.h[0].sg_S || p.sg_rows != B.h[0].sg_rows) ok = false;
    if (ok) {
      B.k1f_LP = B.group_L <= 1 ? 1 : (B.group_L == 2 ? 2 : 4);
      B.k1f_smem = (size_t)ldx * 4 * B.k1f_LP + (size_t)B.h[0].sg_rows * 4 * B.k1f_LP;
      if (B.k1f_smem <= 224 * 1024) { B.k1_fused = 1; B.k1_dyn = 0; B.k1_grid = B.h[0].sg_S; }
    }
  }
  const int gpart_rows = B.k1_fused ? 1 : B.k1_grid;   // the fused kernel keeps its partials in gpart_f (fp32)
  // Cost model for the rebuild policy (seconds, order of magnitude): one K1 pass streams the partition at ~5 TB/s; a rebuild
  // is n*Dt^2 bf16 flop at ~1 PFLOP/s (tcgen05 Gram, lower triangle) plus ~Dt^3 fp64 flop at ~5 TFLOP/s (Cholesky + inverse).
  {
    double bytes = 0;
    for (auto& p : B.h) bytes = std::max(bytes, B.csr ? 8.0 * (double)p.nnz_hint + 17.0 * (double)p.n : (double)p.n * 4.0 * ldx);
    const double t_pass = bytes / 5e12 + 20e-6;
    const double t_rebuild = (double)maxn * B.Dt * B.Dt / 1e15 + (double)B.Dt * B.Dt * B.Dt / 5e12 + 300e-6;
    // only wide systems qualify: small ones (NaiveTrain's per-key fits, cold-started every time) are launch-bound, not
    // flop-bound, and a mid-update rebuild saves them many lock-step slots
    B.rebuild_is_expensive = (t_rebuild > 8.0 * t_pass && B.Dt > 2048) ? 1 : 0;
  }
  // Gram decomposition
  constexpr int MAX_TILES = 1 << 18;   // lower 128x256 tiles of Dp up to ~90k
  std::vector<short> tiles(2 * (size_t)MAX_TILES);
  B.ntiles = gram_tile_list(B.Dp, tiles.data(), MAX_TILES, B.gram_from_csr);
  if (B.ntiles <= 0) return fail(MLEASE_ERR_INVALID, "Gram tile list overflow");
  {
    const long long ksteps = (maxn + 63) / 64;
    const long long base = (long long)B.ntiles * nprob;   // CTAs, or CTA pairs
    const long long cap = std::max(1, num_sms / (B.gram_from_csr ? 2 : 1));
    int best = 1;
    double best_eff = 0;
    for (int s = 1; s <= 16; s++) {
      if (s > ksteps) break;
      const long long ctas = base * s;
      const double eff = (double)ctas / (double)(((ctas + cap - 1) / cap) * cap);
      if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
      if (eff >= 0.93 && ctas >= 2LL * cap) { best = s; break; }
    }
    // bound the split-K scratch to 1 GiB per batch
    while (best > 1 && (double)best * B.Dp * B.Dp * 4.0 * nprob > 1024.0 * 1024 * 1024) best--;
    B.gram_slices = best;
  }
  const size_t nd = (size_t)nprob * ((9 + 2 * BFGS_M) * (size_t)ldx + 2 * BFGS_M + (size_t)gpart_rows * ldx + (size_t)B.k1_grid + 8);
  const size_t nf = (size_t)nprob * 4 * ldx;
  double* dd; float* ff; float* hp; double* lc; double* ld; double* ldi; double* yi; double* hi;
  if (int rc = dev_alloc(B, (void**)&dd, nd * sizeof(double))) return rc;
  if (int rc = dev_alloc(B, (void**)&ff, nf * sizeof(float))) return rc;
  float* gpf = nullptr;
  if (B.k1_fused)
    if (int rc = dev_alloc(B, (void**)&gpf, (size_t)nprob * B.k1_grid * ldx * sizeof(float))) return rc;
  if (int rc = dev_alloc(B, (void**)&hp, (size_t)nprob * B.gram_slices * B.Dp * B.Dp * sizeof(float))) return rc;
  if (int rc = dev_alloc(B, (void**)&lc, (size_t)nprob * B.ldh * B.ldh * sizeof(double))) return rc;
  if (int rc = dev_alloc(B, (void**)&ld, (size_t)nprob * B.ldh * 32 * sizeof(double))) return rc;
  if (int rc = dev_alloc(B, (void**)&ldi, (size_t)nprob * B.ldh * 32 * sizeof(double))) return rc;
  if (int rc = dev_alloc(B, (void**)&yi, (size_t)nprob * B.ldh * B.ldh * sizeof(double))) return rc;
  if (int rc = dev_alloc(B, (void**)&hi, (size_t)nprob * B.ldh * B.ldh * sizeof(double))) return rc;
  __nv_bfloat16* hif = nullptr;
  if (cholesky_factored_direction(B.ldh))
    if (int rc = dev_alloc(B, (void**)&hif, (size_t)nprob * B.ldh * B.ldh * sizeof(__nv_bfloat16))) return rc;
  if (int rc = dev_alloc(B, (void**)&B.d_ctrl, (size_t)nprob * sizeof(Ctrl))) return rc;
  if (int rc = dev_alloc(B, (void**)&B.d, (size_t)nprob * sizeof(Problem))) return rc;
  if (nprob > 64)
    if (int rc = dev_alloc(B, (void**)&B.d_compact, (size_t)nprob * sizeof(Problem))) return rc;
  if (int rc = dev_alloc(B, &B.d_tmaps, (size_t)nprob * sizeof(CUtensorMap))) return rc;
  if (int rc = dev_alloc(B, &B.d_tiles, (size_t)B.ntiles * 2 * sizeof(short))) return rc;
  CK(cudaMemcpy(B.d_tiles, tiles.data(), (size_t)B.ntiles * 2 * sizeof(short), cudaMemcpyHostToDevice));
  std::vector<CUtensorMap> maps(nprob);
  std::vector<size_t> pool_off(nprob);
  size_t pool_bytes = 0;
  for (int b = 0; b < nprob; b++) {
    pool_off[b] = pool_bytes;
    const bool windows = B.gram_from_csr && k1_csr_window(ldx) > 0;   // then a second [n] vector (row residuals) follows sdvec
    const size_t need = B.gram_from_csr ? (size_t)B.h[b].n * sizeof(float) * (windows ? 2 : 1) : (B.h[b].Xt ? 0 : (size_t)B.h[b].n * B.Dp * sizeof(__nv_bfloat16));
    pool_bytes += (need + 255) & ~(size_t)255;
  }
  unsigned char* pool = nullptr;
  if (int rc = dev_alloc(B, (void**)&pool, pool_bytes)) return rc;
  for (int b = 0; b < nprob; b++) {
    Problem& p = B.h[b];
    p.ldx = ldx; p.Dt = B.Dt; p.Dp = B.Dp; p.ldh = B.ldh; p.self_idx = b;
    p.k1_ctas = B.k1_grid;
    p.gram_slices = B.gram_slices;
    double* q = dd;
    p.beta = q; q += ldx; p.beta_t = q; q += ldx; p.m = q; q += ldx; p.q = q; q += ldx;
    p.g_t = q; q += ldx; p.g_acc = q; q += ldx; p.dir = q; q += ldx; p.x_d = q; q += ldx;
    p.qf = reinterpret_cast<float*>(q); p.tf = p.qf + ldx; q += ldx;   // one double-vector slot holds the two fp32 vectors of the triangular GEMVs
    p.bfgs_S = q; q += (size_t)BFGS_M * ldx; p.bfgs_Y = q; q += (size_t)BFGS_M * ldx; p.bfgs_rho = q; q += BFGS_M; p.bfgs_alpha = q; q += BFGS_M;
    p.gpart = q; q += (size_t)gpart_rows * ldx;
    p.gpart_f = gpf ? gpf + (size_t)b * B.k1_grid * ldx : nullptr;
    p.fpart = q; q += B.k1_grid + 8;
    dd = q;
    float* f = ff;
    p.beta_tf = f; f += ldx; p.u_f = f; f += ldx; p.uplusx_f = f; f += ldx; p.x_f = f; f += ldx;
    ff = f;
    p.Hpart = hp + (size_t)b * B.gram_slices * B.Dp * B.Dp;
    p.Lc = lc + (size_t)b * B.ldh * B.ldh;
    p.Ldiag = ld + (size_t)b * B.ldh * 32;
    p.Ldinv = ldi + (size_t)b * B.ldh * 32;
    p.Yinv = yi + (size_t)b * B.ldh * B.ldh;
    p.Hinv = hi + (size_t)b * B.ldh * B.ldh;
    p.Ysym = hif ? hif + (size_t)b * B.ldh * B.ldh : nullptr;
    p.ctrl = B.d_ctrl + b;
    // Gram operand state, carved out of ONE allocation for the whole batch (NaiveTrain batches hold thousands of problems:
    // one cudaMalloc / cudaFree each would cost more than the fits)
    if (B.gram_from_csr) {
      p.sdvec = reinterpret_cast<float*>(pool + pool_off[b]);
      p.rvec = k1_csr_window(ldx) > 0 ? p.sdvec + p.n : nullptr;
      p.gram_from_csr = 1;
      std::memset(&maps[b], 0, sizeof(CUtensorMap));
    } else {
      p.gram_from_csr = 0;
      p.gram_scale = 1.f; p.gram_unscale = 1.f;   // bf16 dense-operand Gram: no operand scale
      if (!p.Xt) p.Xt = reinterpret_cast<__nv_bfloat16*>(pool + pool_off[b]);
      if (gram_make_tensor_map(&maps[b], p.Xt, p.n, B.Dp) != 0) return fail(MLEASE_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    }
  }
  CK(cudaMemcpy(B.d_tmaps, maps.data(), (size_t)nprob * sizeof(CUtensorMap), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(B.d, B.h.data(), (size_t)nprob * sizeof(Problem), cudaMemcpyHostToDevice));
  return 0;
}

// K1 of a slot: the fused multi-lambda CSR kernel when the batch has segment lists, the per-problem kernels otherwise
cudaError_t batch_k1(Batch& B, int force_emit, cudaStream_t st, int* launches) {
  if (B.k1_fused)
    return k1f_launch(B.d, B.nprob / B.group_L, B.group_L, B.h[0].sg_S, B.k1f_LP, B.k1f_smem, B.has_bias, force_emit, st, launches);
  return k1_launch(B.d, B.nprob, B.csr, B.ldx, B.has_bias, B.k1_grid, force_emit, st, launches, B.gram_from_csr, B.k1_dyn);
}

// Gram of a rebuild over d_probs (B.d or its compacted copy): operand tiles assembled from CSR on CTA pairs, or the dense TMA kernel
cudaError_t batch_gram(Batch& B, const Problem* d_probs, int nprob, int force, int share, cudaStream_t st, int* launches) {
  if (B.gram_from_csr)
    return gram_launch_csr_tcgen05(d_probs, nprob, B.d_tiles, B.ntiles, B.gram_slices, force, B.has_bias ? B.Dt - 1 : -1, st, launches, share);
  return gram_launch_tcgen05(d_probs, nprob, B.d_tmaps, B.d_tiles, B.ntiles, B.gram_slices, force, st, launches, share);
}

// One x-update for every problem of the batch: beta (init), m, q must already be on the device.
int batch_xupdate(Batch& B, cudaStream_t st, double xtol, int max_newton, int policy, int invalidate, int* h_flag, int* d_flag,
                  Counters& cnt, Profiler* prof = nullptr, int share_first_gram = 0, int share_first_factor = 0) {
  Profiler nop;
  Profiler& pf = prof ? *prof : nop;
  int launches = 0;
  CK(newton_begin(B.d, B.nprob, xtol, max_newton, policy, invalidate, B.rebuild_is_expensive, st, &launches));
  // The first slot's flags are known on the host: every problem is running, and a rebuild is due iff the policy says
  // always, the factors were invalidated, or the mirrored control blocks say so (no factor yet / refresh requested).
  const bool small = B.nprob <= 64;   // small batches read the whole control array back each slot (one sync, no poll kernel)
  int flag = 1;
  {
    bool emit0 = policy == 1 || invalidate || B.mirror.empty();
    for (auto& c : B.mirror) if (!c.hess_valid || c.refresh_next) emit0 = true;
    if (emit0) flag |= 2;
  }
  B.mirror.resize(B.nprob);
  std::vector<Ctrl>& hc = B.mirror;
  int slots = 0;
  const Problem* d_hess = B.d;   // problems the Gram / Cholesky grids run over (large batches: compacted by poll2_kernel)
  int n_hess = B.nprob;
  double shared_flops = 0;   // Gram builds that were not run because the group's first problem stood in for them
  // One slot's launches.  with_hess: the Gram / Cholesky launches of a rebuild are included; spec: see k1_reduce_decide_kernel.
  auto enqueue_slot = [&](int slot_idx, bool with_hess, bool spec) -> int {
    pf.begin(0, st);
    CK(batch_k1(B, -1, st, &launches));
    pf.end(st);
    pf.begin(1, st);
    CK(k1_reduce_decide(B.d, B.nprob, B.Dt, st, &launches, spec ? 1 : 0));
    pf.end(st);
    if (with_hess && n_hess > 0) {
      pf.begin(2, st);
      // cold start of a multi-lambda run: the L problems of a partition all sit at beta = 0, their Grams are the same
      const int share = (slot_idx == 0) ? share_first_gram : 0;
      if (share > 1)
        for (int b = 0; b < B.nprob; b++) if (b % share != 0) shared_flops += (double)B.h[b].n * (double)B.Dt * (double)(B.Dt + 1);
      CK(batch_gram(B, d_hess, n_hess, 0, share, st, &launches));
      pf.end(st);
      pf.begin(3, st);
      const bool share_fact = share > 1 && share_first_factor;   // same rho too: same H, one factorisation per group
      if (share_fact) CK(cholesky_share_begin(B.d, B.nprob, share, st, &launches));
      CK(cholesky_launch(d_hess, n_hess, B.ldh, st, &launches, share));
      if (share_fact) {
        CK(cholesky_share_end(B.d, B.nprob, share, st, &launches));
        const size_t hh = (size_t)B.ldh * B.ldh;
        for (int b = 0; b < B.nprob; b++) {
          if (b % share == 0) continue;
          const Problem& lead = B.h[b - b % share];
          // wide systems work on the factored form Y = L^-1 (bf16, Ysym): that is all a follower needs
          if (!cholesky_factored_direction(B.ldh)) CK(cudaMemcpyAsync(B.h[b].Hinv, lead.Hinv, hh * sizeof(double), cudaMemcpyDeviceToDevice, st));
          // (Ysym is not copied: chol_share_end_kernel points the follower's Ctrl::ysym_use at the leader's)
        }
      }
      pf.end(st);
    }
    pf.begin(1, st);
    CK(newton_solve(B.d, B.nprob, B.ldh, st, &launches, B.group_L));
    if (!small) { poll2_kernel<<<1, 256, 0, st>>>(B.d, B.nprob, d_flag, B.d_compact); launches++; }
    pf.end(st);
    return 0;
  };
  if (small) {
    // Slot pipeline: the host runs ONE slot ahead of what it knows.  While slot s executes, slot s+1 is already enqueued in
    // speculative form (no rebuild launches; a rebuild that turns out to be due is deferred by the decide kernel and shows
    // up as `emit` in the flags, after which a regular rebuild slot follows).  The read-back of the control blocks goes to
    // pinned double buffers and is awaited per slot (event), so the GPU never idles on the host between slots; a finished
    // x-update leaves at most one slot of early-exit kernels behind.
    for (int i = 0; i < 2; i++) {
      if (!B.h_ctrl[i]) CK(cudaMallocHost((void**)&B.h_ctrl[i], (size_t)B.nprob * sizeof(Ctrl)));
      if (!B.slot_ev[i]) CK(cudaEventCreateWithFlags(&B.slot_ev[i], cudaEventDisableTiming));
    }
    const bool may_spec = policy == 0;
    auto flags_of = [&](const Ctrl* c, bool* all_valid) {
      int f = 0; bool v = true;
      for (int b = 0; b < B.nprob; b++) if (!c[b].done) { f |= 1; if (c[b].emit) f |= 2; if (!c[b].hess_valid) v = false; }
      *all_valid = v;
      return f;
    };
    auto finish_slot = [&](int idx) -> int {
      CK(cudaMemcpyAsync(B.h_ctrl[idx & 1], B.d_ctrl, (size_t)B.nprob * sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
      CK(cudaEventRecord(B.slot_ev[idx & 1], st));
      return 0;
    };
    // what is known before slot 0: every problem runs; a rebuild is due iff emit0; factors are valid iff the mirror says so
    bool known_valid = !(flag & 2);
    if (int rc = enqueue_slot(0, (flag & 2) != 0, false)) return rc;
    if (int rc = finish_slot(0)) return rc;
    int s_cur = 0;          // newest slot in flight whose outcome is not known yet
    bool next_in_flight = false;
    int known_flag = flag;  // flags as of the newest COMPLETED slot (before slot 0: the host-side prediction)
    while (true) {
      // speculate slot s_cur + 1 on what is known (the state BEFORE slot s_cur): no rebuild pending, every factor valid
      const bool spec_next = may_spec && known_valid && !(known_flag & 2) && s_cur + 1 < 400;
      if (spec_next) {
        if (int rc = enqueue_slot(s_cur + 1, false, true)) return rc;
        if (int rc = finish_slot(s_cur + 1)) return rc;
        next_in_flight = true;
      }
      CK(cudaEventSynchronize(B.slot_ev[s_cur & 1]));
      std::memcpy(hc.data(), B.h_ctrl[s_cur & 1], (size_t)B.nprob * sizeof(Ctrl));
      slots = s_cur + 1;
      known_flag = flags_of(hc.data(), &known_valid);
      if (getenv("MLEASE_DEBUG") && atoi(getenv("MLEASE_DEBUG")) >= 2) {
        const Ctrl& c0 = hc[0];
        fprintf(stderr, "[mlease]   slot %d p0: done %d steps %d hb %d emit %d f %.10e |g| %.3e |dir| %.3e phi0 %.3e alpha %.2f wr %.3f\n", slots, c0.done,
                c0.newton_steps, c0.hess_builds, c0.emit, c0.f_acc, c0.gnorm, c0.dirnorm, c0.phi0, c0.alpha, c0.worst_ratio);
      }
      if (!(known_flag & 1) || slots >= 400) break;          // finished (a speculative slot in flight is a no-op)
      if (next_in_flight) { s_cur++; next_in_flight = false; continue; }
      if (int rc = enqueue_slot(s_cur + 1, (known_flag & 2) != 0, false)) return rc;
      if (int rc = finish_slot(s_cur + 1)) return rc;
      s_cur++;
    }
    flag = known_flag;
  }
  while (!small && (flag & 1) && slots < 400) {
    if (int rc = enqueue_slot(slots, (flag & 2) != 0, false)) return rc;
    CK(cudaMemcpyAsync(h_flag, d_flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    flag = h_flag[0];
    n_hess = h_flag[1];
    d_hess = B.d_compact;
    slots++;
  }
  if (!small) {
    CK(cudaMemcpyAsync(hc.data(), B.d_ctrl, (size_t)B.nprob * sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  cnt.launches += launches;
  cnt.last_slots = slots;
  int bad_spd = 0, bad_ls = 0;
  if (pf.on) CK(cudaStreamSynchronize(st));   // a trailing speculative slot may still be running: its events must have completed
  pf.resolve();
  if (getenv("MLEASE_DEBUG")) {
    fprintf(stderr, "[mlease] x-update: %d problems, %d slots;", B.nprob, slots);
    for (int b = 0; b < B.nprob && b < 4; b++)
      fprintf(stderr, " p%d{ev %d st %d rej %d hb %d fail %d stall %d |g| %.2e |dir| %.2e h0s %.3f}", b, hc[b].evals, hc[b].newton_steps, hc[b].rejects,
              hc[b].hess_builds, hc[b].fail, hc[b].stall, hc[b].gnorm, hc[b].dirnorm, hc[b].h0_scale);
    fprintf(stderr, "\n");
  }
  for (int b = 0; b < B.nprob; b++) {
    const Ctrl& c = hc[b];
    const Problem& p = B.h[b];
    const double rowbytes = B.csr ? 17.0 : (4.0 * B.ldx + 9.0);
    cnt.k1_bytes += (double)c.evals * ((double)p.n * rowbytes + (B.csr ? 8.0 * (double)p.nnz_hint : 0.0));
    cnt.gram_flops += (double)c.hess_builds * (double)p.n * (double)B.Dt * (double)(B.Dt + 1);
    cnt.k1_emit_bytes += (double)c.hess_builds * (double)p.n * (double)B.Dp * 2.0;
  }
  cnt.gram_flops -= shared_flops;
  if (B.csr) {
    // the problems of a group advance in lock step from the first slot and drop out as they converge: slot t serves the
    // problems with evals > t, so a group's passes = max evals, and the lambdas served in total = sum of evals
    const int gl = std::max(1, B.group_L);
    for (int g0 = 0; g0 + gl <= B.nprob; g0 += gl) {
      int mx = 0; long long sum = 0;
      for (int l = 0; l < gl; l++) { mx = std::max(mx, hc[g0 + l].evals); sum += hc[g0 + l].evals; }
      const Problem& p = B.h[g0];
      cnt.k1_shared_bytes += (double)mx * (8.0 * (double)p.nnz_hint + 9.0 * (double)p.n) + (double)sum * 8.0 * (double)p.n;
    }
  }
  for (auto& c : hc) {
    cnt.k1_passes += c.evals; cnt.newton_steps += c.newton_steps; cnt.rejected += c.rejects; cnt.gram_builds += c.hess_builds;
    if (c.fail == 3 || !c.done) cnt.not_converged++;
    if (c.fail == 1) bad_spd++;
    if (c.fail == 2) bad_ls++;
  }
  if (bad_spd) return fail(MLEASE_ERR_NUMERIC, "Model fitting error! (Hessian not positive definite in " + std::to_string(bad_spd) + " problem(s))");
  if (bad_ls) return fail(MLEASE_ERR_NUMERIC, "Model fitting error! (line search failed in " + std::to_string(bad_ls) + " problem(s))");
  return 0;
}

}  // namespace

// ============================================================================================
struct mlease_session {
  mlease_admm_config cfg;
  std::vector<float> lambdas, rhos, lambda_map;
  int Dg = 0, Dt = 0, ldx = 0, L = 0, P = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;   // H2D of a CSR partition's arrays, overlapped with the previous partition's layout build
  cudaEvent_t copy_ev = nullptr;        // orders copy_stream after what the caller queued on `stream` (e.g. kernels that produce device inputs)
  int pending_csr = -1;                 // index into parts of the CSR partition whose checks and lists are not built yet
  int num_sms = 148;
  std::vector<PartData> parts;
  std::vector<void*> owned;
  bool any_csr = false, any_dense = false;
  Batch* batch = nullptr;    // ADMM problems, b = local_part * L + l
  Batch* scratch = nullptr;  // 1 problem for mlease_objective / mlease_fit_partition / timing
  int scratch_part = -1;
  double* d_z = nullptr;
  double* d_wz = nullptr;
  double* d_rho = nullptr;   // [L] rho_eff of the coming iteration
  double* d_diff = nullptr;
  double* d_l1thr = nullptr; // [L] soft-threshold of the L1 z-update (regularizer = 1), else NULL
  double* d_exch = nullptr;  // [L][Dt] (+1: failed-fit count of this rank) for mlease_admm_run / mlease_admm_iterate
  mlease_comm* comm = nullptr;   // NCCL communicator of a multi-GPU job (not owned), or NULL
  int* d_flag = nullptr;
  int* h_flag = nullptr;     // pinned
  double* h_small = nullptr; // pinned, >= 4*L doubles
  std::vector<double> rho_fact;  // rho_eff the current Cholesky factors were built with
  int iter = 0;
  float liblinear_eps = 0.01f;
  double mindiff = 99999999;
  double last_maxdiff = 0;
  bool begun = false;
  float boost_rate = 0.f;    // initialize.boost.rate of the current run (0: cold start from z = {})
  Counters cnt;
  Profiler prof;
  double xtol = 1e-8;
  int max_newton = 50;
  ~mlease_session() {
    delete batch;
    delete scratch;
    for (void* p : owned) cudaFree(p);
    if (h_flag) cudaFreeHost(h_flag);
    if (h_small) cudaFreeHost(h_small);
    if (copy_stream) cudaStreamDestroy(copy_stream);
    if (copy_ev) cudaEventDestroy(copy_ev);
  }
};

extern "C" {
static int csr_flush_pending(mlease_session* s);   // builds the deferred lists of the last CSR partition
}

namespace {

int sess_alloc(mlease_session* s, void** p, size_t bytes) {
  CK(cudaMalloc(p, bytes ? bytes : 16));
  s->owned.push_back(*p);
  CK(cudaMemset(*p, 0, bytes ? bytes : 16));
  return 0;
}

int find_part(mlease_session* s, int pid) {
  for (size_t i = 0; i < s->parts.size(); i++)
    if (s->parts[i].pid == pid) return (int)i;
  return -1;
}

void fill_problem_data(Problem& p, const PartData& pd) {
  std::memset(&p, 0, sizeof(Problem));
  p.X = pd.X; p.n = pd.n; p.y = pd.y; p.w = pd.w; p.o = pd.o;
  p.rowptr = pd.rowptr; p.colidx = pd.colidx; p.vals = pd.vals; p.nnz_hint = pd.nnz; p.csr_unique = pd.csr_unique;
  p.bm_offs = pd.bm_offs; p.bm_keys = pd.bm_keys; p.bm_vals = pd.bm_vals; p.bm_groups = pd.bm_groups;
  p.nblk128 = pd.nblk128; p.gram_from_csr = pd.bm_offs ? 1 : 0;
  p.vmax = pd.vmax; p.wmax = pd.wmax;
  p.sg_S = pd.sg_S; p.sg_rows = pd.sg_rows; p.sg_ngrp = pd.sg_ngrp; p.sg_perm = pd.sg_perm; p.sg_depth = pd.sg_depth; p.sg_goff = pd.sg_goff;
  p.sg_row16 = pd.sg_row16; p.sg_val = pd.sg_val;
  p.gram_scale = 1.f; p.gram_unscale = 1.f;
  if (pd.bm_offs) {
    // e4m3 operands of the CSR Gram: |sqrt(d) x| <= 0.5 sqrt(wmax) max(|x|max, 1); scale the largest to ~224 (e4m3 max 448)
    const float amax = 0.5f * std::sqrt(std::max(pd.wmax, 1e-30f)) * std::max(pd.vmax, 1.f);
    int e = 0;
    std::frexp(224.f / amax, &e);
    e = std::max(-60, std::min(60, e - 1));
    p.gram_scale = std::ldexp(1.f, e);
    p.gram_unscale = std::ldexp(1.f, -2 * e);
  }
}

int finalize(mlease_session* s) {
  if (s->batch) return 0;
  if (int rc = csr_flush_pending(s)) return rc;
  if (s->copy_stream) {   // hand the builders' cached temporaries back before the solver state is allocated
    cudaMemPool_t mp;
    if (cudaDeviceGetDefaultMemPool(&mp, s->cfg.device) == cudaSuccess) cudaMemPoolTrimTo(mp, 0);
  }
  if (s->parts.empty()) return fail(MLEASE_ERR_STATE, "no partitions were added to this session");
  if (s->any_csr && s->any_dense) return fail(MLEASE_ERR_INVALID, "a session must hold either dense or CSR partitions, not both");
  std::sort(s->parts.begin(), s->parts.end(), [](const PartData& a, const PartData& b) { return a.pid < b.pid; });
  Batch* B = new Batch();
  s->batch = B;
  B->nprob = (int)s->parts.size() * s->L;
  B->Dt = s->Dt; B->ldx = s->ldx; B->csr = s->any_csr; B->has_bias = 1;
  B->group_L = s->L;
  B->h.resize(B->nprob);
  for (size_t pi = 0; pi < s->parts.size(); pi++)
    for (int l = 0; l < s->L; l++) {
      Problem& p = B->h[pi * s->L + l];
      fill_problem_data(p, s->parts[pi]);
      p.lambda_idx = l; p.part_local = (int)pi;
    }
  if (int rc = batch_alloc(*B, s->num_sms)) return rc;
  const size_t ldv = s->ldx;
  if (int rc = sess_alloc(s, (void**)&s->d_z, s->L * ldv * sizeof(double))) return rc;
  if (int rc = sess_alloc(s, (void**)&s->d_wz, s->L * ldv * sizeof(double))) return rc;
  if (int rc = sess_alloc(s, (void**)&s->d_rho, s->L * sizeof(double))) return rc;
  if (int rc = sess_alloc(s, (void**)&s->d_diff, s->L * sizeof(double))) return rc;
  if (int rc = sess_alloc(s, (void**)&s->d_exch, ((size_t)s->L * s->Dt + 1) * sizeof(double))) return rc;
  // z-update weights (jobs/RegressionAdmmTrain.java:381-386,392-403), in the reference's mixed float/double arithmetic
  std::vector<double> wz(s->L * ldv, 0.0);
  for (int l = 0; l < s->L; l++) {
    const float lf = s->lambdas[l], rf = s->rhos[l];
    const float pr = (float)s->P * rf;
    const double weight = (double)(pr / (lf + pr));
    for (int k = 0; k < s->Dg; k++) {
      double w = weight;
      if (!s->lambda_map.empty() && s->lambda_map[k] > 0.f) w = (double)pr / ((double)(s->lambda_map[k] + pr) + 0.0);
      wz[l * ldv + k] = w;
    }
    wz[l * ldv + s->Dg] = s->cfg.penalize_intercept ? weight : 1.0;
  }
  CK(cudaMemcpy(s->d_wz, wz.data(), wz.size() * sizeof(double), cudaMemcpyHostToDevice));
  if (s->cfg.regularizer == 1) {
    // weight = l / (r * nblocks + 0.0) (jobs/RegressionAdmmTrain.java:409): float product, double division.  The weightmap
    // built from lambda.map (:411-415) is never used by the thresholding loop, so lambda_map has no effect under L1.
    std::vector<double> thr(s->L);
    for (int l = 0; l < s->L; l++) thr[l] = (double)s->lambdas[l] / ((double)(s->rhos[l] * (float)s->P) + 0.0);
    if (int rc = sess_alloc(s, (void**)&s->d_l1thr, s->L * sizeof(double))) return rc;
    CK(cudaMemcpy(s->d_l1thr, thr.data(), thr.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
  return 0;
}

int ensure_scratch(mlease_session* s, int part_idx) {
  if (s->scratch && s->scratch_part == part_idx) return 0;
  if (int rc = csr_flush_pending(s)) return rc;
  delete s->scratch;
  s->scratch = new Batch();
  Batch* B = s->scratch;
  B->nprob = 1; B->Dt = s->Dt; B->ldx = s->ldx; B->csr = s->parts[part_idx].csr; B->has_bias = 1;
  B->h.resize(1);
  fill_problem_data(B->h[0], s->parts[part_idx]);
  s->scratch_part = part_idx;
  return batch_alloc(*B, s->num_sms);
}

double rho_eff_for_iter(mlease_session* s, int l, int iter) {
  // reducer: rho = lambdaRho[lambda] (float -> double), times rho.adapt.rate if != 1 (jobs/RegressionAdmmTrain.java:652-658);
  // rate = (float) exp(-(i-1)*coef) for i > 1 (:323-327)
  double r = (double)s->rhos[l];
  // rho.adapt.rate is a key of the per-iteration JobConf, which the driver re-creates every iteration (:286-291 ->
  // com/linkedin/mapred/AbstractAvroJob.java:101-115): the boost is seen by the reducers of iteration 1 only (:313-316)
  float rate = (iter == 1 && s->boost_rate > 0.f) ? s->boost_rate : 1.0f;
  if (iter > 1 && s->cfg.rho_adapt_coefficient > 0) rate = (float)std::exp(-(iter - 1) * s->cfg.rho_adapt_coefficient);
  if (rate != 1.0f) r = r * (double)rate;
  return r;
}

}  // namespace

namespace {
struct TmpDev {
  std::vector<void*> ptrs;
  ~TmpDev() { for (void* p : ptrs) cudaFree(p); }
  template <class T> int get(T** p, size_t count) {
    CK(cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T)));
    ptrs.push_back(*p);
    return 0;
  }
};
// returns a device pointer for host-or-device input (copies when the pointer is not device memory)
template <class T> int to_device(TmpDev& t, const T* in, size_t count, const T** out, cudaStream_t st) {
  if (!in) { *out = nullptr; return 0; }
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, in);
  if (e == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged)) { *out = in; return 0; }
  cudaGetLastError();
  T* d;
  if (int rc = t.get(&d, count)) return rc;
  CK(cudaMemcpyAsync(d, in, count * sizeof(T), cudaMemcpyDefault, st));
  *out = d;
  return 0;
}

__global__ void naive_init_kernel(const Problem* probs, const double* m, const double* q) {
  const Problem& pb = probs[blockIdx.x];
  for (int k = threadIdx.x; k < pb.ldx; k += blockDim.x) { pb.beta[k] = 0.0; pb.m[k] = m[k]; pb.q[k] = q[k]; }
}
__global__ void gather_beta_kernel(const Problem* probs, int Dt, double* out, const unsigned char* mask) {
  const Problem& pb = probs[blockIdx.x];
  for (int k = threadIdx.x; k < Dt; k += blockDim.x)
    out[(size_t)blockIdx.x * Dt + k] = (!mask || mask[(size_t)blockIdx.x * Dt + k]) ? pb.beta[k] : 0.0;
}
// mask[b][c] = 1 for every feature listed in some row of problem b (+ the intercept)
__global__ void naive_present_kernel(const Problem* probs, int Dt, int has_bias, unsigned char* mask) {
  const Problem& pb = probs[blockIdx.x];
  unsigned char* mk = mask + (size_t)blockIdx.x * Dt;
  const long long j0 = pb.rowptr[0], j1 = pb.rowptr[pb.n];
  for (long long j = j0 + threadIdx.x; j < j1; j += blockDim.x) mk[pb.colidx[j]] = 1;
  if (threadIdx.x == 0 && has_bias) mk[Dt - 1] = 1;
}
__global__ void gather_i64_kernel(const long long* src, const long long* idx, int n, long long* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = src[idx[i]];
}
}  // namespace

// ============================================================================================
extern "C" {

const char* mlease_last_error(void) { return g_err.c_str(); }
int mlease_abi_version(void) { return 2; }

int mlease_session_create(const mlease_admm_config* cfg, mlease_session** out) {
  if (!cfg || !out) return fail(MLEASE_ERR_INVALID, "null argument");
  if (cfg->regularizer != 1 && cfg->regularizer != 2) return fail(MLEASE_ERR_INVALID, "Only L1 and L2 regularization supported!");
  if (cfg->num_blocks <= 0 || cfg->num_features <= 0 || cfg->num_lambdas <= 0 || !cfg->lambdas)
    return fail(MLEASE_ERR_INVALID, "num.blocks, num_features and lambda must be set");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(MLEASE_ERR_CUDA, std::string("no CUDA device: this library has no CPU fallback (") + cudaGetErrorString(e) + ")");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(MLEASE_ERR_INVALID, "bad device ordinal");
  CK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail(MLEASE_ERR_CUDA, "this build targets sm_100a (B200) only; found sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
  mlease_session* s = new mlease_session();
  s->cfg = *cfg;
  s->L = cfg->num_lambdas; s->P = cfg->num_blocks; s->Dg = cfg->num_features; s->Dt = s->Dg + 1;
  s->ldx = round_up(s->Dt, 4);
  s->lambdas.assign(cfg->lambdas, cfg->lambdas + s->L);
  for (int a = 0; a < s->L; a++)
    for (int b = a + 1; b < s->L; b++)
      if (s->lambdas[a] == s->lambdas[b]) { delete s; return fail(MLEASE_ERR_INVALID, "duplicate lambda"); }
  s->rhos.resize(s->L);
  for (int l = 0; l < s->L; l++) s->rhos[l] = cfg->rhos ? cfg->rhos[l] : (s->lambdas[l] <= 100 ? 1.0f : 10.0f);
  if (cfg->lambda_map) s->lambda_map.assign(cfg->lambda_map, cfg->lambda_map + s->Dg);
  s->cfg.lambdas = nullptr; s->cfg.rhos = nullptr; s->cfg.lambda_map = nullptr;
  s->stream = reinterpret_cast<cudaStream_t>(cfg->stream);
  s->num_sms = prop.multiProcessorCount;
  s->xtol = cfg->newton_xtol > 0 ? cfg->newton_xtol : 2e-7;
  s->max_newton = cfg->max_newton > 0 ? cfg->max_newton : 50;
  if (cudaMallocHost((void**)&s->h_flag, 64) != cudaSuccess || cudaMallocHost((void**)&s->h_small, (size_t)(8 * s->L + 8) * sizeof(double)) != cudaSuccess) {
    delete s;
    return fail(MLEASE_ERR_CUDA, "cudaMallocHost failed");
  }
  void* f;
  if (cudaMalloc(&f, 64) != cudaSuccess) { delete s; return fail(MLEASE_ERR_CUDA, "cudaMalloc failed"); }
  s->owned.push_back(f);
  s->d_flag = (int*)f;
  *out = s;
  return 0;
}

int mlease_session_destroy(mlease_session* s) {
  if (!s) return 0;
  cudaSetDevice(s->cfg.device);
  cudaDeviceSynchronize();
  delete s;
  return 0;
}

static int add_common(mlease_session* s, PartData& pd, const int32_t* response, const float* weight, const float* offset) {
  const long long n = pd.n;
  void *y, *w, *o;
  if (int rc = sess_alloc(s, &y, n)) return rc;
  if (int rc = sess_alloc(s, &w, n * 4)) return rc;
  if (int rc = sess_alloc(s, &o, n * 4)) return rc;
  TmpDev t;   // staging copies of the caller's arrays: freed on every return path
  int* tmp_r = nullptr; float *tmp_w = nullptr, *tmp_o = nullptr;
  if (int rc = t.get(&tmp_r, (size_t)std::max<long long>(n, 1))) return rc;
  CK(cudaMemcpyAsync(tmp_r, response, n * 4, cudaMemcpyDefault, s->stream));
  if (weight) { if (int rc = t.get(&tmp_w, (size_t)std::max<long long>(n, 1))) return rc; CK(cudaMemcpyAsync(tmp_w, weight, n * 4, cudaMemcpyDefault, s->stream)); }
  if (offset) { if (int rc = t.get(&tmp_o, (size_t)std::max<long long>(n, 1))) return rc; CK(cudaMemcpyAsync(tmp_o, offset, n * 4, cudaMemcpyDefault, s->stream)); }
  CK(cudaMemsetAsync(s->d_flag, 0, 4, s->stream));
  if (n > 0)
    convert_labels_kernel<<<(int)std::min<long long>((n + 255) / 256, 4096), 256, 0, s->stream>>>(n, tmp_r, tmp_w, tmp_o, (signed char*)y, (float*)w, (float*)o, s->d_flag);
  CK(cudaMemcpyAsync(s->h_flag, s->d_flag, 4, cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  if (*s->h_flag & 1) return fail(MLEASE_ERR_INVALID, "response (only 1, 0, -1 are allowed)");
  if (*s->h_flag & 2) return fail(MLEASE_ERR_INVALID, "weight cannot < 0");
  pd.y = (signed char*)y; pd.w = (float*)w; pd.o = (float*)o;
  if (n > 0) {
    CK(cudaMemsetAsync(s->d_flag, 0, 4, s->stream));
    absmax_kernel<<<(int)std::min<long long>((n + 255) / 256, 2048), 256, 0, s->stream>>>(n, (const float*)w, (unsigned*)s->d_flag);
    CK(cudaMemcpyAsync(s->h_flag, s->d_flag, 4, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    std::memcpy(&pd.wmax, s->h_flag, 4);
  }
  return 0;
}

int mlease_add_partition_dense(mlease_session* s, int32_t pid, int64_t nrows, const float* X, int64_t ldx_in, const int32_t* response,
                               const float* weight, const float* offset) {
  if (!s || !X || !response || nrows <= 0) return fail(MLEASE_ERR_INVALID, "bad argument (null pointer or empty partition)");
  if (s->batch) return fail(MLEASE_ERR_STATE, "partitions must be added before the first ADMM call");
  if (pid < 0 || pid >= s->P) return fail(MLEASE_ERR_INVALID, "Map key is wrong! key has to be in the range of [0,numPartitions-1].");
  if (find_part(s, pid) >= 0) return fail(MLEASE_ERR_INVALID, "partition added twice");
  if (s->cfg.binary_feature) return fail(MLEASE_ERR_INVALID, "binary.feature needs CSR input (every listed feature counts as 1)");
  if (ldx_in < s->Dg) return fail(MLEASE_ERR_INVALID, "ldx < num_features");
  CK(cudaSetDevice(s->cfg.device));
  PartData pd;
  pd.pid = pid; pd.n = nrows; pd.csr = false;
  void* x;
  CK(cudaMalloc(&x, (size_t)nrows * s->ldx * sizeof(float)));
  s->owned.push_back(x);
  pd.X = (float*)x;
  {
    cudaPointerAttributes pa;
    const bool on_device = cudaPointerGetAttributes(&pa, X) == cudaSuccess && (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    if (on_device) {
      CK(cudaMemcpy2DAsync(pd.X, (size_t)s->ldx * 4, X, (size_t)ldx_in * 4, (size_t)s->Dg * 4, (size_t)nrows, cudaMemcpyDeviceToDevice, s->stream));
    } else {
      // Host source: a pitched 2-D DMA of 4 KB rows runs far below PCIe speed, so stream contiguous chunks into two
      // staging buffers on a copy stream and repack them into the padded layout on the compute stream.
      const long long chunk_rows = std::max<long long>(1, (128LL << 20) / (ldx_in * 4));
      struct Staging {   // two staging buffers + their events + the copy stream, released on every return path
        float* buf[2] = {nullptr, nullptr};
        cudaEvent_t h2d_done[2] = {nullptr, nullptr}, repack_done[2] = {nullptr, nullptr};
        cudaStream_t cs = nullptr;
        ~Staging() {
          for (int b = 0; b < 2; b++) { if (buf[b]) cudaFree(buf[b]); if (h2d_done[b]) cudaEventDestroy(h2d_done[b]); if (repack_done[b]) cudaEventDestroy(repack_done[b]); }
          if (cs) cudaStreamDestroy(cs);
        }
      } sg;
      CK(cudaStreamCreateWithFlags(&sg.cs, cudaStreamNonBlocking));
      for (int b = 0; b < 2; b++) {
        CK(cudaMalloc((void**)&sg.buf[b], (size_t)chunk_rows * ldx_in * 4));
        CK(cudaEventCreateWithFlags(&sg.h2d_done[b], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sg.repack_done[b], cudaEventDisableTiming));
      }
      int ci = 0;
      for (long long r0 = 0; r0 < nrows; r0 += chunk_rows, ci++) {
        const int b = ci & 1;
        const long long rows = std::min(chunk_rows, (long long)nrows - r0);
        if (ci >= 2) CK(cudaStreamWaitEvent(sg.cs, sg.repack_done[b], 0));
        const size_t bytes = ((size_t)(rows - 1) * ldx_in + s->Dg) * 4;
        CK(cudaMemcpyAsync(sg.buf[b], X + r0 * ldx_in, bytes, cudaMemcpyHostToDevice, sg.cs));
        CK(cudaEventRecord(sg.h2d_done[b], sg.cs));
        CK(cudaStreamWaitEvent(s->stream, sg.h2d_done[b], 0));
        repack_rows_kernel<<<2048, 256, 0, s->stream>>>(pd.X + r0 * s->ldx, s->ldx, sg.buf[b], ldx_in, rows, s->Dg);
        CK(cudaEventRecord(sg.repack_done[b], s->stream));
      }
      CK(cudaStreamSynchronize(sg.cs));
      CK(cudaStreamSynchronize(s->stream));
    }
  }
  fill_bias_pad_kernel<<<1024, 256, 0, s->stream>>>(pd.X, nrows, s->ldx, s->Dg, 1);
  if (int rc = add_common(s, pd, response, weight, offset)) return rc;
  s->parts.push_back(pd);
  s->any_dense = true;
  return 0;
}

// Checks and derived lists of one uploaded CSR partition (feature range, |value| max, block-major Gram list, K1 segment
// lists). Runs on s->stream; mlease_add_partition_csr defers it by one call so that it overlaps the next partition's H2D copy.
static int csr_build_layout(mlease_session* s, PartData& pd) {
  if (pd.nnz <= 0) return 0;
  const long long nrows = pd.n;
  const std::string who = "partition " + std::to_string(pd.pid) + ": ";
  CK(cudaMemsetAsync(s->d_flag, 0, 4, s->stream));
  check_csr_kernel<<<(int)std::min<long long>((pd.nnz + 255) / 256, 4096), 256, 0, s->stream>>>(pd.nnz, pd.colidx, pd.vals, s->Dg, s->cfg.binary_feature, s->d_flag);
  CK(cudaMemcpyAsync(s->h_flag, s->d_flag, 4, cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  if (*s->h_flag) return fail(MLEASE_ERR_INVALID, who + "feature index out of range");
  CK(cudaMemsetAsync(s->d_flag, 0, 4, s->stream));
  absmax_kernel<<<(int)std::min<long long>((pd.nnz + 255) / 256, 2048), 256, 0, s->stream>>>(pd.nnz, pd.vals, (unsigned*)s->d_flag);
  CK(cudaMemcpyAsync(s->h_flag, s->d_flag, 4, cudaMemcpyDeviceToHost, s->stream));
  CK(cudaMemsetAsync(s->d_flag + 1, 0, 4, s->stream));
  check_rows_sorted_kernel<<<(int)std::min<long long>((nrows + 255) / 256, 4096), 256, 0, s->stream>>>(nrows, pd.rowptr, pd.colidx, s->d_flag + 1);
  CK(cudaMemcpyAsync(s->h_flag + 1, s->d_flag + 1, 4, cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  std::memcpy(&pd.vmax, s->h_flag, 4);
  pd.csr_unique = s->h_flag[1] ? 0 : 1;
  if (pd.csr_unique && pd.nnz < (1LL << 32) - 64) {   // the Gram producers index the entry list with 32 bits
    pd.nblk128 = round_up(s->ldx, 128) / 128;
    pd.bm_groups = (nrows + 31) / 32;
    void *bo, *bk, *bv;
    if (int rc = sess_alloc(s, &bo, ((size_t)pd.nblk128 * pd.bm_groups + 1) * sizeof(long long))) return rc;
    if (int rc = sess_alloc(s, &bk, (size_t)pd.nnz * sizeof(unsigned short))) return rc;
    if (int rc = sess_alloc(s, &bv, (size_t)pd.nnz * sizeof(float))) return rc;
    CK(csr_bm_offsets(nrows, pd.rowptr, pd.colidx, pd.nblk128, pd.bm_groups, (long long*)bo, s->stream));
    CK(csr_bm_fill(nrows, pd.rowptr, pd.colidx, pd.vals, pd.nblk128, pd.bm_groups, (const long long*)bo, (unsigned short*)bk, (float*)bv, s->stream));
    pd.bm_offs = (long long*)bo; pd.bm_keys = (unsigned short*)bk; pd.bm_vals = (float*)bv;
    // segment lists of the fused multi-lambda K1.  MLEASE_NO_FUSED_K1 is a test hook: without the lists batch_alloc falls back to
    // the per-problem CSR kernels, which production runs for NaiveTrain, for more than 4 lambdas and when the fused kernel's
    // shared memory overflows; the hook lets the tests reach them on small inputs
    int S = 0, rows = 0, LP = 0; size_t smem = 0;
    if (!getenv("MLEASE_NO_FUSED_K1") && k1f_plan(nrows, s->ldx, s->L, s->num_sms, &S, &rows, &LP, &smem)) {
      CK(k1f_build(nrows, s->Dg, pd.nnz, pd.rowptr, pd.colidx, pd.vals, S, rows, &pd.sg_ngrp, &pd.sg_perm, &pd.sg_depth, &pd.sg_goff, &pd.sg_row16,
                   &pd.sg_val, &pd.sg_total, s->stream));
      pd.sg_S = S; pd.sg_rows = rows;
      s->owned.push_back(pd.sg_perm); s->owned.push_back(pd.sg_depth); s->owned.push_back(pd.sg_goff);
      s->owned.push_back(pd.sg_row16); s->owned.push_back(pd.sg_val);
    }
  }
  return 0;
}

static int csr_flush_pending(mlease_session* s) {
  if (s->pending_csr < 0) return 0;
  const int idx = s->pending_csr;
  s->pending_csr = -1;
  return csr_build_layout(s, s->parts[idx]);
}

// The big arrays travel on copy_stream while the previous partition's lists are built on s->stream; a malformed colidx of
// partition p is therefore reported by the NEXT session call (add_partition / begin / fit), with the partition id in the message.
int mlease_add_partition_csr(mlease_session* s, int32_t pid, int64_t nrows, const int64_t* rowptr, const int32_t* colidx, const float* vals,
                             const int32_t* response, const float* weight, const float* offset) {
  if (!s || !rowptr || !response || nrows <= 0) return fail(MLEASE_ERR_INVALID, "bad argument (null pointer or empty partition)");
  if (s->batch) return fail(MLEASE_ERR_STATE, "partitions must be added before the first ADMM call");
  if (pid < 0 || pid >= s->P) return fail(MLEASE_ERR_INVALID, "Map key is wrong! key has to be in the range of [0,numPartitions-1].");
  if (find_part(s, pid) >= 0) return fail(MLEASE_ERR_INVALID, "partition added twice");
  CK(cudaSetDevice(s->cfg.device));
  if (!s->copy_stream) {
    CK(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&s->copy_ev, cudaEventDisableTiming));
    // the list builders take their temporaries from the device's stream-ordered pool: keep them cached between partitions
    cudaMemPool_t mp;
    if (cudaDeviceGetDefaultMemPool(&mp, s->cfg.device) == cudaSuccess) {
      unsigned long long keep = 8ULL << 30;
      cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  // the inputs are ready in the order of the session stream (they may be device arrays a kernel on that stream is still writing)
  CK(cudaEventRecord(s->copy_ev, s->stream));
  CK(cudaStreamWaitEvent(s->copy_stream, s->copy_ev, 0));
  PartData pd;
  pd.pid = pid; pd.n = nrows; pd.csr = true;
  long long ends[2];
  CK(cudaMemcpyAsync(&ends[0], rowptr, 8, cudaMemcpyDefault, s->copy_stream));
  CK(cudaMemcpyAsync(&ends[1], rowptr + nrows, 8, cudaMemcpyDefault, s->copy_stream));
  CK(cudaStreamSynchronize(s->copy_stream));
  if (ends[0] != 0) return fail(MLEASE_ERR_INVALID, "rowptr[0] must be 0");
  if (ends[1] < 0) return fail(MLEASE_ERR_INVALID, "rowptr[nrows] < 0");
  pd.nnz = ends[1];
  if (pd.nnz > 0 && (!colidx || !vals)) return fail(MLEASE_ERR_INVALID, "null colidx/vals");
  const bool trace = getenv("MLEASE_UPLOAD_TRACE") != nullptr;   // per-call host timings on stderr (diagnostics)
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  if (int rc = add_common(s, pd, response, weight, offset)) return rc;   // label checks first: nothing is in flight when they fail
  const double t1 = now();
  void *rp, *ci, *vv;
  if (int rc = sess_alloc(s, &rp, (nrows + 1) * 8)) return rc;
  if (int rc = sess_alloc(s, &ci, pd.nnz * 4)) return rc;
  if (int rc = sess_alloc(s, &vv, pd.nnz * 4)) return rc;
  pd.rowptr = (long long*)rp; pd.colidx = (int*)ci; pd.vals = (float*)vv;
  cudaError_t ce = cudaMemcpyAsync(rp, rowptr, (nrows + 1) * 8, cudaMemcpyDefault, s->copy_stream);
  if (ce == cudaSuccess && pd.nnz > 0) ce = cudaMemcpyAsync(ci, colidx, pd.nnz * 4, cudaMemcpyDefault, s->copy_stream);
  if (ce == cudaSuccess && pd.nnz > 0) ce = cudaMemcpyAsync(vv, vals, pd.nnz * 4, cudaMemcpyDefault, s->copy_stream);
  const double t2 = now();
  const int rc_prev = ce == cudaSuccess ? csr_flush_pending(s) : 0;      // overlaps the copies above
  const double t3 = now();
  const cudaError_t cs = cudaStreamSynchronize(s->copy_stream);          // the caller's buffers are free again on every return path
  if (trace)
    fprintf(stderr, "[mlease upload] partition %d: labels %.1f ms, alloc + enqueue %.1f ms, previous partition's lists %.1f ms, copy wait %.1f ms\n",
            pid, (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3, (now() - t3) * 1e3);
  CK(ce);
  CK(cs);
  if (rc_prev) return rc_prev;
  s->parts.push_back(pd);
  s->pending_csr = (int)s->parts.size() - 1;
  s->any_csr = true;
  return 0;
}

static int admm_begin_impl(mlease_session* s, const double* z0, float boost_rate) {
  if (!s) return fail(MLEASE_ERR_INVALID, "null session");
  CK(cudaSetDevice(s->cfg.device));
  if (int rc = finalize(s)) return rc;
  s->boost_rate = z0 ? boost_rate : 0.f;
  s->iter = 0; s->liblinear_eps = 0.01f; s->mindiff = 99999999; s->last_maxdiff = 0;
  for (int l = 0; l < s->L; l++) s->h_small[l] = rho_eff_for_iter(s, l, 1);
  CK(cudaMemcpyAsync(s->d_rho, s->h_small, s->L * sizeof(double), cudaMemcpyHostToDevice, s->stream));
  int launches = 0;
  CK(admm_reset(s->batch->d, s->batch->nprob, s->L, s->d_z, s->ldx, s->d_rho, s->stream, &launches));
  if (z0) {
    std::vector<double> zh((size_t)s->L * s->ldx, 0.0);
    for (int l = 0; l < s->L; l++) std::memcpy(&zh[(size_t)l * s->ldx], z0 + (size_t)l * s->Dt, (size_t)s->Dt * sizeof(double));
    CK(cudaMemcpyAsync(s->d_z, zh.data(), zh.size() * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CK(admm_init(s->batch->d, s->batch->nprob, s->d_z, s->ldx, s->stream, &launches));
    CK(cudaStreamSynchronize(s->stream));   // zh is a stack-lifetime buffer
  }
  CK(cudaStreamSynchronize(s->stream));
  s->cnt.launches += launches;
  s->rho_fact.assign(s->L, -1.0);
  s->begun = true;
  return 0;
}

int mlease_admm_begin(mlease_session* s) { return admm_begin_impl(s, nullptr, 0.f); }

int mlease_admm_begin_initialized(mlease_session* s, const double* z0, float boost_rate) {
  if (!z0) return fail(MLEASE_ERR_INVALID, "null z0");
  if (!(boost_rate > 0.f)) return fail(MLEASE_ERR_INVALID, "initialize.boost.rate must be > 0 to start from a model");
  if (s && s->cfg.regularizer != 2) return fail(MLEASE_ERR_INVALID, "mean-model initialization is an L2 feature (jobs/RegressionAdmmTrain.java:236)");
  return admm_begin_impl(s, z0, boost_rate);
}

int mlease_admm_local_step(mlease_session* s, double* exchange_dev) {
  if (!s || !exchange_dev) return fail(MLEASE_ERR_INVALID, "null argument");
  if (!s->begun) return fail(MLEASE_ERR_STATE, "mlease_admm_begin was not called");
  CK(cudaSetDevice(s->cfg.device));
  s->iter++;
  const int i = s->iter;
  // tolerance schedule: control only (jobs/RegressionAdmmTrain.java:338-346)
  if (i > 1 && s->mindiff < 0.001 && !s->cfg.aggressive_decay) s->liblinear_eps = s->liblinear_eps / 10;
  else if (s->cfg.aggressive_decay && i > 5) s->liblinear_eps = s->liblinear_eps / 10;
  int invalidate = 0;
  for (int l = 0; l < s->L; l++) {
    const double r = rho_eff_for_iter(s, l, i);
    if (r != s->rho_fact[l]) invalidate = 1;   // prior precision changed -> stale factors are for another H
    s->rho_fact[l] = r;
  }
  int same_rho = 1;   // cold start: equal rho across lambdas means equal Hessians (H = G + rho I at beta = 0)
  for (int l = 1; l < s->L; l++) if (s->rho_fact[l] != s->rho_fact[0]) same_rho = 0;
  const int nc_before = s->cnt.not_converged;
  if (int rc = batch_xupdate(*s->batch, s->stream, s->xtol, s->max_newton, s->cfg.hessian_policy, invalidate, s->h_flag, s->d_flag, s->cnt, &s->prof,
                             (i == 1 && s->L > 1 && s->boost_rate == 0.f) ? s->L : 0, same_rho)) return rc;   // sharing needs beta = 0 for every lambda
  // An x-update that ran out of Newton steps (or slots) is a failed fit: the reducer wraps any fit exception as
  // IOException("Model fitting error!") and the job dies (jobs/RegressionAdmmTrain.java:713-716); an unconverged x_p must not
  // be averaged into z silently.
  if (s->cnt.not_converged > nc_before)
    return fail(MLEASE_ERR_NUMERIC, "Model fitting error! (" + std::to_string(s->cnt.not_converged - nc_before) +
                                        " x-update(s) of iteration " + std::to_string(i) + " did not converge within max_newton = " +
                                        std::to_string(s->max_newton) + " steps)");
  int launches = 0;
  CK(admm_pack(s->batch->d, (int)s->parts.size(), s->L, s->Dt, exchange_dev, s->stream, &launches));
  s->cnt.launches += launches;
  return 0;
}

// z/u update of the iteration: enqueue (kernel + read-back of the per-lambda |z - z_prev| into pinned memory), then, after the
// caller's ONE stream synchronisation, finish (convergence scalars, stop rule :493-496).
static int consensus_enqueue(mlease_session* s, const double* exchange_sum_dev) {
  for (int l = 0; l < s->L; l++) s->h_small[l] = rho_eff_for_iter(s, l, s->iter + 1);
  CK(cudaMemcpyAsync(s->d_rho, s->h_small, s->L * sizeof(double), cudaMemcpyHostToDevice, s->stream));
  int launches = 0;
  CK(admm_consensus(s->batch->d, (int)s->parts.size(), s->L, s->Dt, s->ldx, s->P, exchange_sum_dev, s->d_z, s->d_wz, s->d_rho, s->d_diff, s->stream, &launches, s->d_l1thr));
  s->cnt.launches += launches;
  CK(cudaMemcpyAsync(s->h_small + s->L, s->d_diff, s->L * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
  return 0;
}
static void consensus_finish(mlease_session* s, double* maxdiff, int32_t* stop) {
  const double* hd = s->h_small + s->L;
  double mx = 0, mn = 99999999;
  for (int l = 0; l < s->L; l++) { mx = std::max(mx, hd[l]); mn = std::min(mn, hd[l]); }
  s->mindiff = mn; s->last_maxdiff = mx;
  if (maxdiff) *maxdiff = mx;
  const double eps = s->cfg.epsilon >= 0 ? s->cfg.epsilon : 0.0001;   // default 1e-4 (:473); 0 = never stop early
  if (stop) *stop = (mx < eps && s->liblinear_eps <= 0.00001) ? 1 : 0;   // :493-496
}

int mlease_admm_consensus(mlease_session* s, const double* exchange_sum_dev, double* maxdiff, int32_t* stop) {
  if (!s || !exchange_sum_dev) return fail(MLEASE_ERR_INVALID, "null argument");
  if (!s->begun || s->iter < 1) return fail(MLEASE_ERR_STATE, "consensus before local_step");
  CK(cudaSetDevice(s->cfg.device));
  if (int rc = consensus_enqueue(s, exchange_sum_dev)) return rc;
  CK(cudaStreamSynchronize(s->stream));
  consensus_finish(s, maxdiff, stop);
  return 0;
}

int mlease_session_set_comm(mlease_session* s, mlease_comm* comm) {
  if (!s) return fail(MLEASE_ERR_INVALID, "null session");
  s->comm = comm;
  return 0;
}

// One iteration with the exchange inside: local x-updates, all-reduce (NCCL communicator, caller's callback, or nothing for
// a single-process job), z/u update.  A rank whose fit failed still enters the collective -- with its failure counted in the
// extra last element of the buffer -- so that every rank leaves with the same error instead of the others hanging in NCCL
// (the reference: one failed reducer fails the whole iteration job, jobs/RegressionAdmmTrain.java:713-716).
static int admm_iterate_impl(mlease_session* s, mlease_allreduce_fn allreduce, void* ctx, double* maxdiff, int32_t* stop) {
  const size_t cnt = (size_t)s->L * s->Dt;
  int rc_local = mlease_admm_local_step(s, s->d_exch);
  std::string local_msg;
  if (rc_local == MLEASE_ERR_NUMERIC) local_msg = g_err;
  else if (rc_local) return rc_local;                      // CUDA / state errors are not recoverable: no collective
  const bool multi = s->comm != nullptr || allreduce != nullptr;
  if (multi) {
    // all-reduce, z/u update and both read-backs are enqueued back to back; ONE synchronisation per iteration.  (If a fit
    // failed somewhere the z/u update has run on a meaningless sum, but the job is over: every rank returns the error.)
    double* h_flag = s->h_small + 3 * s->L + 1;   // pinned
    *h_flag = rc_local ? 1.0 : 0.0;
    CK(cudaMemcpyAsync(s->d_exch + cnt, h_flag, sizeof(double), cudaMemcpyHostToDevice, s->stream));
    if (s->comm) { if (int rc = mlease_internal_allreduce(s->comm, s->d_exch, cnt + 1, (void*)s->stream)) return rc; }
    else if (allreduce(ctx, s->d_exch, cnt + 1, (void*)s->stream) != 0) return fail(MLEASE_ERR_CUDA, "all-reduce callback failed");
    double* h_failed = s->h_small + 3 * s->L + 2;
    CK(cudaMemcpyAsync(h_failed, s->d_exch + cnt, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (int rc = consensus_enqueue(s, s->d_exch)) return rc;
    CK(cudaStreamSynchronize(s->stream));
    if (rc_local) return fail(rc_local, local_msg);
    if (*h_failed > 0) return fail(MLEASE_ERR_NUMERIC, "Model fitting error! (the x-update failed on " + std::to_string((int)*h_failed) + " other rank(s))");
    consensus_finish(s, maxdiff, stop);
    return 0;
  } else if (rc_local) {
    return fail(rc_local, local_msg);
  }
  return mlease_admm_consensus(s, s->d_exch, maxdiff, stop);
}

static int check_partitions_present(mlease_session* s, bool multi) {
  if (!multi && (int)s->parts.size() != s->P)
    return fail(MLEASE_ERR_STATE, "Some models failed! (" + std::to_string(s->parts.size()) + " of " + std::to_string(s->P) +
                                      " partitions present and neither a communicator nor an all-reduce was given)");
  return 0;
}

int mlease_admm_run(mlease_session* s, int32_t num_iters, mlease_allreduce_fn allreduce, void* ctx, int32_t* iters_done) {
  if (!s) return fail(MLEASE_ERR_INVALID, "null session");
  if (int rc = mlease_admm_begin(s)) return rc;
  if (int rc = check_partitions_present(s, s->comm != nullptr || allreduce != nullptr)) return rc;
  int done = 0;
  for (int i = 1; i <= num_iters; i++) {
    double md; int32_t stop;
    if (int rc = admm_iterate_impl(s, allreduce, ctx, &md, &stop)) return rc;
    done = i;
    if (stop) break;
  }
  if (iters_done) *iters_done = done;
  return 0;
}

int mlease_admm_iterate(mlease_session* s, double* maxdiff, int32_t* stop) {
  if (!s) return fail(MLEASE_ERR_INVALID, "null session");
  if (!s->begun) return fail(MLEASE_ERR_STATE, "mlease_admm_begin was not called");
  if (int rc = check_partitions_present(s, s->comm != nullptr)) return rc;
  return admm_iterate_impl(s, nullptr, nullptr, maxdiff, stop);
}

int mlease_get_z(mlease_session* s, int32_t l, double* out) {
  if (!s || !out || l < 0 || l >= s->L || !s->batch) return fail(MLEASE_ERR_INVALID, "bad argument");
  CK(cudaSetDevice(s->cfg.device));
  CK(cudaMemcpyAsync(out, s->d_z + (size_t)l * s->ldx, s->Dt * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  return 0;
}
int mlease_get_final_model(mlease_session* s, int32_t l, float* out) {
  std::vector<double> z(s ? s->Dt : 0);
  if (int rc = mlease_get_z(s, l, z.data())) return rc;
  for (int k = 0; k < s->Dt; k++) out[k] = (float)z[k];   // models/LinearModel.java:703,716
  return 0;
}
static int get_vec(mlease_session* s, int pid, int l, int which, void* out) {
  if (!s || !out || l < 0 || l >= s->L || !s->batch) return fail(MLEASE_ERR_INVALID, "bad argument");
  const int pi = find_part(s, pid);
  if (pi < 0) return fail(MLEASE_ERR_INVALID, "partition not resident in this session");
  CK(cudaSetDevice(s->cfg.device));
  const Problem& p = s->batch->h[pi * s->L + l];
  const void* src = which == 0 ? (const void*)p.x_d : which == 1 ? (const void*)p.u_f : (const void*)p.uplusx_f;
  CK(cudaMemcpyAsync(out, src, s->Dt * (which == 0 ? 8 : 4), cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  return 0;
}
int mlease_get_x(mlease_session* s, int32_t pid, int32_t l, double* out) { return get_vec(s, pid, l, 0, out); }
int mlease_get_u(mlease_session* s, int32_t pid, int32_t l, float* out) { return get_vec(s, pid, l, 1, out); }
int mlease_get_uplusx(mlease_session* s, int32_t pid, int32_t l, float* out) { return get_vec(s, pid, l, 2, out); }

int mlease_profile(mlease_session* s, int32_t enable, double* ms4, int64_t* count4, double* k1_bytes, double* k1_emit_bytes, double* gram_flops) {
  if (!s) return fail(MLEASE_ERR_INVALID, "null session");
  if (ms4) for (int i = 0; i < 4; i++) ms4[i] = s->prof.ms[i];
  if (count4) for (int i = 0; i < 4; i++) count4[i] = s->prof.n[i];
  if (k1_bytes) *k1_bytes = s->cnt.k1_bytes;
  if (k1_emit_bytes) *k1_emit_bytes = s->cnt.k1_emit_bytes;
  if (gram_flops) *gram_flops = s->cnt.gram_flops;
  if (enable >= 0) {
    s->prof.on = enable != 0;
    if (enable == 2) { for (int i = 0; i < 4; i++) { s->prof.ms[i] = 0; s->prof.n[i] = 0; } s->cnt.k1_bytes = s->cnt.k1_emit_bytes = s->cnt.gram_flops = 0; }
  }
  return 0;
}

int mlease_get_stats(mlease_session* s, mlease_stats* out) {
  if (!s || !out) return fail(MLEASE_ERR_INVALID, "null argument");
  out->k1_passes = s->cnt.k1_passes; out->gram_builds = s->cnt.gram_builds; out->newton_steps = s->cnt.newton_steps;
  out->rejected_steps = s->cnt.rejected; out->kernel_launches = s->cnt.launches; out->not_converged = s->cnt.not_converged;
  out->last_iter_slots = s->cnt.last_slots; out->last_maxdiff = s->last_maxdiff; out->liblinear_epsilon = s->liblinear_eps;
  out->k1_shared_bytes = s->cnt.k1_shared_bytes;
  out->k1_fused = (s->batch && s->batch->k1_fused) ? 1 : 0;
  return 0;
}

// ------------------------------------------------------------------------------------------
// function-level entry points on the scratch problem
// ------------------------------------------------------------------------------------------
static int scratch_set(mlease_session* s, const double* w, const double* m, const double* q) {
  Batch* B = s->scratch;
  const Problem& p = B->h[0];
  std::vector<double> buf(3 * (size_t)s->ldx, 0.0);
  for (int k = 0; k < s->Dt; k++) { buf[k] = w[k]; buf[s->ldx + k] = m[k]; buf[2 * s->ldx + k] = q[k]; }
  for (int k = s->Dt; k < s->ldx; k++) buf[2 * s->ldx + k] = 1.0;
  CK(cudaMemcpyAsync(p.beta, buf.data(), s->ldx * 8, cudaMemcpyHostToDevice, s->stream));
  CK(cudaMemcpyAsync(p.m, buf.data() + s->ldx, s->ldx * 8, cudaMemcpyHostToDevice, s->stream));
  CK(cudaMemcpyAsync(p.q, buf.data() + 2 * s->ldx, s->ldx * 8, cudaMemcpyHostToDevice, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  return 0;
}

int mlease_objective(mlease_session* s, int32_t pid, const double* w, const double* m, const double* q, double* f, double* g, double* H,
                     int32_t tensor) {
  if (!s || !w || !m || !q) return fail(MLEASE_ERR_INVALID, "null argument");
  CK(cudaSetDevice(s->cfg.device));
  const int pi = find_part(s, pid);
  if (pi < 0) return fail(MLEASE_ERR_INVALID, "partition not resident in this session");
  if (int rc = ensure_scratch(s, pi)) return rc;
  Batch* B = s->scratch;
  if (int rc = scratch_set(s, w, m, q)) return rc;
  int launches = 0;
  CK(newton_begin(B->d, 1, 1e-8, 1, 1, 1, 0, s->stream, &launches));
  CK(batch_k1(*B, H ? 1 : 0, s->stream, &launches));
  CK(k1_reduce_decide(B->d, 1, B->Dt, s->stream, &launches));
  const Problem& p = B->h[0];
  Ctrl c;
  CK(cudaMemcpyAsync(&c, B->d_ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, s->stream));
  if (g) CK(cudaMemcpyAsync(g, p.g_acc, s->Dt * 8, cudaMemcpyDeviceToHost, s->stream));   // first evaluation is always accepted: g_acc = gradient at w
  CK(cudaStreamSynchronize(s->stream));
  if (f) *f = c.f_t;
  if (H) {
    if (!tensor && B->gram_from_csr) return fail(MLEASE_ERR_INVALID, "the SIMT debug Gram needs the dense bf16 operand, which CSR partitions with sorted unique rows do not materialise");
    if (tensor) CK(batch_gram(*B, B->d, 1, 1, 0, s->stream, &launches));
    else CK(gram_launch_simt(B->d, 1, B->Dp, 1, s->stream, &launches));
    if (tensor == 2) {
      // the inverse the Newton direction uses: split-K Gram partials + diag(q) -> fp64 Cholesky -> explicit inverse
      Ctrl c2; std::memset(&c2, 0, sizeof(c2)); c2.need_hess = 1;
      CK(cudaMemcpyAsync(B->d_ctrl, &c2, sizeof(Ctrl), cudaMemcpyHostToDevice, s->stream));
      CK(cholesky_launch(B->d, 1, B->ldh, s->stream, &launches, 0, 0, 1));
      std::vector<double> hi((size_t)B->ldh * B->ldh);
      CK(cudaMemcpyAsync(hi.data(), p.Hinv, hi.size() * 8, cudaMemcpyDeviceToHost, s->stream));
      CK(cudaMemcpyAsync(&c2, B->d_ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, s->stream));
      CK(cudaStreamSynchronize(s->stream));
      s->cnt.launches += launches;
      if (c2.fail) return fail(MLEASE_ERR_NUMERIC, "Hessian not positive definite");
      for (int i = 0; i < s->Dt; i++)
        for (int j = 0; j < s->Dt; j++) H[(size_t)i * s->Dt + j] = hi[(size_t)i * B->ldh + j];
      return 0;
    }
    const size_t per = (size_t)B->Dp * B->Dp;
    std::vector<float> hp(per * B->gram_slices);
    CK(cudaMemcpyAsync(hp.data(), p.Hpart, hp.size() * 4, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    const int Dt = s->Dt;
    for (int i = 0; i < Dt; i++)
      for (int j = 0; j <= i; j++) {
        double a = 0;
        for (int t = 0; t < B->gram_slices; t++) a += (double)hp[t * per + (size_t)i * B->Dp + j];
        if (B->gram_from_csr) a *= (double)p.gram_unscale;
        if (i == j) a += q[i];
        H[(size_t)i * Dt + j] = a;
        H[(size_t)j * Dt + i] = a;
      }
  }
  s->cnt.launches += launches;
  return 0;
}

int mlease_fit_partition(mlease_session* s, int32_t pid, double* x, const double* m, const double* q, int32_t* newton_steps) {
  if (!s || !x || !m || !q) return fail(MLEASE_ERR_INVALID, "null argument");
  CK(cudaSetDevice(s->cfg.device));
  const int pi = find_part(s, pid);
  if (pi < 0) return fail(MLEASE_ERR_INVALID, "partition not resident in this session");
  if (int rc = ensure_scratch(s, pi)) return rc;
  if (int rc = scratch_set(s, x, m, q)) return rc;
  Counters c;
  if (int rc = batch_xupdate(*s->scratch, s->stream, s->xtol, s->max_newton, s->cfg.hessian_policy, 1, s->h_flag, s->d_flag, c)) return rc;
  s->cnt.launches += c.launches; s->cnt.k1_passes += c.k1_passes; s->cnt.gram_builds += c.gram_builds;
  s->cnt.newton_steps += c.newton_steps; s->cnt.rejected += c.rejected; s->cnt.not_converged += c.not_converged;
  CK(cudaMemcpyAsync(x, s->scratch->h[0].beta, s->Dt * 8, cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  if (newton_steps) *newton_steps = (int)c.newton_steps;
  if (c.not_converged) return fail(MLEASE_ERR_NUMERIC, "Model fitting error! (Newton did not converge within max_newton steps)");
  return 0;
}

int mlease_posterior_variance(mlease_session* s, int32_t pid, const double* w, const double* q, int32_t full, double* var, double* cov) {
  if (!s || !w || !q || !var) return fail(MLEASE_ERR_INVALID, "null argument");
  if (cov && !full) return fail(MLEASE_ERR_INVALID, "the covariance matrix is only available with full = 1 (computeFullPostVar)");
  CK(cudaSetDevice(s->cfg.device));
  const int pi = find_part(s, pid);
  if (pi < 0) return fail(MLEASE_ERR_INVALID, "partition not resident in this session");
  if (int rc = ensure_scratch(s, pi)) return rc;
  Batch* B = s->scratch;
  const Problem& p = B->h[0];
  if (full && B->csr && !s->parts[pi].csr_unique)
    return fail(MLEASE_ERR_INVALID, "the full Hessian needs rows with strictly increasing column ids (llf/LogisticRegressionL2.java:277)");
  std::vector<double> zero(s->Dt, 0.0);
  if (int rc = scratch_set(s, w, zero.data(), q)) return rc;          // beta = w, q = prior precision (1 on the padding)
  TmpDev t;
  double* dvec;
  if (int rc = t.get(&dvec, (size_t)p.n)) return rc;
  int launches = 0;
  CK(postvar_rowweights(B->d, p.beta, 1, dvec, s->stream, &launches));
  if (!full) {
    // H[k] = 1/priorVar[k] + sum_i weight_i p_i (1-p_i) x_ik^2, postVar = 1/H (llf/LibLinear.java:330-333)
    CK(cudaMemcpyAsync(p.g_t, p.q, (size_t)s->ldx * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
    CK(postvar_diag(B->d, dvec, 1, p.g_t, s->stream, &launches));
    CK(cudaMemcpyAsync(var, p.g_t, (size_t)s->Dt * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    for (int k = 0; k < s->Dt; k++) var[k] = 1.0 / var[k];
    s->cnt.launches += launches;
    return 0;
  }
  // exact fp64 Hessian -> K3's factorisation and explicit inverse (llf/LibLinear.java:318-326)
  CK(postvar_hessian(B->d, B->csr, B->ldh, dvec, p.q, 1, s->stream, &launches));
  Ctrl c; std::memset(&c, 0, sizeof(c)); c.need_hess = 1;
  CK(cudaMemcpyAsync(B->d_ctrl, &c, sizeof(Ctrl), cudaMemcpyHostToDevice, s->stream));
  CK(cholesky_launch(B->d, 1, B->ldh, s->stream, &launches, 0, 1, 1));
  std::vector<double> hi((size_t)B->ldh * B->ldh);
  CK(cudaMemcpyAsync(hi.data(), p.Hinv, hi.size() * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
  CK(cudaMemcpyAsync(&c, B->d_ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  s->cnt.launches += launches;
  if (c.fail) return fail(MLEASE_ERR_NUMERIC, "Model fitting error! (Hessian not positive definite)");
  for (int i = 0; i < s->Dt; i++) {
    var[i] = hi[(size_t)i * B->ldh + i];
    if (cov) for (int j = 0; j < s->Dt; j++) cov[(size_t)i * s->Dt + j] = hi[(size_t)i * B->ldh + j];
  }
  // the stale-factor bookkeeping of the scratch problem no longer matches its Lc/Hinv: force a rebuild on its next use
  Ctrl c2; std::memset(&c2, 0, sizeof(c2));
  CK(cudaMemcpy(B->d_ctrl, &c2, sizeof(Ctrl), cudaMemcpyHostToDevice));
  B->mirror.clear();
  return 0;
}

int mlease_time_kernel(mlease_session* s, int32_t pid, int32_t which, int32_t reps, int32_t emit_scaled, float* avg_ms) {
  if (!s || !avg_ms || reps <= 0) return fail(MLEASE_ERR_INVALID, "bad argument");
  CK(cudaSetDevice(s->cfg.device));
  const int pi = find_part(s, pid);
  if (pi < 0) return fail(MLEASE_ERR_INVALID, "partition not resident in this session");
  if (int rc = ensure_scratch(s, pi)) return rc;
  Batch* B = s->scratch;
  std::vector<double> zero(s->Dt, 0.0), one(s->Dt, 1.0);
  if (int rc = scratch_set(s, zero.data(), zero.data(), one.data())) return rc;
  int launches = 0;
  CK(newton_begin(B->d, 1, 1e-8, 1, 1, 1, 0, s->stream, &launches));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  // warm-up launch (also produces the scaled copy the Gram needs)
  CK(batch_k1(*B, 1, s->stream, &launches));
  if (which == 3) {
    CK(batch_gram(*B, B->d, 1, 1, 0, s->stream, &launches));
    Ctrl c; std::memset(&c, 0, sizeof(c)); c.need_hess = 1;
    CK(cudaMemcpyAsync(B->d_ctrl, &c, sizeof(Ctrl), cudaMemcpyHostToDevice, s->stream));
  }
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaEventRecord(e0, s->stream));
  for (int r = 0; r < reps; r++) {
    if (which == 1) CK(batch_k1(*B, emit_scaled ? 1 : 0, s->stream, &launches));
    else if (which == 2) CK(batch_gram(*B, B->d, 1, 1, 0, s->stream, &launches));
    else if (which == 3) CK(cholesky_launch(B->d, 1, B->ldh, s->stream, &launches));
    else return fail(MLEASE_ERR_INVALID, "which must be 1, 2 or 3");
  }
  CK(cudaEventRecord(e1, s->stream));
  CK(cudaEventSynchronize(e1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *avg_ms = ms / reps;
  s->cnt.launches += launches;
  return 0;
}

// ------------------------------------------------------------------------------------------
// scoring / log-likelihood
// ------------------------------------------------------------------------------------------
static int need_device(int device) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(MLEASE_ERR_CUDA, std::string("no CUDA device: this library has no CPU fallback (") + cudaGetErrorString(e) + ")");
  if (device < 0 || device >= ndev) return fail(MLEASE_ERR_INVALID, "bad device ordinal");
  CK(cudaSetDevice(device));
  return 0;
}

int mlease_score(int32_t device, void* stream, int32_t Dg, int64_t nrows, const int64_t* rowptr, const int32_t* colidx, const float* vals,
                 int64_t ldx, const float* offset, const double* model, int32_t num_click_replicates, int32_t binary_feature, float* pred) {
  if (!vals || !model || !pred || nrows < 0) return fail(MLEASE_ERR_INVALID, "bad argument");
  if (int rc = need_device(device)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  TmpDev t;
  const long long* d_rp = nullptr; const int* d_ci = nullptr; const float* d_v = nullptr; const float* d_o = nullptr; const double* d_m = nullptr;
  long long nnz = nrows * ldx;
  if (colidx) {
    if (!rowptr) return fail(MLEASE_ERR_INVALID, "null rowptr");
    long long last;
    CK(cudaMemcpy(&last, rowptr + nrows, 8, cudaMemcpyDefault));
    nnz = last;
    if (int rc = to_device(t, (const long long*)rowptr, (size_t)nrows + 1, &d_rp, st)) return rc;
    if (int rc = to_device(t, colidx, (size_t)nnz, &d_ci, st)) return rc;
  }
  if (int rc = to_device(t, vals, (size_t)nnz, &d_v, st)) return rc;
  if (int rc = to_device(t, offset, (size_t)nrows, &d_o, st)) return rc;
  if (int rc = to_device(t, model, (size_t)Dg + 1, &d_m, st)) return rc;
  double b;
  CK(cudaMemcpy(&b, model + Dg, 8, cudaMemcpyDefault));
  // intercept term  -log(n - 1 + n exp(-b))  (models/LinearModel.java:243-244)
  const double ic = -std::log((double)num_click_replicates - 1 + (double)num_click_replicates * std::exp(-b));
  cudaPointerAttributes a;
  bool pred_dev = cudaPointerGetAttributes(&a, pred) == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged);
  cudaGetLastError();
  float* d_pred = pred;
  if (!pred_dev) { if (int rc = t.get(&d_pred, (size_t)nrows)) return rc; }
  CK(score_launch(Dg, nrows, d_rp, d_ci, d_v, ldx, d_o, d_m, ic, binary_feature, d_pred, st));
  if (!pred_dev) CK(cudaMemcpyAsync(pred, d_pred, (size_t)nrows * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

int mlease_test_loglik(int32_t device, void* stream, int64_t nrows, const int32_t* response, const float* pred, const float* weight,
                       int64_t combiner_block, float* out_loglik, double* out_count) {
  if (!response || !pred || !out_loglik || !out_count || nrows <= 0) return fail(MLEASE_ERR_INVALID, "bad argument");
  if (int rc = need_device(device)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  TmpDev t;
  const int* d_r; const float* d_p; const float* d_w;
  if (int rc = to_device(t, (const int*)response, (size_t)nrows, &d_r, st)) return rc;
  if (int rc = to_device(t, pred, (size_t)nrows, &d_p, st)) return rc;
  if (int rc = to_device(t, weight, (size_t)nrows, &d_w, st)) return rc;
  const bool combine = combiner_block > 0;
  const long long blk = combine ? combiner_block : 4096;
  const long long nb = (nrows + blk - 1) / blk;
  float* d_ll; double *d_bs, *d_bc; int* d_bad;
  if (int rc = t.get(&d_ll, (size_t)nrows)) return rc;
  if (int rc = t.get(&d_bs, (size_t)nb)) return rc;
  if (int rc = t.get(&d_bc, (size_t)nb)) return rc;
  if (int rc = t.get(&d_bad, 1)) return rc;
  CK(cudaMemsetAsync(d_bad, 0, 4, st));
  CK(loglik_launch(nrows, d_r, d_p, d_w, blk, d_ll, d_bs, d_bc, d_bad, st));
  std::vector<double> bs(nb), bc(nb);
  int bad = 0;
  CK(cudaMemcpyAsync(bs.data(), d_bs, nb * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(bc.data(), d_bc, nb * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (bad) return fail(MLEASE_ERR_INVALID, "response should be 1,0 or -1!");
  double sum = 0, n = 0;
  for (long long b = 0; b < nb; b++) {
    sum += combine ? (double)(float)bs[b] : bs[b];   // combiner casts its partial sum to float (jobs/RegressionTestLoglik.java:197)
    n += bc[b];
  }
  *out_loglik = (float)(sum / n);                    // reducer (:173)
  *out_count = n;
  return 0;
}

// ------------------------------------------------------------------------------------------
// RegressionNaiveTrain: K independent fits per lambda, processed in lockstep chunks.  The rows are uploaded ONCE and serve
// every lambda (the reference fans each record out once per lambda through the shuffle, jobs/RegressionNaiveTrain.java:228-241).
// ------------------------------------------------------------------------------------------
int mlease_naive_train(int32_t device, void* stream, int32_t K, int32_t Dg, const int64_t* key_rowstart, const int64_t* rowptr,
                       const int32_t* colidx, const float* vals, int64_t ldx_in, const int32_t* response, const float* weight,
                       const float* offset, int32_t L, const float* lambdas, const float* lambda_map, float prior_mean,
                       int32_t penalize_intercept, int32_t has_intercept, int32_t data_size_threshold, int32_t binary_feature,
                       double* out_model, int32_t* skipped) {
  if (K <= 0 || Dg <= 0 || L <= 0 || !lambdas || !key_rowstart || !vals || !response || !out_model) return fail(MLEASE_ERR_INVALID, "bad argument");
  const bool csr = rowptr != nullptr;
  if (csr && !colidx) return fail(MLEASE_ERR_INVALID, "null colidx");
  if (!csr && binary_feature) return fail(MLEASE_ERR_INVALID, "binary.feature needs CSR input (every listed feature counts as 1)");
  if (!csr && ldx_in < Dg) return fail(MLEASE_ERR_INVALID, "ldx < num_features");
  if (int rc = need_device(device)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(MLEASE_ERR_CUDA, "this build targets sm_100a (B200) only");
  const int Dt = Dg + 1, ldx = round_up(Dt, 4);
  // MLEASE_DEBUG: wall-clock of the host-side phases (allocation, ingest, solve, read-back)
  const bool dbg = getenv("MLEASE_DEBUG") != nullptr;
  auto t_last = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!dbg) return;
    cudaStreamSynchronize((cudaStream_t)stream);
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[mlease] naive_train %-12s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
    t_last = now;
  };
  std::vector<long long> krs(K + 1);
  CK(cudaMemcpy(krs.data(), key_rowstart, (size_t)(K + 1) * 8, cudaMemcpyDefault));
  const long long ntot = krs[K];
  for (int k = 0; k < K; k++) if (krs[k + 1] < krs[k]) return fail(MLEASE_ERR_INVALID, "key_rowstart must be non-decreasing");
  TmpDev t;
  float* dX = nullptr; signed char* dy; float *dw, *dofs; int* dflag; int* hflag;
  const long long* d_rp = nullptr; const int* d_ci = nullptr; float* d_v = nullptr;
  std::vector<long long> key_nnz0(K + 1, 0);   // CSR: rowptr at the key boundaries
  int csr_unique = 0;
  if (int rc = t.get(&dy, (size_t)ntot)) return rc;
  if (int rc = t.get(&dw, (size_t)ntot)) return rc;
  if (int rc = t.get(&dofs, (size_t)ntot)) return rc;
  if (int rc = t.get(&dflag, 16)) return rc;
  CK(cudaMallocHost((void**)&hflag, 64));
  struct HF { int* p; ~HF() { cudaFreeHost(p); } } hf{hflag};
  lap("alloc");
  if (!csr) {
    if (int rc = t.get(&dX, (size_t)ntot * ldx)) return rc;
    // rows are re-pitched from ldx_in to ldx floats: a kernel for device input (the copy engine moves 1 KB rows slowly),
    // a pitched copy for host input
    cudaPointerAttributes pa;
    const bool on_device = cudaPointerGetAttributes(&pa, vals) == cudaSuccess && (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    if (on_device) repack_rows_kernel<<<4096, 256, 0, st>>>(dX, ldx, vals, ldx_in, ntot, Dg);
    else CK(cudaMemcpy2DAsync(dX, (size_t)ldx * 4, vals, (size_t)ldx_in * 4, (size_t)Dg * 4, (size_t)ntot, cudaMemcpyDefault, st));
    fill_bias_pad_kernel<<<1024, 256, 0, st>>>(dX, ntot, ldx, Dg, has_intercept ? 1 : 0);
  } else {
    if (int rc = to_device(t, (const long long*)rowptr, (size_t)ntot + 1, &d_rp, st)) return rc;
    long long nnz = 0, first = 0;
    CK(cudaMemcpyAsync(&nnz, d_rp + ntot, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&first, d_rp, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (first != 0) return fail(MLEASE_ERR_INVALID, "rowptr[0] must be 0");
    if (int rc = to_device(t, colidx, (size_t)nnz, &d_ci, st)) return rc;
    // values are copied even when they already live on the device: binary.feature rewrites them
    if (int rc = t.get(&d_v, (size_t)std::max<long long>(nnz, 1))) return rc;
    CK(cudaMemcpyAsync(d_v, vals, (size_t)nnz * 4, cudaMemcpyDefault, st));
    CK(cudaMemsetAsync(dflag, 0, 8, st));
    if (nnz > 0) {
      check_csr_kernel<<<(int)std::min<long long>((nnz + 255) / 256, 4096), 256, 0, st>>>(nnz, d_ci, d_v, Dg, binary_feature, dflag);
      check_rows_sorted_kernel<<<(int)std::min<long long>((ntot + 255) / 256, 4096), 256, 0, st>>>(ntot, d_rp, d_ci, dflag + 1);
    }
    CK(cudaMemcpyAsync(hflag, dflag, 8, cudaMemcpyDeviceToHost, st));
    // rowptr at the key boundaries (nnz per key for the cost model and the byte accounting)
    long long* d_kn; long long* d_krs;
    if (int rc = t.get(&d_kn, (size_t)K + 1)) return rc;
    if (int rc = t.get(&d_krs, (size_t)K + 1)) return rc;
    CK(cudaMemcpyAsync(d_krs, krs.data(), (size_t)(K + 1) * 8, cudaMemcpyHostToDevice, st));
    gather_i64_kernel<<<(K + 256) / 256, 256, 0, st>>>(d_rp, d_krs, K + 1, d_kn);
    CK(cudaMemcpyAsync(key_nnz0.data(), d_kn, (size_t)(K + 1) * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (hflag[0]) return fail(MLEASE_ERR_INVALID, "feature index out of range");
    csr_unique = hflag[1] ? 0 : 1;
  }
  lap("ingest X");
  {
    const int* d_r; const float *d_wi, *d_oi;
    if (int rc = to_device(t, (const int*)response, (size_t)ntot, &d_r, st)) return rc;
    if (int rc = to_device(t, weight, (size_t)ntot, &d_wi, st)) return rc;
    if (int rc = to_device(t, offset, (size_t)ntot, &d_oi, st)) return rc;
    CK(cudaMemsetAsync(dflag, 0, 4, st));
    convert_labels_kernel<<<(int)std::min<long long>((ntot + 255) / 256, 4096), 256, 0, st>>>(ntot, d_r, d_wi, d_oi, dy, dw, dofs, dflag);
    CK(cudaMemcpyAsync(hflag, dflag, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (*hflag & 1) return fail(MLEASE_ERR_INVALID, "response (only 1, 0, -1 are allowed)");
    if (*hflag & 2) return fail(MLEASE_ERR_INVALID, "weight cannot < 0");
  }
  lap("labels");
  std::vector<float> lm;
  if (lambda_map) { lm.resize(Dg); CK(cudaMemcpy(lm.data(), lambda_map, (size_t)Dg * 4, cudaMemcpyDefault)); }
  std::vector<float> lams(L);
  CK(cudaMemcpy(lams.data(), lambdas, (size_t)L * 4, cudaMemcpyDefault));
  for (size_t e = 0; e < (size_t)L * K * Dt; e++) out_model[e] = 0.0;
  std::vector<int> todo;
  for (int k = 0; k < K; k++) {
    const long long nk = krs[k + 1] - krs[k];
    if (skipped) skipped[k] = 0;
    if (nk < data_size_threshold || nk <= 0) { if (skipped) skipped[k] = 1; }   // "data size < threshold": no model (:379-382)
    else todo.push_back(k);
  }
  // chunk size bounded by memory: Xt (n*Dp*2) + Hpart + Lc per problem
  const int Dp = round_up(ldx, 128), ldh = round_up(Dt, 32);
  size_t free_b, total_b;
  CK(cudaMemGetInfo(&free_b, &total_b));
  Counters cnt;
  size_t pos = 0;
  while (pos < todo.size()) {
    size_t bytes = 0;
    size_t end = pos;
    while (end < todo.size() && end - pos < 16384) {
      const long long nk = krs[todo[end] + 1] - krs[todo[end]];
      const size_t need = (size_t)nk * Dp * 2 + (size_t)Dp * Dp * 4 + 3 * (size_t)ldh * ldh * 8 + 2 * (size_t)ldh * 32 * 8 + 64 * (size_t)ldx;
      if (end > pos && bytes + need > free_b / 2) break;
      bytes += need;
      end++;
    }
    Batch B;
    B.nprob = (int)(end - pos); B.Dt = Dt; B.ldx = ldx; B.csr = csr; B.has_bias = has_intercept ? 1 : 0;
    B.h.resize(B.nprob);
    for (int b = 0; b < B.nprob; b++) {
      const int k = todo[pos + b];
      Problem& p = B.h[b];
      std::memset(&p, 0, sizeof(Problem));
      p.n = krs[k + 1] - krs[k];
      p.y = dy + krs[k]; p.w = dw + krs[k]; p.o = dofs + krs[k];
      if (csr) {
        // a key = a row range of the one CSR: the row pointers keep their absolute offsets into colidx / vals
        p.rowptr = d_rp + krs[k]; p.colidx = d_ci; p.vals = d_v; p.nnz_hint = key_nnz0[k + 1] - key_nnz0[k]; p.csr_unique = csr_unique;
      } else {
        p.X = dX + (size_t)krs[k] * ldx;
      }
    }
    if (int rc = batch_alloc(B, prop.multiProcessorCount)) return rc;
    lap("batch_alloc");
    double *dm, *dq, *dout; unsigned char* dmask = nullptr;
    if (int rc = t.get(&dm, (size_t)ldx)) return rc;
    if (int rc = t.get(&dq, (size_t)ldx)) return rc;
    if (int rc = t.get(&dout, (size_t)B.nprob * Dt)) return rc;
    if (csr) {
      // features absent from a key's rows are not part of its dataset, hence not of its model (llf/LibLinear.java:343-350;
      // no priorMean map is passed by NaiveTrain, so :374-383 adds nothing): mask them out of the dense result
      if (int rc = t.get(&dmask, (size_t)B.nprob * Dt)) return rc;
      CK(cudaMemsetAsync(dmask, 0, (size_t)B.nprob * Dt, st));
      naive_present_kernel<<<B.nprob, 256, 0, st>>>(B.d, Dt, has_intercept ? 1 : 0, dmask);
    }
    std::vector<double> xs((size_t)B.nprob * Dt);
    for (int l = 0; l < L; l++) {
      // prior (jobs/RegressionNaiveTrain.java:333-343,395): variance 1/lambdaMap[k] for listed features, 1/lambda otherwise,
      // 100000 for the intercept unless penalised; mean prior.mean; the fit starts at 0 (null initParam)
      const float lambda = lams[l];
      std::vector<double> q(ldx, 1.0), m(ldx, 0.0);
      for (int k = 0; k < Dg; k++) {
        q[k] = (!lm.empty() && lm[k] > 0.f) ? 1.0 / (1.0 / (double)lm[k]) : 1.0 / (1.0 / (double)lambda);
        m[k] = (double)prior_mean;
      }
      // without an intercept the bias column is 0 and its coefficient stays at 0
      q[Dg] = has_intercept ? (penalize_intercept ? 1.0 / (1.0 / (double)lambda) : 1.0 / 100000.0) : 1.0;
      m[Dg] = has_intercept ? (double)prior_mean : 0.0;
      CK(cudaMemcpyAsync(dm, m.data(), ldx * 8, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(dq, q.data(), ldx * 8, cudaMemcpyHostToDevice, st));
      CK(cudaStreamSynchronize(st));   // q / m are reused by the next lambda
      naive_init_kernel<<<B.nprob, 128, 0, st>>>(B.d, dm, dq);
      B.mirror.clear();                // the factors of the previous lambda belong to another prior
      if (int rc = batch_xupdate(B, st, 2e-7, 100, 0, 1, hflag, dflag, cnt)) return rc;
      lap("solve");
      gather_beta_kernel<<<B.nprob, 128, 0, st>>>(B.d, Dt, dout, dmask);
      CK(cudaMemcpyAsync(xs.data(), dout, xs.size() * 8, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      for (int b = 0; b < B.nprob; b++) {
        double* dst = out_model + ((size_t)l * K + todo[pos + b]) * Dt;
        std::memcpy(dst, xs.data() + (size_t)b * Dt, Dt * 8);
        if (!has_intercept) dst[Dg] = 0.0;
      }
      lap("read-back");
    }
    pos = end;
  }
  if (cnt.not_converged) return fail(MLEASE_ERR_NUMERIC, "Model fitting error! (" + std::to_string(cnt.not_converged) + " fits did not converge)");
  return 0;
}

int mlease_naive_train_dense(int32_t device, void* stream, int32_t K, int32_t Dg, const int64_t* key_rowstart, const float* X, int64_t ldx_in,
                             const int32_t* response, const float* weight, const float* offset, float lambda, const float* lambda_map,
                             float prior_mean, int32_t penalize_intercept, int32_t has_intercept, int32_t data_size_threshold,
                             double* out_model, int32_t* skipped) {
  return mlease_naive_train(device, stream, K, Dg, key_rowstart, nullptr, nullptr, X, ldx_in, response, weight, offset, 1, &lambda, lambda_map,
                            prior_mean, penalize_intercept, has_intercept, data_size_threshold, 0, out_model, skipped);
}

}  // extern "C"
