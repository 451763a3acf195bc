// newton.cu -- the device-side Newton / line-search state machine around K1-K3.
//
// One "slot" = K1 (evaluate f,g at the trial point) -> k1_reduce_decide (accept / shrink) ->
// [Gram K2 -> chol_prep -> Cholesky K3] (only when ctrl.need_hess) -> newton_solve (two
// triangular solves, next trial point, termination test).  All decisions are taken on the
// device from Ctrl flags; the host launches the same kernel sequence every slot.
//
// Replaces bw/Tron.java:30-124 (TRON outer loop) + :126-179 (CG) for the x-update
// argmin_b  sum_i w_i log(1+exp(-y_i(x_i.b+o_i))) + 1/2 sum_k q_k (b_k-m_k)^2
// (llf/LogisticRegressionL2.java:30-47).  Same unique minimiser; the reference stops TRON at a
// loose tolerance, this path solves to |dir|_inf <= xtol*max(|b|_inf,1e-2) (DESIGN.md, parity protocol).
#include "kernels.cuh"

namespace mlease {

constexpr int NT = 256;

__device__ __forceinline__ double block_sum(double v, double* sc) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sc[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += sc[w];
  return s;
}
__device__ __forceinline__ double block_max(double v, double* sc) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sc[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); w++) s = fmax(s, sc[w]);
  return s;
}

// Start of an x-update: beta = beta_t = init, flags reset.  init/m/q were written by the caller
// (ADMM consensus kernel or mlease_fit_partition).
__global__ void newton_begin_kernel(const Problem* __restrict__ probs, double xtol, int max_newton, int hess_policy,
                                    int invalidate_hess, int rebuild_is_expensive) {
  const Problem& pb = probs[blockIdx.x];
  Ctrl* c = pb.ctrl;
  for (int k = threadIdx.x; k < pb.ldx; k += blockDim.x) {
    const double b = k < pb.Dt ? pb.beta[k] : 0.0;
    // Trial points live on the float lattice: K1 reads beta as fp32, so the gradient it returns is the
    // gradient AT float(beta_t).  Keeping beta_t == (double)float(beta_t) makes the iteration consistent;
    // only the final (unevaluated) Newton correction is applied in double.
    const float bf = (float)b;
    pb.beta[k] = (double)bf;
    pb.beta_t[k] = (double)bf;
    pb.beta_tf[k] = bf;
    pb.dir[k] = 0.0;
  }
  if (threadIdx.x == 0) {
    if (invalidate_hess) c->hess_valid = 0;
    if (!(c->h0_scale > 0.0)) c->h0_scale = 1.0;
    c->done = 0; c->have_dir = 0; c->need_solve = 0; c->need_hess = 0; c->fail = 0;
    c->newton_steps = 0; c->evals = 0; c->rejects = 0; c->hess_builds = 0; c->stall = 0; c->build_step = 0; c->warm_used = 0;
    c->alpha = 1.0; c->phi0 = 0.0; c->f_acc = 0.0; c->f_t = 0.0; c->gnorm = 0.0; c->gnorm_prev = 0.0; c->dirnorm = 0.0; c->dirnorm_prev = 0.0;
    c->xtol = xtol; c->max_newton = max_newton; c->hess_policy = hess_policy; c->rebuild_is_expensive = rebuild_is_expensive;
    if (!rebuild_is_expensive) c->h0_scale = 1.0;
    // Rebuild at the start point when there is no factor, when the policy says always, or when the previous
    // x-update's chord steps contracted slowly: a factor taken at a (nearly) converged point makes every later
    // x-update of the ADMM run a 2-3 pass affair, and costs about as much as 2.5 K1 passes.
    c->emit = (hess_policy == 1 || !c->hess_valid || c->refresh_next) ? 1 : 0;
    c->refresh_next = 0;
    if (c->emit) c->skip_eval = 0;   // a rebuild at the start point needs K1's sqrt(d) there: regular first slot
    c->worst_ratio = 0.0;
  }
}

// Fixed-order (deterministic) reduction of the per-CTA K1 partials, parallel over columns: CTA = 32 columns x 8 groups of
// partials; g_t[k] = sum_t gpart[t][k] (data term only; the prior term is added by the decide kernel).
__global__ void __launch_bounds__(256) k1_partial_reduce_kernel(const Problem* __restrict__ probs) {
  const Problem& pb = probs[blockIdx.y];
  if (pb.ctrl->done || pb.ctrl->skip_eval) return;   // skip_eval: g_t already holds the data-term gradient of the start point
  __shared__ double sh[8][33];
  const int c = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int k = blockIdx.x * 32 + c;
  const int nct = pb.ctrl->k1_chunks, ldx = pb.ldx;
  double s = 0.0;
  if (k < pb.Dt) {
    if (pb.gpart_f) { for (int t = grp; t < nct; t += 8) s += (double)pb.gpart_f[(size_t)t * ldx + k]; }   // fused CSR K1: fp32 per-segment partials
    else { for (int t = grp; t < nct; t += 8) s += pb.gpart[(size_t)t * ldx + k]; }
  }
  sh[grp][c] = s;
  __syncthreads();
  if (grp == 0 && k < pb.Dt) {
    double a = 0.0;
#pragma unroll
    for (int g = 0; g < 8; g++) a += sh[g][c];
    pb.g_t[k] = a;
  }
}

// Prior term, objective, then the accept/shrink decision and (fused) the first L-BFGS loop of the next direction.
//   g_t = sum_cta gpart + q*(beta_t - m)           (llf/LogisticRegressionL2.java:223-224)
//   f_t = sum_cta fpart + 1/2 sum q (beta_t-m)^2   (:181-190)
// spec != 0: the host enqueued this slot before it knew the outcome of the previous one (slot pipelining), hence WITHOUT the
// Gram / Cholesky launches a rebuild needs: a rebuild that is due is deferred (emit stays set, the step is a chord step on
// the factor at hand; the host sees emit in the next flag word and runs a regular rebuild slot).
__global__ void __launch_bounds__(1024) k1_reduce_decide_kernel(const Problem* __restrict__ probs, int spec) {
  const Problem& pb = probs[blockIdx.x];
  Ctrl* c = pb.ctrl;
  if (c->done) return;
  __shared__ double sc[32];
  const int NTD = blockDim.x;   // 256 threads, or 1024 for wide systems (one CTA per problem walks D'-long vectors a dozen times)
  __shared__ int s_action;  // 1 accept, 0 retry
  __shared__ double s_alpha;
  const int Dt = pb.Dt, ldx = pb.ldx, nct = c->k1_chunks;
  const bool have_dir = c->have_dir != 0;
  double prior2 = 0.0, ginf = 0.0, phi = 0.0;
  for (int k = threadIdx.x; k < Dt; k += NTD) {
    const double dlt = pb.beta_t[k] - pb.m[k];
    const double g = pb.g_t[k] + pb.q[k] * dlt;   // g_t holds the reduced data term (k1_partial_reduce_kernel)
    pb.g_t[k] = g;
    prior2 += pb.q[k] * dlt * dlt;
    ginf = fmax(ginf, fabs(g));
    if (have_dir) phi += g * pb.dir[k];
  }
  double lossp = 0.0;
  for (int t = threadIdx.x; t < nct; t += NTD) lossp += pb.fpart[t];
  // secant pair of this step (used only if the step is accepted): s = beta_t - beta, y = g_t - g_acc
  double sy = 0.0, ss = 0.0, yy2 = 0.0;
  if (have_dir) {
    for (int k = threadIdx.x; k < Dt; k += NTD) {
      const double sk = pb.beta_t[k] - pb.beta[k], yk = pb.g_t[k] - pb.g_acc[k];
      sy += sk * yk; ss += sk * sk; yy2 += yk * yk;
    }
  }
  sy = block_sum(sy, sc);
  ss = block_sum(ss, sc);
  yy2 = block_sum(yy2, sc);
  __shared__ int s_slot;
  prior2 = block_sum(prior2, sc);
  phi = block_sum(phi, sc);
  lossp = block_sum(lossp, sc);
  ginf = block_max(ginf, sc);
  if (threadIdx.x == 0) {
    const double f_t = lossp + 0.5 * prior2;
    c->f_t = f_t;
    if (!c->skip_eval) { c->evals++; c->tot_evals++; }   // skip_eval: no pass was run for this "evaluation"
    else c->warm_used = 1;
    c->skip_eval = 0;
    // first exact evaluation after a start on the estimated gradient: this point becomes the base point whatever the
    // directional derivative says (like the first evaluation of a regular x-update, which is always accepted)
    const bool first_exact = have_dir && c->warm_used && c->evals == 1;
    int action = 1;
    double alpha = c->alpha;
    if (have_dir && !first_exact) {
      // phi'(alpha) = g(beta + alpha dir).dir ; phi'(0) = phi0 < 0.  Accept while the directional
      // derivative has not overshot by more than half of |phi'(0)| (a relaxed curvature condition on
      // a convex 1-D function); otherwise shrink alpha towards the secant root of phi'.
      const double a0 = fabs(c->phi0);
      if (!(phi <= 0.5 * a0)) {
        action = 0;
        double an = alpha * a0 / (phi + a0);  // secant between (0,-a0) and (alpha,phi)
        an = fmin(fmax(an, 0.1 * alpha), 0.6 * alpha);
        alpha = an;
        c->rejects++; c->tot_rejects++;
        if (c->rejects > 40 || !(phi == phi)) { c->fail = 2; c->done = 1; }
      }
    }
    if (action == 1) {
      c->gnorm_prev = c->gnorm;
      c->gnorm = ginf;
      c->f_acc = f_t;
      if (have_dir) {
        c->newton_steps++; c->tot_newton++;
        if (c->gnorm_prev > 0.0 && c->evals >= 2) c->worst_ratio = fmax(c->worst_ratio, ginf / c->gnorm_prev);
      }
      if (ginf == 0.0) {
        c->done = 1; c->need_solve = 0; c->need_hess = 0;
      } else if (c->newton_steps >= c->max_newton) {
        c->done = 1; c->fail = 3; c->need_solve = 0; c->need_hess = 0;
      } else {
        c->need_solve = 1;
        // a rebuild happens only if K1 wrote the scaled copy at THIS point (emit was set before the pass)
        const int deferred = (spec && c->emit) ? 1 : 0;
        c->need_hess = (c->emit && !spec) ? 1 : 0;
        // policy for the NEXT accepted point: refresh when the chord step contracted poorly
        if (c->hess_policy == 1) {
          c->emit = 1;
        } else {
          // Wide systems (a rebuild costs more than ~8 passes) lean on the secant pairs instead of refactorising -- but not for
          // ever: a dozen steps on the same factor that still contract by less than 2x mean the factor was taken too far
          // away (a cold fit whose IRLS weights moved a lot), and one rebuild here is cheaper than the steps it saves.
          const bool stuck = c->rebuild_is_expensive && have_dir && c->gnorm_prev > 0.0 && ginf > 0.5 * c->gnorm_prev &&
                             c->newton_steps - c->build_step >= 12;
          // (evals >= 2: after a warm start the previous norm is the ESTIMATED start gradient; contraction is judged between exact ones)
          const bool poor = stuck || (!c->rebuild_is_expensive && have_dir && c->evals >= 2 && c->gnorm_prev > 0.0 && ginf > 0.25 * c->gnorm_prev);
          c->emit = (poor && !c->need_hess) ? 1 : 0;
          if (!c->need_hess && !c->hess_valid) { c->emit = 1; }
          if (deferred) c->emit = 1;
        }
      }
    } else {
      c->need_solve = 0; c->need_hess = 0;
    }
    c->alpha = alpha;
    s_action = action;
    s_alpha = alpha;
    s_slot = -1;
    // A rebuild at this accepted point supersedes the secant pairs: drop them HERE (before the fused first L-BFGS loop
    // below runs), so that both loops of the recursion see the same, empty, pair set.
    if (action == 1 && c->need_hess) c->bfgs_count = 0;
    if (action == 1 && have_dir && !c->need_hess && sy > 1e-10 * sqrt(ss * yy2) && sy > 0.0) {   // strictly convex => s.y > 0 up to rounding
      s_slot = c->bfgs_count % BFGS_M;
      pb.bfgs_rho[s_slot] = 1.0 / sy;
      c->bfgs_count++;
      // Self-scaling of the stale inverse (systems too wide to refactorise mid-run keep the factor of the cold start, where
      // every IRLS weight is at its maximum 1/4: H0 is uniformly too small an inverse).  Along the accepted step the model
      // predicted a gradient change of -alpha*phi0, the data returned s.y: their ratio is how much longer the step should
      // have been.  Standard L-BFGS practice (gamma = s.y / y.y for H0 = I), taken along s so that it costs no extra GEMV.
      if (c->rebuild_is_expensive) {
        const double tau = fmin(fmax(-(alpha * c->phi0) / sy, 0.5), 2.0);
        c->h0_scale = fmin(fmax(c->h0_scale * tau, 0.25), 16.0);
      }
    }
  }
  __syncthreads();
  if (s_action == 1) {
    if (s_slot >= 0) {
      double* S = pb.bfgs_S + (size_t)s_slot * ldx;
      double* Y = pb.bfgs_Y + (size_t)s_slot * ldx;
      for (int k = threadIdx.x; k < ldx; k += NTD) {
        S[k] = k < Dt ? pb.beta_t[k] - pb.beta[k] : 0.0;
        Y[k] = k < Dt ? pb.g_t[k] - pb.g_acc[k] : 0.0;
      }
    }
    for (int k = threadIdx.x; k < ldx; k += NTD) {
      pb.beta[k] = pb.beta_t[k];
      pb.g_acc[k] = k < Dt ? pb.g_t[k] : 0.0;
    }
  } else {
    const double a = s_alpha;
    for (int k = threadIdx.x; k < ldx; k += NTD) {
      const float btf = k < Dt ? (float)(pb.beta[k] + a * pb.dir[k]) : 0.f;
      pb.beta_t[k] = (double)btf;
      pb.beta_tf[k] = btf;
    }
  }
  // ---- fused: first loop of the L-BFGS two-loop recursion for the next direction (q -> g_t scratch) ----
  __syncthreads();
  if (c->done || !c->need_solve) return;
  {
    const int npairs = min(c->bfgs_count, BFGS_M);
    double* q = pb.g_t;   // free scratch from here until the next K1 reduce
    for (int k = threadIdx.x; k < Dt; k += NTD) q[k] = pb.g_acc[k];
    __syncthreads();
    for (int j = 0; j < npairs; j++) {
      const int slot = (c->bfgs_count - 1 - j) % BFGS_M;
      const double* S = pb.bfgs_S + (size_t)slot * ldx;
      const double* Y = pb.bfgs_Y + (size_t)slot * ldx;
      double d = 0.0;
      for (int k = threadIdx.x; k < Dt; k += NTD) d += S[k] * q[k];
      d = block_sum(d, sc);
      const double a = pb.bfgs_rho[slot] * d;
      if (threadIdx.x == 0) pb.bfgs_alpha[slot] = a;
      for (int k = threadIdx.x; k < Dt; k += NTD) q[k] -= a * Y[k];
      __syncthreads();
    }
    // wide systems: the triangular GEMVs take their vector in fp32 (the operand Ysym is bf16: nothing is lost)
    if (pb.Ysym) for (int k = threadIdx.x; k < ldx; k += NTD) pb.qf[k] = k < Dt ? (float)q[k] : 0.f;
  }
}

// Quasi-Newton direction: the explicit inverse of the last Hessian rebuild is the initial matrix H0^-1 of an
// L-BFGS two-loop recursion over the last BFGS_M secant pairs (exact gradients => s.y > 0), so chord steps
// converge superlinearly instead of at the linear rate |I - H0^-1 H|.
//   pre  (tail of k1_reduce_decide_kernel): q = g_acc; for newest..oldest: a_i = rho_i s_i.q ; q -= a_i y_i  -> g_t (scratch)
//   gemv (multi-CTA)    : r = Hinv q                                                                -> dir
//   post (in newton_solve_kernel): for oldest..newest: b = rho_i y_i.r ; r += s_i (a_i - b) ; dir = -r
__global__ void __launch_bounds__(NT) newton_gemv_kernel(const Problem* __restrict__ probs) {
  const Problem& pb = probs[blockIdx.y];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_solve) return;
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (NT / 32) + (threadIdx.x >> 5);
  if (r >= pb.Dt) return;
  const double* q = pb.g_t;
  double a = 0.0;
  const double* Hr = pb.Hinv + (size_t)r * pb.ldh;
  for (int k = lane; k < pb.Dt; k += 32) a += Hr[k] * q[k];
  a = warp_sum(a);
  if (lane == 0) pb.dir[r] = a;   // r = Hinv q (sign applied after the second loop)
}

// Wide systems: r = Y^T (Y q) on the symmetric bf16 storage of Y = L^-1 (Ysym, see ysym_kernel).  phase 0: t = Y q (row r of
// the lower part, columns 0..r); phase 1: dir = Y^T t (row c of the upper part incl. the diagonal, columns c..Dt-1).
// bf16 operand (8 elements per 16-byte load), fp64 accumulation; each phase reads half of the matrix.
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }          // bf16 -> fp32 is a 16-bit shift
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

// group_L > 1: problems b = g*group_L .. +group_L-1 are the lambdas of one partition.  After a shared cold-start factorisation
// they all point at the leader's Y (Ctrl::ysym_use), and the FIRST active problem of such a set streams Y once for every active
// member (up to 4 vectors per pass); a problem with its own factor, or alone in its set, runs by itself.
constexpr int GEMV_MAXV = 4;
constexpr int GEMV_RB = 4;     // rows per warp pass
__global__ void __launch_bounds__(NT) newton_gemv_tri_kernel(const Problem* __restrict__ probs, int phase, int group_L) {
  const int b = blockIdx.y;
  const Problem& pb = probs[b];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_solve) return;
  const __nv_bfloat16* __restrict__ Y = reinterpret_cast<const __nv_bfloat16*>(c->ysym_use ? c->ysym_use : (const void*)pb.Ysym);
  const int gl = (group_L > 1 && group_L <= GEMV_MAXV) ? group_L : 1;
  const int g0 = b - b % gl;
  const float* xs[GEMV_MAXV];
  float* tfs[GEMV_MAXV];
  double* dirs[GEMV_MAXV];
  unsigned mask = 0;   // members of the set {active, same Y}; slot v = problem g0 + v (static indexing keeps the pointers in registers)
#pragma unroll
  for (int v = 0; v < GEMV_MAXV; v++) {
    const int j = g0 + v;
    bool same = false;
    if (v < gl && j < (int)gridDim.y) {
      const Ctrl* cj = probs[j].ctrl;
      same = !cj->done && cj->need_solve && (cj->ysym_use ? cj->ysym_use : (const void*)probs[j].Ysym) == (const void*)Y;
    }
    const Problem& pj = probs[same ? j : b];
    xs[v] = phase == 0 ? pj.qf : pj.tf; tfs[v] = pj.tf; dirs[v] = pj.dir;
    if (same) mask |= 1u << v;
  }
  if (__ffs(mask) - 1 != b - g0) return;   // an earlier active member of the set takes this problem's vector along
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * (NT / 32) + (threadIdx.x >> 5);
  const int Dt = pb.Dt;
  const int nblk = (Dt + GEMV_RB - 1) / GEMV_RB;
  if (w >= (nblk + 1) / 2) return;
  // A warp takes a block of GEMV_RB rows and the mirrored block: together they hold the same number of triangle elements whatever w
  // is (balanced).  Per k-chunk a lane loads its 8 elements of every vector ONCE (L1) and of each of the block's rows (the HBM
  // stream, GEMV_RB independent 16-byte loads in flight per lane); fp32 products and per-lane sums (Y is bf16: 3e-3 per element),
  // fp64 only across the warp.
#pragma unroll 1
  for (int half = 0; half < 2; half++) {
    const int rb = half == 0 ? w : nblk - 1 - w;
    if (half == 1 && rb == w) break;
    const int r0 = rb * GEMV_RB;
    const int kbeg = phase == 0 ? 0 : (r0 & ~7), kend = phase == 0 ? min(r0 + GEMV_RB, Dt) : Dt;
    float acc[GEMV_RB][GEMV_MAXV];
#pragma unroll
    for (int j = 0; j < GEMV_RB; j++)
#pragma unroll
      for (int v = 0; v < GEMV_MAXV; v++) acc[j][v] = 0.f;
    for (int k = kbeg + lane * 8; k < kend; k += 256) {
      uint4 h[GEMV_RB];
#pragma unroll
      for (int j = 0; j < GEMV_RB; j++)   // rows are ldh (multiple of 32) elements long: a chunk that starts below Dt stays inside its row
        h[j] = (r0 + j < Dt) ? *reinterpret_cast<const uint4*>(Y + (size_t)(r0 + j) * pb.ldh + k) : make_uint4(0u, 0u, 0u, 0u);
      float xv[GEMV_MAXV][8];
      const bool second = k + 4 < pb.ldx;   // vectors are ldx (multiple of 4) long and 32-byte aligned at k
#pragma unroll
      for (int v = 0; v < GEMV_MAXV; v++) {
        if ((mask >> v) & 1u) {
          const float4 x0 = *reinterpret_cast<const float4*>(xs[v] + k);
          const float4 x1 = second ? *reinterpret_cast<const float4*>(xs[v] + k + 4) : make_float4(0.f, 0.f, 0.f, 0.f);
          xv[v][0] = x0.x; xv[v][1] = x0.y; xv[v][2] = x0.z; xv[v][3] = x0.w; xv[v][4] = x1.x; xv[v][5] = x1.y; xv[v][6] = x1.z; xv[v][7] = x1.w;
        }
      }
      // triangle edge: phase 0 keeps k+e <= row, phase 1 keeps row <= k+e < Dt
      const bool edge = phase == 0 ? (k + 8 > r0 + 1) : (k < r0 + GEMV_RB || k + 8 > Dt);
#pragma unroll
      for (int j = 0; j < GEMV_RB; j++) {
        float hv[8] = {bf16_lo(h[j].x), bf16_hi(h[j].x), bf16_lo(h[j].y), bf16_hi(h[j].y), bf16_lo(h[j].z), bf16_hi(h[j].z), bf16_lo(h[j].w), bf16_hi(h[j].w)};
        if (edge) {
          const int row = r0 + j;
#pragma unroll
          for (int e = 0; e < 8; e++) {
            const bool keep = phase == 0 ? (k + e <= row) : (k + e >= row && k + e < Dt);
            if (!keep) hv[e] = 0.f;
          }
        }
#pragma unroll
        for (int v = 0; v < GEMV_MAXV; v++) {
          if ((mask >> v) & 1u) {
            float p = acc[j][v];
#pragma unroll
            for (int e = 0; e < 8; e++) p = fmaf(hv[e], xv[v][e], p);
            acc[j][v] = p;
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < GEMV_RB; j++) {
#pragma unroll
      for (int v = 0; v < GEMV_MAXV; v++) {
        if ((mask >> v) & 1u) {
          const double sv = warp_sum((double)acc[j][v]);
          if (lane == 0 && r0 + j < Dt) {
            if (phase == 0) tfs[v][r0 + j] = (float)sv;
            else dirs[v][r0 + j] = sv;
          }
        }
      }
    }
  }
}

// Direction bookkeeping: norms, termination test, next trial point.  One CTA per problem.
__global__ void __launch_bounds__(1024) newton_solve_kernel(const Problem* __restrict__ probs) {
  const Problem& pb = probs[blockIdx.x];
  Ctrl* c = pb.ctrl;
  if (c->done || !c->need_solve) return;
  __shared__ double sc[32];
  const int NTD = blockDim.x;
  const int tid = threadIdx.x;
  const int Dt = pb.Dt, ldx = pb.ldx;
  double* rhs = pb.dir;
  {
    const int npairs = min(c->bfgs_count, BFGS_M);
    const double h0s = c->h0_scale;
    if (h0s != 1.0) {
      for (int k = tid; k < Dt; k += NTD) rhs[k] *= h0s;
      __syncthreads();
    }
    for (int j = npairs - 1; j >= 0; j--) {
      const int slot = (c->bfgs_count - 1 - j) % BFGS_M;
      const double* S = pb.bfgs_S + (size_t)slot * ldx;
      const double* Y = pb.bfgs_Y + (size_t)slot * ldx;
      double d = 0.0;
      for (int k = tid; k < Dt; k += NTD) d += Y[k] * rhs[k];
      d = block_sum(d, sc);
      const double coef = pb.bfgs_alpha[slot] - pb.bfgs_rho[slot] * d;
      for (int k = tid; k < Dt; k += NTD) rhs[k] += coef * S[k];
      __syncthreads();
    }
    for (int k = tid; k < Dt; k += NTD) rhs[k] = -rhs[k];
    __syncthreads();
  }
  double dinf = 0.0, binf = 0.0, phi0 = 0.0;
  for (int k = tid; k < Dt; k += NTD) {
    const double d = rhs[k];
    dinf = fmax(dinf, fabs(d));
    binf = fmax(binf, fabs(pb.beta[k]));
    phi0 += d * pb.g_acc[k];
  }
  dinf = block_max(dinf, sc);
  binf = block_max(binf, sc);
  phi0 = block_sum(phi0, sc);
  __shared__ int s_final;
  if (tid == 0) {
    c->dirnorm_prev = c->dirnorm;
    c->dirnorm = dinf;
    c->phi0 = phi0;
    c->alpha = 1.0;
    c->have_dir = 1;
    c->need_solve = 0;
    c->rejects = 0;
    int fin = 0;
    if (!(phi0 < 0.0) || !(dinf == dinf)) { c->fail = 1; c->done = 1; fin = 2; }  // factor unusable
    else if (dinf <= c->xtol * fmax(binf, 1e-2) && c->evals > 0) { c->done = 1; fin = 1; }   // never before the first exact evaluation
    else if (c->newton_steps >= 2 && dinf <= 1e-5 * fmax(binf, 1e-2) && dinf > 0.5 * c->dirnorm_prev) {
      // rounding floor of the fp32 data path: the step no longer shrinks -> take it and stop
      if (++c->stall >= 2) { c->done = 1; fin = 1; }
    } else {
      c->stall = 0;
    }
    c->need_hess = 0;
    if (fin && c->hess_policy == 0 && c->newton_steps >= (c->rebuild_is_expensive ? 16 : 6) && c->hess_builds == 0) c->refresh_next = 1;   // a stale model needed many steps
    s_final = fin;
  }
  __syncthreads();
  if (s_final == 2) return;
  const bool fin = s_final == 1;
  for (int k = tid; k < pb.ldx; k += NTD) {
    const double bt = k < Dt ? pb.beta[k] + rhs[k] : 0.0;
    const float btf = (float)bt;
    pb.beta_t[k] = (double)btf;
    pb.beta_tf[k] = btf;
    if (fin) pb.beta[k] = bt;  // final tiny step taken in double, without another pass
  }
}

cudaError_t newton_begin(const Problem* d_probs, int nprob, double xtol, int max_newton, int hess_policy,
                         int invalidate_hess, int rebuild_is_expensive, cudaStream_t st, int* launches) {
  newton_begin_kernel<<<nprob, 256, 0, st>>>(d_probs, xtol, max_newton, hess_policy, invalidate_hess, rebuild_is_expensive);
  if (launches) *launches += 1;
  return cudaGetLastError();
}
cudaError_t k1_reduce_decide(const Problem* d_probs, int nprob, int Dt, cudaStream_t st, int* launches, int spec) {
  k1_partial_reduce_kernel<<<dim3((Dt + 31) / 32, nprob), 256, 0, st>>>(d_probs);
  k1_reduce_decide_kernel<<<nprob, Dt > 2048 ? 1024 : NT, 0, st>>>(d_probs, spec);
  if (launches) *launches += 2;
  return cudaGetLastError();
}
cudaError_t newton_solve(const Problem* d_probs, int nprob, int ldh, cudaStream_t st, int* launches, int group_L) {
  const dim3 grid((ldh + NT / 32 - 1) / (NT / 32), nprob);
  if (cholesky_factored_direction(ldh)) {
    const int nblk2 = ((ldh + GEMV_RB - 1) / GEMV_RB + 1) / 2;   // row blocks, two (a block and its mirror) per warp
    const dim3 gtri((nblk2 + NT / 32 - 1) / (NT / 32), nprob);
    newton_gemv_tri_kernel<<<gtri, NT, 0, st>>>(d_probs, 0, group_L);
    newton_gemv_tri_kernel<<<gtri, NT, 0, st>>>(d_probs, 1, group_L);
    if (launches) *launches += 1;
  } else {
    newton_gemv_kernel<<<grid, NT, 0, st>>>(d_probs);
  }
  newton_solve_kernel<<<nprob, ldh > 2048 ? 1024 : NT, 0, st>>>(d_probs);
  if (launches) *launches += 2;
  return cudaGetLastError();
}
}  // namespace mlease
