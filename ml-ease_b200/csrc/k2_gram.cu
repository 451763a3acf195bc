// k2_gram.cu -- K2: weighted Gram  G = Xt^T Xt  (Xt = diag(sqrt d) X in bf16, written by K1), the
// data term of LogisticRegressionL2.hessian (llf/LogisticRegressionL2.java:258-297):
//     H[m][n] = (m==n ? 1/priorVar[m] : 0) + sum_i D_ii x_im x_in ,  D_ii = w_i p_i (1-p_i).
// It genuinely is a dense GEMM (K = rows, M = N = features), so it runs on the 5th-gen tensor
// cores: TMA (tensor map, 128B swizzle) -> shared memory -> tcgen05.mma (bf16 x bf16 -> fp32 in
// TMEM) -> tcgen05.ld epilogue.  Both operands are tiles of the SAME row-major matrix, i.e. they are
// MN-major ("transposed") UMMA operands: no transpose pass over X is ever made.
//
// Work decomposition: output tiles of 128 (M) x 256 (N) restricted to the lower block triangle,
// split-K over row slices; each CTA owns one (tile, slice), accumulates it in TMEM (256 columns)
// and stores the fp32 partial to Hpart[slice] (plain stores, deterministic).  chol_prep_kernel
// (k3_cholesky.cu) sums the slices in fixed order and adds diag(q).
//
// Warp roles (192 threads): warp 0 = TMA producer (one elected lane), warp 1 = MMA issuer (one
// elected lane) + TMEM allocator, warps 2-5 = epilogue (tcgen05.ld 32x32b, one TMEM lane quadrant
// each: warp_id % 4).
//
// A fp32 SIMT kernel computing the same partials from the same bf16 operand is kept ONLY as a
// debug cross-check reachable through mlease_objective(tensor=0); the product path never uses it.
#include <cuda.h>
#include <cuda_fp8.h>

#include <algorithm>
#include <cub/device/device_scan.cuh>

#include "kernels.cuh"

namespace mlease {

// ------------------------------------------------------------------------------------------
// tcgen05 kernel
// ------------------------------------------------------------------------------------------
constexpr int GM = 128;          // tile rows  (UMMA M)
constexpr int GN = 256;          // tile cols  (UMMA N)
constexpr int GK = 64;           // K (data rows) per pipeline stage
constexpr int UK = 16;           // K per tcgen05.mma (bf16)
constexpr int GSTAGES = 4;
constexpr int G_A_BYTES = GK * GM * 2;   // 16 KB : 2 boxes of [64 k][64 feat]
constexpr int G_B_BYTES = GK * GN * 2;   // 32 KB : 4 boxes
constexpr int G_STAGE_BYTES = G_A_BYTES + G_B_BYTES;
constexpr int G_BOX_BYTES = GK * 64 * 2; // 8 KB, one TMA box = 64 k-rows x 128 B
constexpr int G_THREADS = 192;
constexpr size_t G_SMEM = (size_t)GSTAGES * G_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;

// UMMA shared-memory descriptor, MN-major operand, SWIZZLE_128B (cute::UMMA::SmemDescriptor layout):
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=2 (SW128)
// canonical MN-major SW128 layout (bf16): ((64 elems,m),(8,k)) : ((1,LBO),(128B,SBO)):
//   SBO = 1024 B between 8-row K groups, LBO = GK*128 B between 64-element MN groups (one TMA box).
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) @4, a/b_format BF16 (1) @7/@10,
// a_major/b_major = MN (1) @15/@16, N>>3 @17, M>>4 @24.
__device__ __forceinline__ uint32_t umma_idesc_bf16_mn(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

struct GramTile { short bi, bj; };   // 128-row block index, 256-col block index

__global__ void __launch_bounds__(G_THREADS, 1)
gram_tcgen05_kernel(const Problem* __restrict__ probs, const CUtensorMap* __restrict__ tmaps, const GramTile* __restrict__ tiles,
                    int ntiles, int force, int share) {
  // share = L > 1: the L problems of one partition are at the same iterate (cold start), so their Grams are identical;
  // only the first of each group is built and chol_prep_kernel reads it for the whole group
  if (share > 1 && blockIdx.z % share != 0) return;
  const int pidx = blockIdx.z;
  const Problem& pb = probs[pidx];
  Ctrl* ctrl = pb.ctrl;
  if (!force && (ctrl->done || !ctrl->need_hess)) return;
  const CUtensorMap* tmap = &tmaps[pb.self_idx];   // not blockIdx.z: large batches launch over a compacted copy of the problem array
  const GramTile tile = tiles[blockIdx.x];
  const int slice = blockIdx.y, nslices = gridDim.y;
  const int Dp = pb.Dp;
  const long long ksteps_total = (pb.n + GK - 1) / GK;
  const long long per = (ksteps_total + nslices - 1) / nslices;
  const long long ks0 = slice * per;
  const long long ks1 = min(ksteps_total, ks0 + per);
  const int nk = (int)max(0LL, ks1 - ks0);

  extern __shared__ unsigned char g_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(g_smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)GSTAGES * G_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + GSTAGES;
  uint64_t* acc_bar = empty_bar + GSTAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(tmap);
    for (int s = 0; s < GSTAGES; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(acc_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, GN);   // 256 columns x 128 lanes fp32
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      for (int k = 0; k < nk; k++) {
        const int st = k % GSTAGES;
        if (k >= GSTAGES) mbar_wait(&empty_bar[st], (uint32_t)(((k / GSTAGES) - 1) & 1));
        unsigned char* a_dst = smem + (size_t)st * G_STAGE_BYTES;
        unsigned char* b_dst = a_dst + G_A_BYTES;
        mbar_arrive_expect_tx(&full_bar[st], G_STAGE_BYTES);
        const int krow = (int)((ks0 + k) * GK);
#pragma unroll
        for (int b = 0; b < GM / 64; b++) tma_load_2d(a_dst + b * G_BOX_BYTES, tmap, tile.bi * GM + b * 64, krow, &full_bar[st]);
#pragma unroll
        for (int b = 0; b < GN / 64; b++) tma_load_2d(b_dst + b * G_BOX_BYTES, tmap, tile.bj * GN + b * 64, krow, &full_bar[st]);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc = umma_idesc_bf16_mn(GM, GN);
      for (int k = 0; k < nk; k++) {
        const int st = k % GSTAGES;
        mbar_wait(&full_bar[st], (uint32_t)((k / GSTAGES) & 1));
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + (size_t)st * G_STAGE_BYTES);
        const uint32_t b_addr = a_addr + G_A_BYTES;
#pragma unroll
        for (int kk = 0; kk < GK / UK; kk++) {
          // 16 k-rows = 2 swizzle atoms of 1024 B along K
          const uint64_t da = umma_desc_mn_sw128(a_addr + kk * (UK * 128), G_BOX_BYTES, 1024);
          const uint64_t db = umma_desc_mn_sw128(b_addr + kk * (UK * 128), G_BOX_BYTES, 1024);
          umma_f16(tmem_base, da, db, idesc, (k | kk) != 0 ? 1u : 0u);
        }
        umma_commit(&empty_bar[st]);   // frees the smem stage when these MMAs retire
      }
      umma_commit(acc_bar);            // accumulator complete
    }
  } else {
    // ===== epilogue: warps 2..5 -> TMEM lane quadrant (warp % 4) =====
    const int quad = warp & 3;
    float* out = pb.Hpart + (size_t)slice * Dp * Dp;
    const int row = tile.bi * GM + quad * 32 + lane;
    if (nk > 0) {
      mbar_wait(acc_bar, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int c0 = 0; c0 < GN; c0 += 32) {
      uint32_t r[32];
      if (nk > 0) {
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, r);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; j++) r[j] = 0u;
      }
      const int col = tile.bj * GN + c0;
      if (row < Dp && col < Dp) {
        float4* dst = reinterpret_cast<float4*>(out + (size_t)row * Dp + col);
#pragma unroll
        for (int j = 0; j < 8; j++)
          dst[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                               __uint_as_float(r[4 * j + 3]));
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, GN);
  }
}

// ------------------------------------------------------------------------------------------
// Sparse variant: the same split-K tcgen05 Gram, but the operand tiles are ASSEMBLED IN SHARED MEMORY, as e4m3, from the
// partition's block-major entry list (no dense Xt in HBM: at 1 % density that copy is 100x the input and makes the dense
// kernel HBM-bound).  One K-step = one 32-row group; its entries for a 128-column block are one contiguous run of
// (key, value), the key being the byte offset of the element inside the canonical MN-major SWIZZLE_128B operand block the
// UMMA descriptors expect (sw128_off).  24 producer warps, one per operand block of a stage: load the run coalesced, scale
// by sqrt(d_row) * 2^e, round to e4m3, store one byte at the key.  Positions outside the sparsity pattern are zero: the ring
// is cleared once, and a producer re-clears exactly the entries it wrote when it gets its stage back.  Generic-proxy stores
// are published to the tensor core's async proxy with fence.proxy.async before the mbarrier arrive.
// Warp roles (29 warps): 0 = MMA issuer (leader CTA) + TMEM allocator, 1..24 = producers, 25..28 = epilogue.
// Measured at 1M x 10k x 1 % (8 builds): bf16 operands 628 ms (1.27 PFLOP/s); e4m3 531 ms; unrolled issue loop 374 ms;
// CTA pairs 353 ms; shared-space byte stores (the generic ones rebuilt the shared window base at every store) 337 ms =
// 2.37 PFLOP/s.  What bounds it now is the MMA stream itself: with producers that ONLY hand stages over (no loads, no
// stores) a build takes 40.0 ms instead of 44.7 (tools/time_gram.py), i.e. 2.5 PFLOP/s is what one tcgen05.mma.kind::f8f6f4
// per K = 32 step delivers at the clocks a tensor-bound kernel sustains on this part (cuBLAS bf16 holds 1.43 PFLOP/s at a
// median 1365 MHz, MEASURED_PEAKS.json).
// ------------------------------------------------------------------------------------------
constexpr int SK = 32;                       // data rows (K) per stage
constexpr int S_BOX_BYTES = SK * 128;        // 4 KB = one [32 k][128 cols] e4m3 operand block
// A CTA PAIR (cluster of 2, cta_group::2) owns a 256 x 256 tile: each CTA assembles ITS 128 rows of A and ITS 128 of the B tile's
// 256 columns (8 KB per stage); 24 stages, 12 producer pairs.  K-step k lives in stage k % S_SST and belongs to producer group
// k % S_NGRP (S_SST = 2 S_NGRP: a group alternates between two stages, because the refill round trip is several MMA periods long).
constexpr int S_SPW = 2;                       // producer warps per stage: one per operand block (A, B)
constexpr int S_NGRP = 24 / S_SPW;             // producer groups
constexpr int S_SST = 2 * S_NGRP;              // ring stages
constexpr int S_STAGE_BYTES = S_SPW * S_BOX_BYTES;
constexpr size_t S_SMEM = (size_t)S_SST * S_STAGE_BYTES + 1024 /*align*/ + 512 /*barriers*/;
constexpr int S_THREADS = (1 + 24 + 4) * 32;   // MMA warp, 24 producer warps, 4 epilogue warps

// byte offset of element (K-row k, column col < 128) inside one [32 k][128 cols] operand block of 1-byte elements: the canonical
// MN-major SWIZZLE_128B layout has 128 B (= 128 e4m3 elements along MN) per K-row, 8 K-rows per 1024-B swizzle atom, and the
// 16-byte chunk index XOR-ed with the row inside the atom
__device__ __forceinline__ uint32_t sw128_off(int k, int col) {
  return (uint32_t)(k * 128 + ((((col >> 4) ^ (k & 7)) << 4) | (col & 15)));
}
// Instruction descriptor for kind::f8f6f4: c_format F32 (1) @4, a/b_format E4M3 (0) @7/@10, a_major/b_major = MN (1) @15/@16
// (valid for the 8-bit formats, cute/arch/mma_sm100_desc.hpp), N>>3 @17, M>>4 @24.
__device__ __forceinline__ uint32_t umma_idesc_e4m3_mn(int M, int N) {
  return (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__global__ void __launch_bounds__(S_THREADS, 1)
gram_csr_tcgen05_kernel(const Problem* __restrict__ probs, const GramTile* __restrict__ tiles, int ntiles, int force, int bias_col, int share) {
  if (share > 1 && blockIdx.z % share != 0) return;   // see gram_tcgen05_kernel (both CTAs of a pair take the same exit)
  const Problem& pb = probs[blockIdx.z];
  Ctrl* ctrl = pb.ctrl;
  if (!force && (ctrl->done || !ctrl->need_hess)) return;
  // the tile list holds (BI, bj) of 256 x 256 tiles; this CTA's rows are the 128-block 2 BI + rank
  const uint32_t rank = cluster_ctarank();
  const GramTile tile_in = tiles[blockIdx.x >> 1];
  const int tile_bi = tile_in.bi * 2 + (int)rank;
  const int tile_bj = tile_in.bj;
  const int slice = blockIdx.y, nslices = gridDim.y;
  const int Dp = pb.Dp;
  const long long n = pb.n;
  const long long ksteps_total = (n + SK - 1) / SK;
  const long long per = (ksteps_total + nslices - 1) / nslices;
  const long long ks0 = slice * per;
  const long long ks1 = min(ksteps_total, ks0 + per);
  const int nk = (int)max(0LL, ks1 - ks0);

  extern __shared__ unsigned char g_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(g_smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)S_SST * S_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + S_SST;
  uint64_t* acc_bar = empty_bar + S_SST;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // clear the whole ring once
  for (int e = threadIdx.x; e < S_SST * S_STAGE_BYTES / 16; e += S_THREADS) reinterpret_cast<uint4*>(smem)[e] = make_uint4(0u, 0u, 0u, 0u);
  if (warp == 1 && lane == 0) {
    // full: one arrival per producer warp of the stage, of BOTH CTAs (the barrier the MMA thread waits on is the leader's)
    for (int s = 0; s < S_SST; s++) { mbar_init(&full_bar[s], S_SPW * 2); mbar_init(&empty_bar[s], 1); }
    mbar_init(acc_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) { tmem_alloc2(tmem_slot, GN); tmem_relinquish2(); }
  fence_proxy_async_smem();   // the zero fill must be visible to the async proxy too
  tc_fence_before();
  cluster_sync_all();   // the peer must see initialised barriers before its first remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0 && rank == 0) {
      // ===== MMA issuer (the leader CTA's) =====
      // one tcgen05.mma.kind::f8f6f4 per stage: K = 32 = the stage's 32-row group (4 swizzle atoms, SBO = 1024 B apart), M = 256;
      // each CTA holds one A block and one B block at the same offsets.  The loop over the ring is unrolled so that a stage's
      // barrier addresses and descriptors are constants: at the e4m3 rate an MMA lasts ~130-220 clk, and the ~45 dependent
      // single-thread instructions of a rolled iteration (address math, R2UR moves) were the bottleneck (ncu r02: tensor pipe 35 %).
      const uint32_t idesc = umma_idesc_e4m3_mn(GM * 2, GN);
      const uint32_t smem_base = smem_u32(smem);
      const uint64_t da0 = umma_desc_mn_sw128(smem_base, S_BOX_BYTES, 1024);
      const uint64_t db0 = umma_desc_mn_sw128(smem_base + S_BOX_BYTES, S_BOX_BYTES, 1024);
      constexpr uint64_t DSTEP = (uint64_t)(S_STAGE_BYTES >> 4);   // the address field counts 16-byte units; the ring stays below its 14 bits
      for (int k0 = 0; k0 < nk; k0 += S_SST) {
        const uint32_t par = (uint32_t)((k0 / S_SST) & 1);
#pragma unroll
        for (int st = 0; st < S_SST; st++) {
          if (k0 + st < nk) {
            mbar_wait_cluster(&full_bar[st], par);
            tc_fence_after();
            umma_f8_2cta(tmem_base, da0 + (uint64_t)st * DSTEP, db0 + (uint64_t)st * DSTEP, idesc, (k0 + st) != 0 ? 1u : 0u);
            umma_commit_2cta(&empty_bar[st]);
          }
        }
      }
      umma_commit_2cta(acc_bar);
    }
  } else if (warp <= 24) {
    // ===== producers: S_SPW warps per stage, one per 128-column operand block (the A block and the B block this CTA holds).
    // One K-step = one 32-row group, whose entries for a 128-column block are one contiguous run of the block-major list.
    // Offsets are fetched three uses ahead and the first 64 entries of a run two uses ahead, so the loads of a use are in flight
    // during the whole previous uses.  Group t = (warp - 1) / S_SPW owns the K-steps k = t, t + S_NGRP, ...; K-step k lives in
    // ring stage k % S_SST, so a group alternates between the stages t and t + S_NGRP.
    const int grp = (warp - 1) / S_SPW, strm = (warp - 1) % S_SPW;
    const size_t strm_off = (size_t)strm * S_BOX_BYTES;
    const int blk = strm == 0 ? tile_bi : tile_bj * 2 + (int)rank;
    const bool valid = blk < pb.nblk128;
    const long long ngroups = pb.bm_groups;
    const long long* __restrict__ my_offs = pb.bm_offs + (size_t)(valid ? blk : 0) * ngroups + (lane & 1);
    const unsigned short* __restrict__ keys = pb.bm_keys;
    const float* __restrict__ bvals = pb.bm_vals;
    const float* __restrict__ sdv = pb.sdvec;
    // the bias column (value 1 in every row, llf/LibLinearDataset.java:592-614) is not stored in the CSR rows
    const bool has_bias_col = valid && bias_col >= blk * 128 && bias_col < blk * 128 + 128;
    const uint32_t bias_off = has_bias_col ? sw128_off(lane, bias_col - blk * 128) : 0u;
    constexpr uint32_t NOKEY = 0xFFFFFFFFu;
    const bool fetch = valid && lane < 2;
    // the full barriers the MMA thread waits on are the leader's: the producers arrive through the cluster address space
    const uint32_t full0_remote = mapa_u32(&full_bar[0], 0);

    // Pipeline registers: offsets three uses ahead (o_c), entries + sqrt(d) two uses ahead (set 2), one use ahead (set 1),
    // current (set 0); what the last TWO uses stored (p1 = previous use = the other stage, p2 = the use before = this stage).
    auto ld_offs = [&](int k) -> uint32_t { return (fetch && k < nk) ? (uint32_t)__ldg(my_offs + ks0 + k) : 0u; };   // the list holds < 2^32 entries (checked at upload)
    uint32_t lo0, hi0, lo1, hi1, lo2, hi2, p1lo = 0, p1hi = 0, p2lo = 0, p2hi = 0;
    uint32_t key0[2], key1[2], key2[2], p1key[2] = {NOKEY, NOKEY}, p2key[2] = {NOKEY, NOKEY};
    float val0[2], val1[2], val2[2], sd0, sd1, sd2;
    auto ld_entries = [&](uint32_t lo, uint32_t hi, uint32_t* key, float* val) {
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const uint32_t e = lo + lane + 32 * q;
        key[q] = e < hi ? (uint32_t)__ldg(keys + e) : NOKEY;
        val[q] = e < hi ? __ldg(bvals + e) : 0.f;
      }
    };
    const float gscale = pb.gram_scale;   // power of two: keeps sqrt(d) x in e4m3's normal range; undone exactly by chol_prep
    auto ld_sd = [&](int k) -> float {
      const long long r = (ks0 + k) * SK + lane;
      return (k < nk && r < n) ? sdv[r] * gscale : 0.f;   // sdvec is rewritten by K1 between builds: a plain load
    };
    auto to_e4m3 = [](float x) -> uint32_t { return (uint32_t)__nv_cvt_float_to_fp8(x, __NV_SATFINITE, __NV_E4M3); };
    const uint32_t smem_base_u32 = smem_u32(smem);
    {
      const uint32_t oa = ld_offs(grp), ob = ld_offs(grp + S_NGRP);
      lo0 = __shfl_sync(0xffffffffu, oa, 0); hi0 = __shfl_sync(0xffffffffu, oa, 1);
      lo1 = __shfl_sync(0xffffffffu, ob, 0); hi1 = __shfl_sync(0xffffffffu, ob, 1);
    }
    uint32_t o_c = ld_offs(grp + 2 * S_NGRP);
    ld_entries(lo0, hi0, key0, val0); sd0 = ld_sd(grp);
    ld_entries(lo1, hi1, key1, val1); sd1 = ld_sd(grp + S_NGRP);
    bool p1row = false, p2row = false;
    for (int k = grp, use = 0; k < nk; k += S_NGRP, use++) {
      const int st = k % S_SST;
      const uint32_t sbase = smem_base_u32 + (uint32_t)st * (uint32_t)S_STAGE_BYTES + (uint32_t)strm_off;   // shared-space address
      // ---- un-write what the previous use of THIS STAGE (two uses ago) stored (same addresses, zero)
      const int fill = k / S_SST;   // how many times this stage has been filled before
      if (fill > 0) {
        mbar_wait(&empty_bar[st], (uint32_t)((fill - 1) & 1));
#pragma unroll
        for (int q = 0; q < 2; q++)
          if (p2key[q] != NOKEY) sts_u8(sbase + p2key[q], 0u);
        for (uint32_t e0 = p2lo + 64; e0 < p2hi; e0 += 32) {
          const uint32_t e = e0 + lane;
          if (e < p2hi) sts_u8(sbase + (uint32_t)__ldg(keys + e), 0u);
        }
        if (p2row && has_bias_col) sts_u8(sbase + bias_off, 0u);
      }
      // ---- write this use
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const bool v = key0[q] != NOKEY;
        const uint32_t key = v ? key0[q] : 0u;
        const float sdk = __shfl_sync(0xffffffffu, sd0, (key >> 7) & 31);
        if (v) sts_u8(sbase + key, to_e4m3(val0[q] * sdk));
      }
      for (uint32_t e0 = lo0 + 64; e0 < hi0; e0 += 32) {
        const uint32_t e = e0 + lane;
        const bool v = e < hi0;
        const uint32_t key = v ? (uint32_t)__ldg(keys + e) : 0u;
        const float val = v ? __ldg(bvals + e) : 0.f;
        const float sdk = __shfl_sync(0xffffffffu, sd0, (key >> 7) & 31);
        if (v) sts_u8(sbase + key, to_e4m3(val * sdk));
      }
      const bool row_now = (ks0 + k) * SK + lane < n;
      if (row_now && has_bias_col) sts_u8(sbase + bias_off, to_e4m3(sd0));
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(full0_remote + (uint32_t)st * 8u);
      // ---- issue the loads of the use after next.  AFTER the hand-over, not before this use's stores: the fence above compiles to
      // MEMBAR.ALL.CTA, which waits for every load this thread still has in flight -- issued at the top of the use they would
      // make each hand-over wait out a DRAM round trip; issued here they have the whole next use to arrive.
      lo2 = __shfl_sync(0xffffffffu, o_c, 0); hi2 = __shfl_sync(0xffffffffu, o_c, 1);
      o_c = ld_offs(k + 3 * S_NGRP);
      ld_entries(lo2, hi2, key2, val2); sd2 = ld_sd(k + 2 * S_NGRP);
      // ---- rotate
      p2lo = p1lo; p2hi = p1hi; p2row = p1row; p1lo = lo0; p1hi = hi0; p1row = row_now;
      lo0 = lo1; hi0 = hi1; lo1 = lo2; hi1 = hi2;
#pragma unroll
      for (int q = 0; q < 2; q++) { p2key[q] = p1key[q]; p1key[q] = key0[q]; key0[q] = key1[q]; val0[q] = val1[q]; key1[q] = key2[q]; val1[q] = val2[q]; }
      sd0 = sd1; sd1 = sd2;
    }
  } else {
    // ===== epilogue: the last four warps -> TMEM lane quadrant (warp % 4); each CTA of the pair holds its own 128 rows of the tile =====
    const int quad = warp & 3;
    float* out = pb.Hpart + (size_t)slice * Dp * Dp;
    const int row = tile_bi * GM + quad * 32 + lane;
    if (nk > 0) {
      while (!mbar_try_wait(acc_bar, 0)) __nanosleep(512);   // the whole main loop long: do not spend issue slots on polling
      tc_fence_after();
    }
#pragma unroll 1
    for (int c0 = 0; c0 < GN; c0 += 32) {
      uint32_t r[32];
      if (nk > 0) {
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, r);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; j++) r[j] = 0u;
      }
      const int col = tile_bj * GN + c0;
      if (row < Dp && col < Dp) {
        float4* dst = reinterpret_cast<float4*>(out + (size_t)row * Dp + col);
#pragma unroll
        for (int j = 0; j < 8; j++)
          dst[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                               __uint_as_float(r[4 * j + 3]));
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  cluster_sync_all();   // neither CTA may leave (or free its TMEM) while the pair's MMAs, commits or remote arrives can still touch it
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, GN);
  }
}

// Block-major entry list for the CSR Gram.  For every 128-column block b and every 32-row group g the entries
// (row in group, column in block, value) are stored contiguously at [offs[b*ngroups+g], offs[b*ngroups+g+1]); the key is
// the byte offset of the element inside a swizzled [32 k][128 col] operand block (sw128_off), the value the stored float.
// Rows must be sorted by column (strictly increasing), which the upload checks.
__global__ void __launch_bounds__(256) csr_bm_count_kernel(long long n, const long long* __restrict__ rowptr, const int* __restrict__ colidx,
                                                           int nblk, long long ngroups, long long* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < ngroups; g += nw) {
    const long long r = g * 32 + lane;
    long long j = r < n ? rowptr[r] : 0;
    const long long j1 = r < n ? rowptr[r + 1] : 0;
    for (int b = 0; b < nblk; b++) {
      const long long s = j;
      while (j < j1 && colidx[j] < (b + 1) * 128) j++;
      int c = (int)(j - s);
      c = __reduce_add_sync(0xffffffffu, c);
      if (lane == 0) counts[(size_t)b * ngroups + g] = c;
    }
  }
}

__global__ void __launch_bounds__(256) csr_bm_fill_kernel(long long n, const long long* __restrict__ rowptr, const int* __restrict__ colidx,
                                                          const float* __restrict__ vals, int nblk, long long ngroups,
                                                          const long long* __restrict__ offs, unsigned short* __restrict__ keys,
                                                          float* __restrict__ bvals) {
  const int lane = threadIdx.x & 31;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < ngroups; g += nw) {
    const long long r = g * 32 + lane;
    long long j = r < n ? rowptr[r] : 0;
    const long long j1 = r < n ? rowptr[r + 1] : 0;
    for (int b = 0; b < nblk; b++) {
      const long long s = j;
      while (j < j1 && colidx[j] < (b + 1) * 128) j++;
      const int c = (int)(j - s);
      int incl = c;   // inclusive warp scan
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
      }
      long long pos = offs[(size_t)b * ngroups + g] + (incl - c);
      for (long long e = s; e < j; e++, pos++) {
        keys[pos] = (unsigned short)sw128_off(lane, colidx[e] - b * 128);
        bvals[pos] = vals[e];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// fp32 SIMT debug kernel: same operand (bf16 Xt), same output format (slice 0; other slices zeroed).
// 64x64 lower tiles, 256 threads x (4x4).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gram_simt_kernel(const Problem* __restrict__ probs, int force) {
  const Problem& pb = probs[blockIdx.z];
  Ctrl* ctrl = pb.ctrl;
  if (!force && (ctrl->done || !ctrl->need_hess)) return;
  if (blockIdx.x > blockIdx.y) return;
  const int Dp = pb.Dp;
  const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
  __shared__ float Ai[16][64 + 1];
  __shared__ float Aj[16][64 + 1];
  const int tid = threadIdx.x;
  const int ti = (tid / 16) * 4, tj = (tid % 16) * 4;
  float acc[4][4] = {};
  for (long long r0 = 0; r0 < pb.n; r0 += 16) {
    for (int e = tid; e < 16 * 64; e += 256) {
      const int r = e / 64, c = e % 64;
      const long long rr = r0 + r;
      Ai[r][c] = rr < pb.n ? __bfloat162float(pb.Xt[(size_t)rr * Dp + i0 + c]) : 0.f;
      Aj[r][c] = rr < pb.n ? __bfloat162float(pb.Xt[(size_t)rr * Dp + j0 + c]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 16; r++) {
      float x[4], y[4];
#pragma unroll
      for (int a = 0; a < 4; a++) { x[a] = Ai[r][ti + a]; y[a] = Aj[r][tj + a]; }
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = fmaf(x[a], y[b], acc[a][b]);
    }
    __syncthreads();
  }
  for (int s = 0; s < pb.gram_slices; s++) {
    float* out = pb.Hpart + (size_t)s * Dp * Dp;
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) out[(size_t)(i0 + ti + a) * Dp + j0 + tj + b] = (s == 0) ? acc[a][b] : 0.f;
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Tensor map over Xt [n][Dp] bf16 row-major: dim0 = feature (contiguous), dim1 = row; box 64 x GK, 128B swizzle.
int gram_make_tensor_map(void* out_map_host /*CUtensorMap, 128 B*/, const void* xt, long long n, int Dp) {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || !p) return 1;
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  cuuint64_t dims[2] = {(cuuint64_t)Dp, (cuuint64_t)n};
  cuuint64_t strides[1] = {(cuuint64_t)Dp * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)GK};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(reinterpret_cast<CUtensorMap*>(out_map_host), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(xt), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 2;
}

// Lower block-triangle tile list for a Dp x Dp output (Dp multiple of 128): 128 x 256 tiles (bi, bj), or, for the CTA-pair CSR
// kernel, 256 x 256 tiles (BI, bj) whose two row blocks 2 BI and 2 BI + 1 belong to the two CTAs of the pair.
int gram_tile_list(int Dp, short* bi_bj_pairs /*[2*max]*/, int max_tiles, int pair_tiles) {
  int n = 0;
  const int rows = pair_tiles ? 2 * GM : GM;
  const int nbi = (Dp + rows - 1) / rows, nbj = (Dp + GN - 1) / GN;
  for (int bi = 0; bi < nbi; bi++)
    for (int bj = 0; bj < nbj; bj++)
      if (bj * GN <= bi * rows + rows - 1) {
        if (n >= max_tiles) return -1;
        bi_bj_pairs[2 * n] = (short)bi; bi_bj_pairs[2 * n + 1] = (short)bj; n++;
      }
  return n;
}

cudaError_t gram_launch_tcgen05(const Problem* d_probs, int nprob, const void* d_tmaps, const void* d_tiles, int ntiles,
                                int nslices, int force, cudaStream_t st, int* launches, int share) {
  {
    // the attribute is per device: set it once for every device this process launches on
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
      cudaError_t e = cudaFuncSetAttribute(gram_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_SMEM);
      if (e != cudaSuccess) return e;
      if (dev >= 0 && dev < 64) configured[dev] = true;
    }
  }
  gram_tcgen05_kernel<<<dim3(ntiles, nslices, nprob), G_THREADS, G_SMEM, st>>>(
      d_probs, reinterpret_cast<const CUtensorMap*>(d_tmaps), reinterpret_cast<const GramTile*>(d_tiles), ntiles, force, share);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// d_tiles holds 256 x 256 pair tiles (gram_tile_list(..., 1)); the grid is a list of 2-CTA clusters along x.
cudaError_t gram_launch_csr_tcgen05(const Problem* d_probs, int nprob, const void* d_tiles, int ntiles, int nslices, int force,
                                    int bias_col, cudaStream_t st, int* launches, int share) {
  {
    // the attribute is per device: set it once for every device this process launches on
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
      cudaError_t e = cudaFuncSetAttribute(gram_csr_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_SMEM);
      if (e != cudaSuccess) return e;
      if (dev >= 0 && dev < 64) configured[dev] = true;
    }
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * ntiles, nslices, nprob);
  cfg.blockDim = dim3(S_THREADS, 1, 1);
  cfg.dynamicSmemBytes = S_SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, gram_csr_tcgen05_kernel, d_probs, reinterpret_cast<const GramTile*>(d_tiles), ntiles, force, bias_col, share);
  if (e != cudaSuccess) return e;
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// counts -> exclusive offsets in place: offs has nblk*ngroups+1 entries (the last one = total entries)
cudaError_t csr_bm_offsets(long long n, const long long* rowptr, const int* colidx, int nblk, long long ngroups, long long* offs,
                           cudaStream_t st) {
  const long long m = (long long)nblk * ngroups;
  cudaError_t e = cudaMemsetAsync(offs, 0, (size_t)(m + 1) * sizeof(long long), st);
  if (e != cudaSuccess) return e;
  const int grid = (int)std::min<long long>((ngroups + 7) / 8, 148 * 32);
  csr_bm_count_kernel<<<std::max(grid, 1), 256, 0, st>>>(n, rowptr, colidx, nblk, ngroups, offs);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  size_t tmp_bytes = 0;
  if ((e = cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, offs, offs, (long long)(m + 1), st)) != cudaSuccess) return e;
  void* tmp = nullptr;
  if ((e = cudaMallocAsync(&tmp, tmp_bytes ? tmp_bytes : 16, st)) != cudaSuccess) return e;   // stream-ordered: no device-wide wait
  e = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, offs, offs, (long long)(m + 1), st);
  cudaError_t e2 = cudaFreeAsync(tmp, st);
  return e != cudaSuccess ? e : e2;
}

cudaError_t csr_bm_fill(long long n, const long long* rowptr, const int* colidx, const float* vals, int nblk, long long ngroups,
                        const long long* offs, unsigned short* keys, float* bvals, cudaStream_t st) {
  const int grid = (int)std::min<long long>((ngroups + 7) / 8, 148 * 32);
  csr_bm_fill_kernel<<<std::max(grid, 1), 256, 0, st>>>(n, rowptr, colidx, vals, nblk, ngroups, offs, keys, bvals);
  return cudaGetLastError();
}

cudaError_t gram_launch_simt(const Problem* d_probs, int nprob, int Dp, int force, cudaStream_t st, int* launches) {
  const int T = Dp / 64;
  gram_simt_kernel<<<dim3(T, T, nprob), 256, 0, st>>>(d_probs, force);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

}  // namespace mlease
