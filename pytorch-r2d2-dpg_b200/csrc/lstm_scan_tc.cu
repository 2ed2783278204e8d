// tcgen05 / TMEM version of the persistent cluster LSTM scan (forward + BPTT) for sm_100a.
//
// Same decomposition as the mma.sync kernels in lstm_scan.cu (cluster of C = H/32 CTAs per <= 32 batch rows,
// CTA `rank` owns hidden units [32 rank, 32 rank + 32) = 128 gate rows of W_hh), but
//   * the W_hh slice is written ONCE into tensor memory (bf16 hi/lo planes, tcgen05.st) and stays there as the A
//     operand of every step; per cell step one elected thread issues (H/16) x 3 tcgen05.mma (M=128 gate rows,
//     N = 16 | 32 batch columns, K=16; passes lo*hi, hi*lo, hi*hi; B = the h tile in shared memory) that accumulate in
//     TMEM; tcgen05.commit -> mbarrier tells the cell warps;
//   * the cell warps read the accumulator with tcgen05.ld (lane = gate row), transpose it through shared memory,
//     finish the LSTM cell in registers and stage h_t (bf16 hi/lo, already in the operand layout of the next step);
//   * the h_t all-gather inside the cluster is bulk shared->remote-shared copies (cp.async.bulk.shared::cluster)
//     that complete transaction bytes on the DESTINATION's mbarrier: no cluster-wide barrier and no memory fence
//     on the global stores of gates / h / c on the serial chain (the v1 kernel spent 24% of its samples in the
//     barrier's release fence, profiles/r01_*);
//   * lstm_scan_fwd_pp_kernel (clusters with 17..32 rows, the cfg-2 case) alternates two <= 16-row sub-tiles through
//     this pipeline with a dedicated MMA warp.
// Backward: P[H x NB] = W_slice^T [H x 128] * dG^T via tcgen05 (W^T tiles in TMEM), fp32 partial sums reduce-scattered
// with bulk copies; dG also leaves as the packed operand images of the GEMMs that consume it, bias sums fused.
#include <cooperative_groups.h>
#include <stdlib.h>

#include <map>
#include <mutex>

#include "lstm_scan.cuh"
#include "tc05.cuh"

namespace cg = cooperative_groups;

namespace r2d2 {

int* scan_error_flag();  // device int, 0 = ok (defined below)
unsigned char* scan_xchg_scratch(size_t* bytes);   // per-device global scratch of the H = 512 exchanges through L2

namespace {

constexpr int TC_THREADS = 512, TC_WARPS = 16;
#ifndef R2D2_SCAN_NACC
#define R2D2_SCAN_NACC 1   // TMEM accumulators per tile (>1: independent chains summed in the epilogue; measured: no gain, 4x the tcgen05.ld traffic)
#endif
constexpr int GT_LD = 128 + 4;

// Cell non-linearities on the serial chain: exp via MUFU.EX2 (__expf, ~2 ulp) and an approximate reciprocal
// (1 ulp); absolute error ~1e-7, far below the bf16x3 operand split (~1e-5) and the 1e-3 parity bar.  The
// library versions (expf / tanhf / IEEE divide) cost ~0.85 us per step here: two dependent elements per thread.
__device__ __forceinline__ float fast_sigmoid(float x) { return tc::sigmoid_fast(x); }
__device__ __forceinline__ float fast_tanh(float x) { return tc::tanh_fast(x); }

__device__ __forceinline__ long long gtime() {
  long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define TRACE_STAMP(slot) do { if (p.trace && tid == 0) p.trace[((size_t)blockIdx.x * S + s) * 8 + (slot)] = gtime(); } while (0)

__device__ __forceinline__ void split8_store(const float4 v0, const float4 v1, unsigned char* hi_dst, unsigned char* lo_dst) {
  uint4 h, l;
  split_pack2(v0.x, v0.y, h.x, l.x);
  split_pack2(v0.z, v0.w, h.y, l.y);
  split_pack2(v1.x, v1.y, h.z, l.z);
  split_pack2(v1.z, v1.w, h.w, l.w);
  *reinterpret_cast<uint4*>(hi_dst) = h;
  *reinterpret_cast<uint4*>(lo_dst) = l;
}

template <int H, int NB>
struct TcFwdSmem {
  static constexpr int C = H / 32, KC = H / 8, RG = NB / 8;
  // h operand tile, ROW-GROUP major so that (a) only row groups that hold real batch rows travel through DSMEM and
  // (b) a row group can leave as soon as its cells are done:  [buf][row group g][slice r = source CTA][plane hi/lo]
  // [4 k-chunks][8 rows][16 B]  ->  MMA descriptor LBO (k-chunk stride) = 128, SBO (row-group stride) = C*1024
  static constexpr int SLICE = 1024;                 // one CTA's 32 units x 8 rows x (hi+lo)
  static constexpr int RG_BYTES = C * SLICE;
  static constexpr int BUF_BYTES = RG * RG_BYTES;    // = NB * H * 4
  static constexpr int OFF_HB = 0;
  static constexpr int NACC = (H / 16) < R2D2_SCAN_NACC ? (H / 16) : R2D2_SCAN_NACC;
  // tensor memory columns: NACC independent accumulators D_a at [a*NB, ..), then the W_hh slice: hi plane at TM_A_HI
  // (H/2 columns: two bf16 per column), lo plane after it.  H = 512 (BIG): hi + lo of a 128 x 512 slice are the whole
  // 512 columns, so the accumulators get 64 columns, the lo plane keeps its first KS_TM_LO k-steps in tensor memory
  // and the last KS_TAIL k-steps live in shared memory (SS-mode MMAs: same instruction, A through a descriptor)
  static constexpr bool BIG = H > 256;
  static constexpr int TM_A_HI = BIG ? 64 : 128, TM_A_LO = TM_A_HI + H / 2, TM_COLS = 512;
  static constexpr int KS_TM_LO = BIG ? (TM_COLS - TM_A_LO) / 8 : H / 16, KS_TAIL = H / 16 - KS_TM_LO;
  static_assert(NACC * NB <= TM_A_HI, "accumulators overlap the weight slice in tensor memory");
  static constexpr int OFF_GT = OFF_HB + 2 * BUF_BYTES;            // fp32 [NB][GT_LD]
  static constexpr int OFF_HSTAGE = OFF_GT + NB * GT_LD * 4;       // [dbuf][row group][plane][4 chunks][8][16 B]
  static constexpr int OFF_BAR = OFF_HSTAGE + 2 * RG * SLICE;      // 3 mbarriers + tmem slot + dead flag
  // lo-plane tail of W_hh: per k-step one 4 KB K-major block [2 k-chunks][16 row groups][8 rows][16 B]
  // (descriptor LBO = 2048, SBO = 128)
  static constexpr int OFF_WTAIL = OFF_BAR + 128;
  static constexpr int BYTES = OFF_WTAIL + KS_TAIL * 4096;
  static_assert(BYTES <= 232448, "forward scan tile does not fit in 227 KB of shared memory");
  static_assert(OFF_WTAIL % 128 == 0, "descriptor alignment");
};

template <int H, int NB>
__global__ void __launch_bounds__(TC_THREADS, 1) lstm_scan_fwd_tc_kernel(ScanFwdParams p, int* err) {
  using SM = TcFwdSmem<H, NB>;
  constexpr int C = SM::C, KC = SM::KC, KS = H / 16, RG = SM::RG, NT = RG / 2;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int b0 = (blockIdx.x / C) * p.rows_per_cluster;  // this cluster's batch rows [b0, b_end), at most NB of them
  const int b_end = min(p.B, b0 + p.rows_per_cluster);
  const int n_rg_valid = (b_end - b0 + 7) >> 3;          // row groups that carry real rows
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int w_u = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp-uniform warp index (role dispatch)
  const int r8 = w & 7, half = w >> 3;                   // pointwise role: row r8 of row groups e = half, half+2, ...
  const int B = p.B, S = p.T * p.repeat;

  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* hb = smem + SM::OFF_HB;
  float* gt = reinterpret_cast<float*>(smem + SM::OFF_GT);
  unsigned char* hstage = smem + SM::OFF_HSTAGE;
  uint64_t* h_full = reinterpret_cast<uint64_t*>(smem + SM::OFF_BAR);  // [2]
  uint64_t* mma_done = h_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_done + 1);
  volatile int* dead = reinterpret_cast<volatile int*>(tmem_slot + 1);

  if (tid == 0) {
    tc::mbar_init(&h_full[0], 1);
    tc::mbar_init(&h_full[1], 1);
    tc::mbar_init(mma_done, 1);
    tc::fence_mbar_init_cluster();
    *dead = 0;
  }
  if (w == 1) { __syncwarp(); tc::tmem_alloc(tmem_slot, SM::TM_COLS); }
  // ---- initial h tile (all H units of my rows) -> operand buffer 0 (zeros for rows past b_end)
  for (int idx = tid; idx < NB * KC; idx += TC_THREADS) {
    const int n = idx % NB, kc = idx / NB, b = b0 + n;
    float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
    if (b < b_end && p.h0) {
      const float* src = p.h0 + (size_t)b * H + kc * 8;
      v0 = __ldg(reinterpret_cast<const float4*>(src));
      v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
    }
    unsigned char* dst = hb + (n >> 3) * SM::RG_BYTES + (kc >> 2) * SM::SLICE + (kc & 3) * 128 + (n & 7) * 16;
    split8_store(v0, v1, dst, dst + 512);
  }
  const int ug = rank * 32 + lane;
  float cst[NT];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int b = b0 + 8 * (half + 2 * j) + r8;
    cst[j] = 0.f;
    if (b < b_end) {
      const float hv = p.h0 ? __ldg(p.h0 + (size_t)b * H + ug) : 0.f;
      const float cv = p.c0 ? __ldg(p.c0 + (size_t)b * H + ug) : 0.f;
      p.hs[(size_t)b * H + ug] = hv;
      p.cs[(size_t)b * H + ug] = cv;
      cst[j] = cv;
    }
  }
  tc::fence_proxy_async_smem();
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  // ---- W_hh slice -> TENSOR MEMORY, resident for the whole launch: TMEM lane r = local gate row (gate = r/32 =
  // lane quarter, unit = r%32), columns = K packed two bf16 per 32-bit word (hi plane, then lo plane).
  {
    const int q = w & 3;
    const float* wrow = p.whh + (size_t)(q * H + rank * 32 + lane) * H;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    __syncwarp();
#pragma unroll 1
    for (int ks = (w >> 2); ks < KS; ks += TC_WARPS / 4) {
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(wrow + ks * 16 + i * 4));
        split_pack2(v.x, v.y, hi[2 * i], lo[2 * i]);
        split_pack2(v.z, v.w, hi[2 * i + 1], lo[2 * i + 1]);
      }
      tc::tmem_st_32x32b_x8(lane_base + SM::TM_A_HI + ks * 8, hi);
      if (ks < SM::KS_TM_LO) {
        tc::tmem_st_32x32b_x8(lane_base + SM::TM_A_LO + ks * 8, lo);
      } else {   // lo-plane tail -> shared memory, K-major core matrices: row = local gate row q*32 + lane
        unsigned char* d = smem + SM::OFF_WTAIL + (ks - SM::KS_TM_LO) * 4096 + (q * 4 + (lane >> 3)) * 128 + (lane & 7) * 16;
        *reinterpret_cast<uint4*>(d) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        *reinterpret_cast<uint4*>(d + 2048) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
      }
    }
    tc::tmem_wait_st();
  }
  tc::fence_proxy_async_smem();
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  cluster.sync();  // every CTA's barriers are initialised before any remote copy can target them

  const uint32_t idesc = tc::make_idesc_bf16_f32(128, NB);
  const uint32_t hb_addr = tc::smem_u32(hb);
  // the operand descriptor is loop invariant up to its 16-byte start-address field: build once, add offsets per k-step
  const uint64_t db_hi0 = tc::make_smem_desc(hb_addr, 128, SM::RG_BYTES);   // buffer 0, slice 0, plane hi
  const uint64_t wtail_desc0 = tc::make_smem_desc(tc::smem_u32(smem + SM::OFF_WTAIL), 2048, 128);
  const size_t gstride = (size_t)4 * H;
  const uint32_t step_tx = (uint32_t)(C * n_rg_valid * SM::SLICE);

  for (int s = 0; s < S; ++s) {
    const int cur = s & 1, nxt = cur ^ 1;
    const int t = s / p.repeat;

    float gpre[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const int b = b0 + 8 * (half + 2 * j) + r8;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        gpre[j][q] = (b < b_end) ? p.gin[((size_t)t * B + b) * gstride + q * H + ug] : 0.f;  // plain load: gates may alias gin
    }

    TRACE_STAMP(0);
    if (w_u == 0) {  // MMA warp (warp-uniform branch); one elected lane issues
      if (s + 1 < S && tc::elect_one()) tc::mbar_arrive_expect_tx(&h_full[nxt], step_tx);  // h_s of all C CTAs -> buffer nxt
      if (s > 0 && !*dead) {
        if (!tc::mbar_wait(&h_full[cur], ((s - 1) >> 1) & 1)) { *dead = 1; atomicExch(err, 1); }
      }
      __syncwarp();
      TRACE_STAMP(1);
      tc::fence_after_thread_sync();
      const uint64_t db_cur = db_hi0 + (uint64_t)((cur * SM::BUF_BYTES) >> 4);
      if (tc::elect_one()) {
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const uint32_t ta_hi = tmem_base + SM::TM_A_HI + ks * 8, ta_lo = tmem_base + SM::TM_A_LO + ks * 8;
        const uint64_t db_hi = db_cur + (uint64_t)(((ks >> 1) * SM::SLICE + (ks & 1) * 256) >> 4);
        const uint64_t db_lo = db_hi + (uint64_t)(512 >> 4);
        const uint32_t d = tmem_base + (ks % SM::NACC) * NB;
        if (ks < SM::KS_TM_LO) tc::mma_bf16_ts(d, ta_lo, db_hi, idesc, ks >= SM::NACC);
        else tc::mma_bf16_ss(d, wtail_desc0 + (uint64_t)(((ks - SM::KS_TM_LO) * 4096) >> 4), db_hi, idesc, ks >= SM::NACC);
        tc::mma_bf16_ts(d, ta_hi, db_lo, idesc, true);
        tc::mma_bf16_ts(d, ta_hi, db_hi, idesc, true);
      }
      tc::mma_commit(mma_done);
      }
      __syncwarp();
      TRACE_STAMP(2);
    }
    if (!*dead) {
      if (!tc::mbar_wait(mma_done, s & 1)) { *dead = 1; atomicExch(err, 2); }
    }
    TRACE_STAMP(3);
    tc::fence_after_thread_sync();
    __syncwarp();  // tcgen05.ld is .sync.aligned: reconverge after the spin wait

    // ---- accumulator -> gate tile: warp w reads TMEM lanes 32*(w&3).. (gate w&3, unit = lane), 8-column block w>>2
    if ((w >> 2) * 8 < NB) {
      const int q = w & 3, c0 = (w >> 2) * 8;
      float v[8];
      tc::tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
      for (int a = 1; a < SM::NACC; ++a) {
        float u[8];
        tc::tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * NB + c0), u);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] += u[j];
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) gt[(c0 + j) * GT_LD + q * 32 + lane] = v[j];
    }
    tc::fence_before_thread_sync();
    __syncthreads();
    TRACE_STAMP(4);

    // ---- pointwise LSTM cell, one row group at a time: thread = (unit = lane, row r8 of group e); as soon as the 8
    // warps of this half have finished a group, its 1 KB slice (hi+lo) leaves for every CTA of the cluster, overlapping
    // the DSMEM transfer (~20 B/clk/SM) with the cells of the next group and with the other half's work
    unsigned char* hs_buf = hstage + (s & 1) * RG * SM::SLICE;
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const int e = half + 2 * j;
      if (e < n_rg_valid) {
        const int n = 8 * e + r8, b = b0 + n;
        __nv_bfloat16 hi = __float2bfloat16_rn(0.f), lo = hi;
        float ig = 0.f, fg = 0.f, gg = 0.f, og = 0.f, cn = 0.f, hn = 0.f;
        const bool on = b < b_end;
        if (on) {
          const float* gr = gt + n * GT_LD + lane;
          ig = fast_sigmoid(gr[0] + gpre[j][0]);
          fg = fast_sigmoid(gr[32] + gpre[j][1]);
          gg = fast_tanh(gr[64] + gpre[j][2]);
          og = fast_sigmoid(gr[96] + gpre[j][3]);
          cn = fg * cst[j] + ig * gg;
          hn = og * fast_tanh(cn);
          cst[j] = cn;
          split_bf16(hn, hi, lo);
        }
        unsigned char* dst = hs_buf + e * SM::SLICE + (lane >> 3) * 128 + r8 * 16 + (lane & 7) * 2;  // [plane][chunk][row][8]
        *reinterpret_cast<__nv_bfloat16*>(dst) = hi;
        *reinterpret_cast<__nv_bfloat16*>(dst + 512) = lo;
        tc::fence_proxy_async_smem();
        asm volatile("bar.sync %0, 256;" ::"r"(1 + half) : "memory");   // the 8 warps that own this row group
        if (s + 1 < S && r8 < C && tc::elect_one()) {
          const uint32_t dst_local = hb_addr + nxt * SM::BUF_BYTES + e * SM::RG_BYTES + rank * SM::SLICE;
#pragma unroll
          for (uint32_t d = r8; d < (uint32_t)C; d += 8)   // 8 warps per row group: one (C <= 8) or two (C = 16) destinations each
            tc::bulk_copy_to_cluster(tc::mapa(dst_local, d), tc::smem_u32(hs_buf + e * SM::SLICE), SM::SLICE,
                                     tc::mapa(tc::smem_u32(&h_full[nxt]), d));
        }
        if (on) {   // saved activations leave after the exchange has been started: off the serial chain
          float* go = p.gates + ((size_t)s * B + b) * gstride + ug;
          go[0] = ig; go[H] = fg; go[2 * H] = gg; go[3 * H] = og;
          p.hs[((size_t)(s + 1) * B + b) * H + ug] = hn;
          p.cs[((size_t)(s + 1) * B + b) * H + ug] = cn;
          if (p.head_in && (s % p.repeat) == p.repeat - 1)
            p.head_in[((size_t)t * B + b) * H + ug] = fast_tanh(hn);
        }
      }
    }
    TRACE_STAMP(7);
  }
  tc::fence_before_thread_sync();
  cluster.sync();
  if (w == 1) { __syncwarp(); tc::tmem_dealloc(tmem_base, SM::TM_COLS); }
}

// ------------------------------------------------------------------------------------------------
// forward, ping-pong variant for clusters that own 17..32 batch rows: the rows are split into two sub-tiles of
// <= 16 rows (one N=16 MMA tile each) that alternate through the pipeline, so the DSMEM all-gather and the cell math
// of one sub-tile overlap with the tensor-core step of the other.  A dedicated 17th warp issues the MMAs; the 16
// cell warps never block on the exchange.  Iteration k handles sub-tile k % 2 of cell step k / 2.
// ------------------------------------------------------------------------------------------------
constexpr int PP_THREADS = 544, PP_CELL_WARPS = 16;

template <int H>
struct PpFwdSmem {
  static constexpr int C = H / 32, KC = H / 8;
  static constexpr int SLICE = 1024;                      // one CTA's 32 units x 8 rows x (hi+lo)
  static constexpr int RG_BYTES = C * SLICE;
  static constexpr int BUF_BYTES = 2 * RG_BYTES;          // 16 rows
  static constexpr int OFF_HB = 0;                        // [sub][buf][row group][slice][plane][4 chunks][8][16 B]
  static constexpr int TM_A_HI = 128, TM_A_LO = 128 + H / 2, TM_COLS = 512;   // D[sub][acc] at (sub*4 + acc)*16
  static constexpr int OFF_GT = OFF_HB + 4 * BUF_BYTES;   // fp32 [2 (iteration parity)][16][GT_LD]
  static constexpr int OFF_HSTAGE = OFF_GT + 2 * 16 * GT_LD * 4;   // [sub][step parity][row group][SLICE]
  static constexpr int OFF_BAR = OFF_HSTAGE + 8 * SLICE;  // h_full[sub][2], mma_done[sub], tmem slot, dead
  static constexpr int BYTES = OFF_BAR + 96;
  static_assert(BYTES <= 232448, "ping-pong scan tile does not fit in shared memory");
};

template <int H, bool TRACE>
__global__ void __launch_bounds__(PP_THREADS, 1) lstm_scan_fwd_pp_kernel(ScanFwdParams p, int* err) {
  using SM = PpFwdSmem<H>;
  constexpr int C = SM::C, KC = SM::KC, KS = H / 16;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int b0 = (blockIdx.x / C) * p.rows_per_cluster;
  const int b_end = min(p.B, b0 + p.rows_per_cluster);
  const int n_rows = b_end - b0;                                   // 1..32
  const int n_sub = n_rows > 16 ? 2 : 1;
  const int rows0 = n_sub == 2 ? (n_rows + 1) / 2 : n_rows;         // rows of sub-tile 0; sub-tile 1 gets the rest
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int w_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int B = p.B, S = p.T * p.repeat;

  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* hb = smem + SM::OFF_HB;
  float* gt_all = reinterpret_cast<float*>(smem + SM::OFF_GT);
  unsigned char* hstage = smem + SM::OFF_HSTAGE;
  uint64_t* h_full = reinterpret_cast<uint64_t*>(smem + SM::OFF_BAR);   // [sub][2]
  uint64_t* mma_done = h_full + 4;                                      // [sub]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_done + 2);
  volatile int* dead = reinterpret_cast<volatile int*>(tmem_slot + 1);

  if (tid == 0) {
    for (int i = 0; i < 4; ++i) tc::mbar_init(&h_full[i], 1);
    tc::mbar_init(&mma_done[0], 1);
    tc::mbar_init(&mma_done[1], 1);
    tc::fence_mbar_init_cluster();
    *dead = 0;
  }
  if (w == 1) { __syncwarp(); tc::tmem_alloc(tmem_slot, SM::TM_COLS); }
  auto sub_row0 = [&](int sub) { return sub == 0 ? 0 : rows0; };          // first cluster-local row of a sub-tile
  auto sub_rows = [&](int sub) { return sub == 0 ? rows0 : n_rows - rows0; };
  // ---- initial h tiles -> buffer 0 of each sub-tile (zeros for rows that do not exist)
  for (int idx = tid; idx < 2 * 16 * KC; idx += PP_THREADS) {
    const int sub = idx / (16 * KC), rem = idx % (16 * KC);
    const int n = rem % 16, kc = rem / 16;
    const int b = b0 + sub_row0(sub) + n;
    float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
    if (sub < n_sub && n < sub_rows(sub) && p.h0) {
      const float* src = p.h0 + (size_t)b * H + kc * 8;
      v0 = __ldg(reinterpret_cast<const float4*>(src));
      v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
    }
    unsigned char* dst = hb + (sub * 2 + 0) * SM::BUF_BYTES + (n >> 3) * SM::RG_BYTES + (kc >> 2) * SM::SLICE + (kc & 3) * 128 + (n & 7) * 16;
    split8_store(v0, v1, dst, dst + 512);
  }
  const int ug = rank * 32 + lane;
  float cst[2] = {0.f, 0.f};
  if (w < PP_CELL_WARPS) {
#pragma unroll
    for (int sub = 0; sub < 2; ++sub) {
      if (sub < n_sub && w < sub_rows(sub)) {
        const int b = b0 + sub_row0(sub) + w;
        const float hv = p.h0 ? __ldg(p.h0 + (size_t)b * H + ug) : 0.f;
        const float cv = p.c0 ? __ldg(p.c0 + (size_t)b * H + ug) : 0.f;
        p.hs[(size_t)b * H + ug] = hv;
        p.cs[(size_t)b * H + ug] = cv;
        cst[sub] = cv;
      }
    }
  }
  tc::fence_proxy_async_smem();
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  if (w < PP_CELL_WARPS) {   // W_hh slice -> tensor memory (as in the single-tile kernel)
    const int q = w & 3;
    const float* wrow = p.whh + (size_t)(q * H + rank * 32 + lane) * H;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    __syncwarp();
#pragma unroll 1
    for (int ks = (w >> 2); ks < KS; ks += PP_CELL_WARPS / 4) {
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(wrow + ks * 16 + i * 4));
        split_pack2(v.x, v.y, hi[2 * i], lo[2 * i]);
        split_pack2(v.z, v.w, hi[2 * i + 1], lo[2 * i + 1]);
      }
      tc::tmem_st_32x32b_x8(lane_base + SM::TM_A_HI + ks * 8, hi);
      tc::tmem_st_32x32b_x8(lane_base + SM::TM_A_LO + ks * 8, lo);
    }
    tc::tmem_wait_st();
  }
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  cluster.sync();

  const uint32_t hb_addr = tc::smem_u32(hb);
  const size_t gstride = (size_t)4 * H;
  const int n_iter = n_sub * S;   // trace slot index = s * n_sub + sub
  // The loop bodies below are written per (cell step s, sub-tile `sub`) with `sub` a COMPILE-TIME index: the issue
  // slots of this kernel went to index arithmetic (k % n_sub, s / repeat, 64-bit row addresses), not to the LSTM math
  // (profiles/r01_summary.md), so everything that depends only on the sub-tile lives in registers and the global
  // pointers advance by a constant per step.
  const int rows_of[2] = {rows0, n_rows - rows0};
  const int rgv_of[2] = {(rows0 + 7) >> 3, (n_rows - rows0 + 7) >> 3};

  if (w_u == PP_CELL_WARPS) {
    // ================= MMA warp =================
    const uint32_t idesc = tc::make_idesc_bf16_f32(128, 16);
    const uint64_t db0 = tc::make_smem_desc(hb_addr, 128, SM::RG_BYTES);
    for (int s = 0; s < S; ++s) {
      const int cur = s & 1, nxt = cur ^ 1;
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        if (sub >= n_sub) break;
        if (s + 1 < S && tc::elect_one())
          tc::mbar_arrive_expect_tx(&h_full[sub * 2 + nxt], (uint32_t)(C * rgv_of[sub] * SM::SLICE));
        if (TRACE && lane == 0) p.trace[((size_t)blockIdx.x * n_iter + s * n_sub + sub) * 8 + 0] = gtime();
        if (s > 0 && !*dead) {
          if (!tc::mbar_wait(&h_full[sub * 2 + cur], ((s - 1) >> 1) & 1)) { *dead = 1; atomicExch(err, 5); }
        }
        __syncwarp();
        if (TRACE && lane == 0) p.trace[((size_t)blockIdx.x * n_iter + s * n_sub + sub) * 8 + 1] = gtime();
        tc::fence_after_thread_sync();
        if (tc::elect_one()) {
          const uint64_t db_cur = db0 + (uint64_t)(((sub * 2 + cur) * SM::BUF_BYTES) >> 4);
          const uint32_t d = tmem_base + sub * 64;
#pragma unroll
          for (int ks = 0; ks < KS; ++ks) {
            const uint32_t ta_hi = tmem_base + SM::TM_A_HI + ks * 8, ta_lo = tmem_base + SM::TM_A_LO + ks * 8;
            const uint64_t db_hi = db_cur + (uint64_t)(((ks >> 1) * SM::SLICE + (ks & 1) * 256) >> 4);
            const uint64_t db_lo = db_hi + (uint64_t)(512 >> 4);
            tc::mma_bf16_ts(d, ta_lo, db_hi, idesc, ks != 0);
            tc::mma_bf16_ts(d, ta_hi, db_lo, idesc, true);
            tc::mma_bf16_ts(d, ta_hi, db_hi, idesc, true);
          }
          tc::mma_commit(&mma_done[sub]);
        }
        __syncwarp();
        if (TRACE && lane == 0) p.trace[((size_t)blockIdx.x * n_iter + s * n_sub + sub) * 8 + 2] = gtime();
      }
    }
  } else {
    // ================= cell warps: warp w = row w of the current sub-tile, lane = hidden unit =================
    const int rg = w >> 3, r8 = w & 7;
    const bool on_of[2] = {w < rows_of[0], n_sub == 2 && w < rows_of[1]};
    // running pointers of this thread's (row, unit) in each sub-tile
    const float* gin_next[2];     // gin row of step s + 1
    float* gate_ptr[2];           // gates row of step s
    float* hs_ptr[2];             // hs / cs row s + 1 (cs at the same offset from p.cs)
    float* head_ptr[2];           // head_in row t
    float gnx[2][4];              // prefetched input projection of this sub-tile's next step
#pragma unroll
    for (int sub = 0; sub < 2; ++sub) {
      const size_t brow = (size_t)(b0 + (sub == 0 ? 0 : rows0) + w);
      gate_ptr[sub] = p.gates + brow * gstride + ug;
      hs_ptr[sub] = p.hs + ((size_t)B + brow) * H + ug;
      head_ptr[sub] = p.head_in ? p.head_in + brow * H + ug : nullptr;
      const float* g0 = p.gin + brow * gstride + ug;
#pragma unroll
      for (int q = 0; q < 4; ++q) gnx[sub][q] = on_of[sub] ? g0[q * H] : 0.f;
      // row of step 1: the same input row while s + 1 < repeat
      gin_next[sub] = (p.repeat > 1) ? g0 : g0 + (size_t)B * gstride;
    }
    const ptrdiff_t cs_off = p.cs - p.hs;
    const size_t gate_step = (size_t)B * gstride, h_step = (size_t)B * H;
    int rep = 0;                   // s % repeat
    for (int s = 0; s < S; ++s) {
      const int par = s & 1, nxt = par ^ 1;
      const bool last_rep = rep == p.repeat - 1;
      // after this step: rep' = (s + 1) % repeat; the input row of step s + 2 moves on when step s + 2 starts a new row
      const int rep1 = last_rep ? 0 : rep + 1;
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        if (sub >= n_sub) break;
        float gpre[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) gpre[q] = gnx[sub][q];
        if (s + 1 < S && on_of[sub]) {
#pragma unroll
          for (int q = 0; q < 4; ++q) gnx[sub][q] = gin_next[sub][q * H];
        }
        if (TRACE && tid == 0) p.trace[((size_t)blockIdx.x * n_iter + s * n_sub + sub) * 8 + 5] = gtime();
        if (!*dead) {
          if (!tc::mbar_wait(&mma_done[sub], par)) { *dead = 1; atomicExch(err, 6); }
        }
        if (TRACE && tid == 0) p.trace[((size_t)blockIdx.x * n_iter + s * n_sub + sub) * 8 + 3] = gtime();
        tc::fence_after_thread_sync();
        __syncwarp();
        float* gt = gt_all + (n_sub == 2 ? sub : par) * 16 * GT_LD;
        if ((w & 7) < 4) {    // the first 4 warps of each row group read that group's 8 accumulator columns (lane quarter
          const int q = w & 3, c0 = rg * 8;   // = warp % 4): the two row groups never wait for each other
          float v[8];
          tc::tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(sub * 64 + c0), v);
#pragma unroll
          for (int j = 0; j < 8; ++j) gt[(c0 + j) * GT_LD + q * 32 + lane] = v[j];
        }
        tc::fence_before_thread_sync();
        if (rg == 0) asm volatile("bar.sync 2, 256;" ::: "memory");
        else         asm volatile("bar.sync 3, 256;" ::: "memory");
        if (TRACE && tid == 0) p.trace[((size_t)blockIdx.x * n_iter + s * n_sub + sub) * 8 + 4] = gtime();

        if (rg < rgv_of[sub]) {
          unsigned char* hs_buf = hstage + ((sub * 2 + par) * 2 + rg) * SM::SLICE;
          __nv_bfloat16 hi = __float2bfloat16_rn(0.f), lo = hi;
          float ig = 0.f, fg = 0.f, gg = 0.f, og = 0.f, cn = 0.f, hn = 0.f;
          const bool on = on_of[sub];
          if (on) {
            const float* gr = gt + w * GT_LD + lane;
            ig = fast_sigmoid(gr[0] + gpre[0]);
            fg = fast_sigmoid(gr[32] + gpre[1]);
            gg = fast_tanh(gr[64] + gpre[2]);
            og = fast_sigmoid(gr[96] + gpre[3]);
            cn = fg * cst[sub] + ig * gg;
            hn = og * fast_tanh(cn);
            cst[sub] = cn;
            split_bf16(hn, hi, lo);
          }
          unsigned char* dst = hs_buf + (lane >> 3) * 128 + r8 * 16 + (lane & 7) * 2;
          *reinterpret_cast<__nv_bfloat16*>(dst) = hi;
          *reinterpret_cast<__nv_bfloat16*>(dst + 512) = lo;
          tc::fence_proxy_async_smem();
          if (rg == 0) asm volatile("bar.sync 2, 256;" ::: "memory");   // the 8 warps of this row group
          else         asm volatile("bar.sync 3, 256;" ::: "memory");
          if (s + 1 < S && r8 < C && tc::elect_one()) {
            const uint32_t d = r8;
            const uint32_t dst_local = hb_addr + (sub * 2 + nxt) * SM::BUF_BYTES + rg * SM::RG_BYTES + rank * SM::SLICE;
            tc::bulk_copy_to_cluster(tc::mapa(dst_local, d), tc::smem_u32(hs_buf), SM::SLICE,
                                     tc::mapa(tc::smem_u32(&h_full[sub * 2 + nxt]), d));
          }
          if (on) {   // the saved activations leave AFTER the exchange has been started: they are off the serial chain
            float* go = gate_ptr[sub];
            go[0] = ig; go[H] = fg; go[2 * H] = gg; go[3 * H] = og;
            hs_ptr[sub][0] = hn;
            hs_ptr[sub][cs_off] = cn;
            if (head_ptr[sub] && last_rep) head_ptr[sub][0] = fast_tanh(hn);
          }
        }
        gate_ptr[sub] += gate_step;
        hs_ptr[sub] += h_step;
        if (last_rep && head_ptr[sub]) head_ptr[sub] += h_step;
        // gin_next must point at the input row of step s + 2 = row (s + 2) / repeat
        if (p.repeat == 1 || rep1 == p.repeat - 1) gin_next[sub] += gate_step;
        if (TRACE && tid == 0) p.trace[((size_t)blockIdx.x * n_iter + s * n_sub + sub) * 8 + 7] = gtime();
      }
      rep = rep1;
    }
  }
  tc::fence_before_thread_sync();
  cluster.sync();
  if (w == 1) { __syncwarp(); tc::tmem_dealloc(tmem_base, SM::TM_COLS); }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
template <int H, int NB>
struct TcBwdSmem {
  static constexpr int C = H / 32;
  static constexpr int MT = (H + 127) / 128;                      // M tiles of 128 output units (rows >= H are zero)
  static constexpr int DG_PLANE = 16 * NB * 16;                   // [k-chunk][n][8 bf16]
  static constexpr int PS_SLOT = NB * 32 * 4;                     // fp32 [n][32 units] from one source CTA
  static constexpr int OFF_DG = 0;                                // [plane]
  // tensor memory: NACC independent accumulators per M tile, D_(mt,a) at [(mt*NACC + a)*NB, ..); W^T tiles from
  // column 256: (mt, plane) -> 256 + (2 mt + plane) * 64
  static constexpr int NACC = R2D2_SCAN_NACC;
  // H = 512 (BIG): four 128-unit tiles of W^T (hi + lo = 512 columns) do not leave room for the accumulators:
  // accumulators [0, 128), hi tiles [128, 384), lo tiles 0 and 1 [384, 512), lo tiles 2 and 3 in SHARED memory (SS-mode
  // MMAs); the partial-sum receive buffer and its staging copy are single-buffered (2 x 64 KB would not fit) behind a
  // "receive buffer consumed" handshake (ps_free) and cp.async.bulk.wait_group.read
  static constexpr bool BIG = H > 256;
  static constexpr int TM_A = BIG ? 128 : 256, TM_COLS = 512;
  static constexpr int MT_TM_LO = BIG ? 2 : MT;                   // M tiles whose lo plane is in tensor memory
  __host__ __device__ static constexpr int tm_hi(int mt) { return BIG ? TM_A + mt * 64 : TM_A + (2 * mt) * 64; }
  __host__ __device__ static constexpr int tm_lo(int mt) { return BIG ? TM_A + (MT + mt) * 64 : TM_A + (2 * mt + 1) * 64; }
  static_assert(MT * NACC * NB <= TM_A, "accumulators overlap the weight tiles in tensor memory");
  static constexpr int NBUF = BIG ? 1 : 2;
  static constexpr int OFF_PS = OFF_DG + 2 * DG_PLANE;            // [buf][src][n][32]
  static constexpr int OFF_PSTAGE = OFF_PS + NBUF * C * PS_SLOT;  // [dbuf][owner][n][32]
  static constexpr int OFF_BAR = OFF_PSTAGE + NBUF * C * PS_SLOT;
  static constexpr int OFF_GSTAGE = OFF_BAR + 128;                // [plane][k-chunk][n][8 bf16]: per-row dgin sums (repeat > 1)
  // lo planes of the W^T tiles that are not in tensor memory: per (tile, k-step) one 4 KB K-major block
  // [2 k-chunks][16 row groups][8 rows][16 B] (descriptor LBO = 2048, SBO = 128)
  static constexpr int OFF_WLO = OFF_GSTAGE + 2 * DG_PLANE;
  static constexpr int BYTES = OFF_WLO + (MT - MT_TM_LO) * 8 * 4096;
  static_assert(BYTES <= 232448, "backward scan tile does not fit in 227 KB of shared memory");
  static_assert(OFF_WLO % 128 == 0, "descriptor alignment");
};

#define BWD_STAMP(cond, slot) do { if (SM::BIG && p.trace && (cond)) p.trace[((size_t)blockIdx.x * S + it) * 8 + (slot)] = gtime(); } while (0)

template <int H, int NB>
__global__ void __launch_bounds__(TC_THREADS, 1) lstm_scan_bwd_tc_kernel(ScanBwdParams p, int* err) {
  using SM = TcBwdSmem<H, NB>;
  constexpr int C = SM::C, MT = SM::MT, RG = NB / 8, NT = RG / 2;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int b0 = p.row_begin + (blockIdx.x / C) * p.rows_per_cluster;  // this cluster's batch rows [b0, b_end), at most NB of them
  const int b_end = min(p.row_end > 0 ? p.row_end : p.B, b0 + p.rows_per_cluster);
  const int n_valid = b_end - b0;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int w_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int r8 = w & 7, half = w >> 3;                   // pointwise role: row r8 of row groups e = half, half+2, ...
  const int B = p.B, S = p.T * p.repeat;
  // H = 512, 32-row tiles: thread = (row tid / 16, the two ADJACENT units 2 (tid % 16), +1) instead of (two rows, one
  // unit): partial sums, saved activations and operand-tile writes become 8-byte / 4-byte accesses - half the memory
  // instructions of the cell phase (0.9 of the 3.9 us of a step, tools/trace_bwd.py)
  constexpr bool PAIR = SM::BIG && NB == 32;
  auto cell_row = [&](int j) { return PAIR ? (tid >> 4) : 8 * (half + 2 * j) + r8; };
  auto cell_unit = [&](int j) { return PAIR ? 2 * (tid & 15) + j : lane; };

  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* dgs = smem + SM::OFF_DG;
  float* ps = reinterpret_cast<float*>(smem + SM::OFF_PS);
  float* pstage = reinterpret_cast<float*>(smem + SM::OFF_PSTAGE);
  uint64_t* ps_full = reinterpret_cast<uint64_t*>(smem + SM::OFF_BAR);  // [2]
  uint64_t* mma_done = ps_full + 2;
  uint64_t* ps_free = mma_done + 1;                                     // BIG only: C arrivals per step
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ps_free + 1);
  volatile int* dead = reinterpret_cast<volatile int*>(tmem_slot + 1);
  uint64_t* mma_tile = ps_free + 2;                                     // BIG only: [MT] one completion barrier per M tile
  unsigned char* gst = smem + SM::OFF_GSTAGE;
  const int kt_k = 4 * H / 32;                                    // k tiles of the K-major image (gate columns / 32)
  const int kt_mn_dg = (S * B + 31) / 32, kt_mn_gin = (p.T * B + 31) / 32;

  if (tid == 0) {
    tc::mbar_init(&ps_full[0], 1);
    tc::mbar_init(&ps_full[1], 1);
    tc::mbar_init(mma_done, 1);
    tc::mbar_init(ps_free, C);
    for (int i = 0; i < 4; ++i) tc::mbar_init(&mma_tile[i], 1);
    tc::fence_mbar_init_cluster();
    *dead = 0;
  }
  if (w == 1) { __syncwarp(); tc::tmem_alloc(tmem_slot, SM::TM_COLS); }
  const int ug = rank * 32 + lane;
  const size_t gstride = (size_t)4 * H;
  float dcn[NT], keep[NT][4];
  float bsum[PAIR ? 2 : 1][4];            // this thread's share of the bias gradient: sum of dG over its rows and all steps (per unit)
#pragma unroll
  for (int j = 0; j < (PAIR ? 2 : 1); ++j)
#pragma unroll
    for (int q = 0; q < 4; ++q) bsum[j][q] = 0.f;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    dcn[j] = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) keep[j][q] = 0.f;
  }
  // rows of the operand tile that never carry a batch row stay zero for the whole launch
  for (int idx = tid; idx < 2 * SM::DG_PLANE / 16; idx += TC_THREADS) reinterpret_cast<uint4*>(dgs)[idx] = make_uint4(0, 0, 0, 0);
  tc::fence_proxy_async_smem();
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  // ---- A(j, r) = W_hh[grow(r)][j] -> TENSOR MEMORY: lane = output unit j within the 128-row tile mt, K index
  // r = local gate row (gate*32 + unit) packed two per column; rows j >= H are zero
  {
    const int q = w & 3;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    __syncwarp();
#pragma unroll 1
    for (int mt = 0; mt < MT; ++mt) {
      const int j = mt * 128 + q * 32 + lane;
#pragma unroll 1
      for (int ks = (w >> 2); ks < 8; ks += TC_WARPS / 4) {
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = ks * 16 + 2 * i;
          const size_t row0 = (size_t)((r >> 5) * H + rank * 32 + (r & 31));
          const float v0 = (j < H) ? __ldg(p.whh + row0 * H + j) : 0.f;
          const float v1 = (j < H) ? __ldg(p.whh + (row0 + 1) * H + j) : 0.f;
          split_pack2(v0, v1, hi[i], lo[i]);
        }
        tc::tmem_st_32x32b_x8(lane_base + SM::tm_hi(mt) + ks * 8, hi);
        if (mt < SM::MT_TM_LO) {
          tc::tmem_st_32x32b_x8(lane_base + SM::tm_lo(mt) + ks * 8, lo);
        } else {   // lo plane of this tile -> shared memory, K-major core matrices: row = output unit within the tile
          unsigned char* d = smem + SM::OFF_WLO + ((mt - SM::MT_TM_LO) * 8 + ks) * 4096 + (q * 4 + (lane >> 3)) * 128 + (lane & 7) * 16;
          *reinterpret_cast<uint4*>(d) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(d + 2048) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
        }
      }
    }
    tc::tmem_wait_st();
  }
  tc::fence_proxy_async_smem();
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  cluster.sync();

  const uint32_t idesc = tc::make_idesc_bf16_f32(128, NB);
  const uint64_t db_hi0 = tc::make_smem_desc(tc::smem_u32(dgs), NB * 16, 128);
  const uint64_t wlo_desc0 = tc::make_smem_desc(tc::smem_u32(smem + SM::OFF_WLO), 2048, 128);
  const uint32_t slot_bytes = (uint32_t)n_valid * 128u;            // only rows that exist travel: [n][32 units] fp32
  const uint32_t step_tx = (uint32_t)C * slot_bytes;

  // ---- per-thread constants and running pointers (index arithmetic, not LSTM math, dominated the issue slots of this
  // loop: no division, no 64-bit row address is recomputed per step)
  bool rowon[NT];
  const float* gates_nx[NT];    // gates row of the step that is prefetched next (s - 1)
  const float* cs_nx[NT];       // cs row s - 1
  const float* head_nx[NT];     // dh_head row consumed at step s - 1 (valid while hrow_nx >= 0)
  const size_t g_step = (size_t)B * gstride, h_step = (size_t)B * H;
  // head gradient bookkeeping for the step being prefetched: rel = s' - head_first_step, relm = rel % repeat,
  // consumed when rel >= 0 and relm == repeat - 1
  int rel_nx = (S - 1) - p.head_first_step;
  int relm_nx = rel_nx >= 0 ? rel_nx % p.repeat : 0;
  // first head row that will be consumed: the largest rel' <= rel with rel' % repeat == repeat - 1
  const int hrow0 = rel_nx >= 0 ? (rel_nx / p.repeat - (relm_nx == p.repeat - 1 ? 0 : 1)) : 0;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int b = b0 + cell_row(j);
    const int uj = rank * 32 + cell_unit(j);
    rowon[j] = b < b_end;
    const size_t bb = rowon[j] ? (size_t)b : (size_t)b0;
    gates_nx[j] = p.gates + ((size_t)(S - 1) * B + bb) * gstride + uj;
    cs_nx[j] = p.cs + ((size_t)(S - 1) * B + bb) * H + uj;
    head_nx[j] = (p.dh_head && hrow0 >= 0) ? p.dh_head + ((size_t)hrow0 * B + bb) * H + uj : nullptr;
  }
  float pg[NT][4], pc_prev[NT], pc_new[NT], phead[NT];   // saved activations of the step being processed
  auto fetch = [&](float (&g)[NT][4], float (&c)[NT], float (&hd)[NT], bool any) {
    const bool head_now = head_nx[0] != nullptr && rel_nx >= 0 && relm_nx == p.repeat - 1;
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      c[j] = hd[j] = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) g[j][q] = 0.f;
    }
    if constexpr (PAIR) {   // the two cells are adjacent units of one row: 8-byte loads
      if (any && rowon[0] && !(p.dbg & 2)) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 v = *reinterpret_cast<const float2*>(gates_nx[0] + q * H);   // plain load: dgates may alias gates
          g[0][q] = v.x; g[1][q] = v.y;
        }
        const float2 cv = __ldg(reinterpret_cast<const float2*>(cs_nx[0]));
        c[0] = cv.x; c[1] = cv.y;
        if (head_now) { const float2 hv = __ldg(reinterpret_cast<const float2*>(head_nx[0])); hd[0] = hv.x; hd[1] = hv.y; }
      }
    } else {
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        if (any && rowon[j] && !(p.dbg & 2)) {
#pragma unroll
          for (int q = 0; q < 4; ++q) g[j][q] = gates_nx[j][q * H];
          c[j] = __ldg(cs_nx[j]);
          if (head_now) hd[j] = __ldg(head_nx[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      gates_nx[j] -= g_step;
      cs_nx[j] -= h_step;
      if (head_now) head_nx[j] -= h_step;
    }
    // advance the bookkeeping to the next older step
    --rel_nx;
    relm_nx = relm_nx == 0 ? p.repeat - 1 : relm_nx - 1;
  };
#pragma unroll
  for (int j = 0; j < NT; ++j) pc_new[j] = rowon[j] ? __ldg(cs_nx[j] + h_step) : 0.f;   // cs[S]
  fetch(pg, pc_prev, phead, true);

  int rep = (S - 1) % p.repeat, t = (S - 1) / p.repeat;   // s % repeat and s / repeat, kept by counting
  for (int it = 0; it < S; ++it) {
    const int s = S - 1 - it;
    const int buf = it & 1;

    // software pipeline of the saved activations: the operands of THIS step were loaded one step ago (an HBM round
    // trip is ~half a cell step and used to sit on the serial chain); now fetch the ones of step s-1.
    // cs[s] is c_prev of this step and c_new of the next one, so only one new cell state per step.
    float ng[NT][4], nc[NT], nh[NT];
    fetch(ng, nc, nh, s > 0);   // (issuing these behind the proxy fence below instead was measured SLOWER: 11.7 -> 12.7 us per step)
    BWD_STAMP(tid == 0, 0);
    if (it > 0 && !*dead) {
      if (!tc::mbar_wait(&ps_full[buf], ((it - 1) >> 1) & 1)) { *dead = 1; atomicExch(err, 3); }
    }
    BWD_STAMP(tid == 0, 1);

    const bool emit_gin = p.repeat > 1 && rep == 0;
    // ---- pointwise backward of the cell (thread = (unit = lane, row r8 of row group e)); the dG values go to the MMA
    // operand tile first - their HBM copies are written below, after the tensor-core step has been started
    float dgr[NT][4];
    float dhs[NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) dhs[j] = phead[j];
    if (it > 0) {
      if constexpr (PAIR) {
        if (rowon[0]) {
          const float* psr = ps + (size_t)cell_row(0) * 32 + cell_unit(0);
#pragma unroll
          for (int src = 0; src < C; ++src) {
            const float2 v = *reinterpret_cast<const float2*>(psr + (size_t)src * NB * 32);
            dhs[0] += v.x; dhs[1] += v.y;
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          const int n = cell_row(j);
          if (rowon[j]) {
#pragma unroll
            for (int src = 0; src < C; ++src) dhs[j] += ps[(((SM::BIG ? 0 : buf) * C + src) * NB + n) * 32 + lane];
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) {
#pragma unroll
      for (int q = 0; q < 4; ++q) dgr[j][q] = 0.f;
      if (rowon[j]) {
        const float dh = dhs[j];
        const float ig = pg[j][0], fg = pg[j][1], gg = pg[j][2], og = pg[j][3];
        const float tcn = fast_tanh(pc_new[j]);
        const float dc = dcn[j] + dh * og * (1.f - tcn * tcn);
        dgr[j][3] = dh * tcn * og * (1.f - og);
        dgr[j][0] = dc * gg * ig * (1.f - ig);
        dgr[j][1] = dc * pc_prev[j] * fg * (1.f - fg);
        dgr[j][2] = dc * ig * (1.f - gg * gg);
        dcn[j] = dc * fg;
#pragma unroll
        for (int q = 0; q < 4; ++q) bsum[PAIR ? j : 0][q] += dgr[j][q];
        if (p.repeat > 1) {   // dgin row = sum of dG over the steps that share the input row
#pragma unroll
          for (int q = 0; q < 4; ++q) keep[j][q] += dgr[j][q];
        }
      }
    }
    // ---- operand tile of the MMA: K index r = gate*32 + unit -> chunk (gate*4 + unit/8), element unit%8; per-row dgin sums
    // (repeat > 1) go to their own tile and to HBM when the input row is complete
    if constexpr (PAIR) {
      if (rowon[0]) {
        const int n = cell_row(0), u0 = cell_unit(0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t hi, lo;
          split_pack2(dgr[0][q], dgr[1][q], hi, lo);
          const int off = ((q * 4 + (u0 >> 3)) * NB + n) * 16 + (u0 & 7) * 2;
          *reinterpret_cast<uint32_t*>(dgs + off) = hi;
          *reinterpret_cast<uint32_t*>(dgs + SM::DG_PLANE + off) = lo;
          if (emit_gin) {
            if (!p.skip_fp32)
              *reinterpret_cast<float2*>(p.dgin + ((size_t)t * B + b0 + n) * gstride + q * H + rank * 32 + u0) = make_float2(keep[0][q], keep[1][q]);
            split_pack2(keep[0][q], keep[1][q], hi, lo);
            *reinterpret_cast<uint32_t*>(gst + off) = hi;
            *reinterpret_cast<uint32_t*>(gst + SM::DG_PLANE + off) = lo;
            keep[0][q] = keep[1][q] = 0.f;
          }
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        const int n = cell_row(j), b = b0 + n;
        if (rowon[j]) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            __nv_bfloat16 hi, lo;
            split_bf16(dgr[j][q], hi, lo);
            const int off = ((q * 4 + (lane >> 3)) * NB + n) * 16 + (lane & 7) * 2;
            *reinterpret_cast<__nv_bfloat16*>(dgs + off) = hi;
            *reinterpret_cast<__nv_bfloat16*>(dgs + SM::DG_PLANE + off) = lo;
            if (emit_gin) {
              if (!p.skip_fp32) p.dgin[((size_t)t * B + b) * gstride + q * H + ug] = keep[j][q];
              split_bf16(keep[j][q], hi, lo);
              *reinterpret_cast<__nv_bfloat16*>(gst + off) = hi;
              *reinterpret_cast<__nv_bfloat16*>(gst + SM::DG_PLANE + off) = lo;
              keep[j][q] = 0.f;
            }
          }
        }
      }
    }
    auto store_dg = [&]() {
      if (!p.skip_fp32) {
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          if (rowon[j]) {
            float* go = p.dgates + ((size_t)s * B + b0 + cell_row(j)) * gstride + rank * 32 + cell_unit(j);
            go[0] = dgr[j][0]; go[H] = dgr[j][1]; go[2 * H] = dgr[j][2]; go[3 * H] = dgr[j][3];
          }
        }
      }
      // ---- packed operand images straight from the MMA operand tile in shared memory.  Eight lanes = the eight rows
      // of one core matrix (128 contiguous bytes in either image), four core matrices per warp instruction.
      if (p.img_k || p.img_mn_dg || p.img_mn_gin) {
        for (int idx = w * 4 + (lane >> 3); idx < RG * 16; idx += TC_WARPS * 4) {
          const int kc = idx & 15, n = (idx >> 4) * 8 + (lane & 7);
          if (n >= n_valid) continue;
          const int c8 = (kc >> 2) * (H / 8) + rank * 4 + (kc & 3);          // global gate column / 8
          const uint4 hi = *reinterpret_cast<const uint4*>(dgs + (kc * NB + n) * 16);
          const uint4 lo = *reinterpret_cast<const uint4*>(dgs + SM::DG_PLANE + (kc * NB + n) * 16);
          const size_t m = (size_t)s * B + b0 + n;
          if (p.img_mn_dg) {
            unsigned char* d = p.img_mn_dg + ((size_t)(c8 >> 4) * kt_mn_dg + (m >> 5)) * 16384 +
                               ((((m & 31) >> 3) * 128) + (c8 & 15) * 8 + (m & 7)) * 16;
            *reinterpret_cast<uint4*>(d) = hi;
            *reinterpret_cast<uint4*>(d + 8192) = lo;
          }
          if (p.img_k && p.repeat == 1) {
            unsigned char* d = p.img_k + ((size_t)(m >> 7) * kt_k + (c8 >> 2)) * 16384 +
                               ((((m & 127) >> 3) * 32) + (c8 & 3) * 8 + (m & 7)) * 16;
            *reinterpret_cast<uint4*>(d) = hi;
            *reinterpret_cast<uint4*>(d + 8192) = lo;
          }
          if (emit_gin) {
            const uint4 ghi = *reinterpret_cast<const uint4*>(gst + (kc * NB + n) * 16);
            const uint4 glo = *reinterpret_cast<const uint4*>(gst + SM::DG_PLANE + (kc * NB + n) * 16);
            const size_t mg = (size_t)t * B + b0 + n;
            if (p.img_mn_gin) {
              unsigned char* d = p.img_mn_gin + ((size_t)(c8 >> 4) * kt_mn_gin + (mg >> 5)) * 16384 +
                                 ((((mg & 31) >> 3) * 128) + (c8 & 15) * 8 + (mg & 7)) * 16;
              *reinterpret_cast<uint4*>(d) = ghi;
              *reinterpret_cast<uint4*>(d + 8192) = glo;
            }
            if (p.img_k) {
              unsigned char* d = p.img_k + ((size_t)(mg >> 7) * kt_k + (c8 >> 2)) * 16384 +
                                 ((((mg & 127) >> 3) * 32) + (c8 & 3) * 8 + (mg & 7)) * 16;
              *reinterpret_cast<uint4*>(d) = ghi;
              *reinterpret_cast<uint4*>(d + 8192) = glo;
            }
          }
        }
      }
    };
    BWD_STAMP(tid == 0, 2);
    tc::fence_proxy_async_smem();
    tc::fence_before_thread_sync();
    __syncthreads();
    BWD_STAMP(tid == 32, 3);   // warp 1: a dependent instruction follows (the barrier itself defers blocking)
    if (s == 0) { store_dg(); break; }  // dh_{-1} is not needed: the initial state is data, not a parameter
    if (SM::BIG && w_u == 1 && lane < C) {   // every thread of this CTA has consumed its receive buffer (phase `it`)
      tc::mbar_arrive_remote_relaxed(ps_free, (uint32_t)lane);   // relaxed: the release form is a MEMBAR.GPU behind this thread's dG stores
    }

    if (w_u == 0) {
      tc::fence_after_thread_sync();
      if (tc::elect_one()) {
      tc::mbar_arrive_expect_tx(&ps_full[buf ^ 1], step_tx);
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint32_t ta_hi = tmem_base + SM::tm_hi(mt) + ks * 8;
          const uint32_t ta_lo = tmem_base + SM::tm_lo(mt) + ks * 8;
          const uint64_t db_hi = db_hi0 + (uint64_t)((ks * 2 * NB * 16) >> 4);
          const uint64_t db_lo = db_hi + (uint64_t)(SM::DG_PLANE >> 4);
          const uint32_t d = tmem_base + (mt * SM::NACC + (ks % SM::NACC)) * NB;
          if (mt < SM::MT_TM_LO) tc::mma_bf16_ts(d, ta_lo, db_hi, idesc, ks >= SM::NACC);
          else tc::mma_bf16_ss(d, wlo_desc0 + (uint64_t)((((mt - SM::MT_TM_LO) * 8 + ks) * 4096) >> 4), db_hi, idesc, ks >= SM::NACC);
          tc::mma_bf16_ts(d, ta_hi, db_lo, idesc, true);
          tc::mma_bf16_ts(d, ta_hi, db_hi, idesc, true);
        }
        if (SM::BIG) tc::mma_commit(&mma_tile[mt]);   // the warps that own this tile's units start their exchange while the next tiles run
      }
      if (!SM::BIG) tc::mma_commit(mma_done);
      }
      __syncwarp();
      BWD_STAMP(tid == 0, 4);
    }
    if (!(p.dbg & 1)) store_dg();   // HBM copies of dG (and the per-row dgin sums) overlap with the tensor-core step
    if constexpr (SM::BIG) {
      // ---- warp w reads the accumulator of M tile w / 4, lane quarter w % 4: exactly the 32 units owned by CTA w of the
      // cluster.  It stages that owner's slice [n][32 units] alone and sends it: no block barrier between the tensor
      // core step and the exchange, and tile 0 is on its way while tiles 1..3 are still in the pipe.
      const int mt = w >> 2, q = w & 3;
      if (!*dead) {
        if (!tc::mbar_wait(&mma_tile[mt], it & 1)) { *dead = 1; atomicExch(err, 4); }
      }
      if (!*dead) {
        // single receive / staging buffers: phase `it` of ps_free completes when every CTA of the cluster has consumed
        // the sums of this step, i.e. (a) all my copies of the previous step have landed and (b) every receive buffer
        // may be overwritten by the copies issued below
        if (!tc::mbar_wait(ps_free, it & 1)) { *dead = 1; atomicExch(err, 7); }
      }
      tc::fence_after_thread_sync();
      __syncwarp();
      BWD_STAMP(tid == 15 * 32, 5);
      float* pst_w = pstage + (size_t)w * NB * 32;
#pragma unroll
      for (int cb = 0; cb < RG; ++cb) {
        float v[8];
        tc::tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mt * NB + cb * 8), v);
#pragma unroll
        for (int i = 0; i < 8; ++i) pst_w[(cb * 8 + i) * 32 + lane] = v[i];
      }
      tc::fence_before_thread_sync();
      tc::fence_proxy_async_smem();
      __syncwarp();
      if (tc::elect_one()) {
        const uint32_t d = w_u;
        const uint32_t src = tc::smem_u32(pst_w);
        const uint32_t dst_local = tc::smem_u32(ps + (size_t)rank * NB * 32);
        if (p.xchg) {
          // through L2 (profiles/r02_xchg_bench.txt): store my partials for owner d, wait for the writes, then a bulk
          // load "multicast" to that single CTA: it lands at the same CTA-relative offset in d and completes d's mbarrier
          unsigned char* g = p.xchg + ((((size_t)(blockIdx.x / C) * 2 + (it & 1)) * C + rank) * C + d) * (size_t)(NB * 128);
          BWD_STAMP(w_u == 15, 6);
          tc::bulk_store_s2g(g, src, slot_bytes);
          tc::bulk_commit_wait_all();
          tc::bulk_copy_g2s_multicast(dst_local, g, slot_bytes, tc::smem_u32(&ps_full[buf ^ 1]), (uint16_t)(1u << d));
          BWD_STAMP(w_u == 15, 7);
        } else {
          tc::bulk_copy_to_cluster(tc::mapa(dst_local, d), src, slot_bytes, tc::mapa(tc::smem_u32(&ps_full[buf ^ 1]), d));
        }
      }
      __syncwarp();
    } else {
    if (!*dead) {
      if (!tc::mbar_wait(mma_done, it & 1)) { *dead = 1; atomicExch(err, 4); }
    }
    if (SM::BIG && !*dead) {
      // single receive / staging buffers: phase `it` of ps_free completes when every CTA of the cluster has consumed
      // the sums of this step, i.e. (a) all my copies of the previous step have landed - the staging buffer may be
      // overwritten - and (b) every receive buffer may be overwritten by the copies issued below
      if (!tc::mbar_wait(ps_free, it & 1)) { *dead = 1; atomicExch(err, 7); }
    }
    tc::fence_after_thread_sync();
    __syncwarp();

    // ---- partial sums -> staging [owner CTA][n][32 units]; lane = output unit j within the 128-row tile
    float* pst = pstage + (size_t)(SM::BIG ? 0 : (it & 1)) * C * NB * 32;
    {
      const int q = w & 3;
      for (int idx = (w >> 2); idx < MT * RG; idx += TC_WARPS / 4) {
        const int mt = idx / RG, c0 = (idx % RG) * 8;
        const int j = mt * 128 + q * 32 + lane;
        float v[8];
        tc::tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mt * SM::NACC * NB + c0), v);
#pragma unroll
        for (int a = 1; a < SM::NACC; ++a) {
          float u[8];
          tc::tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((mt * SM::NACC + a) * NB + c0), u);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] += u[i];
        }
        if (j < H) {
#pragma unroll
          for (int i = 0; i < 8; ++i) pst[(((j >> 5) * NB) + c0 + i) * 32 + (j & 31)] = v[i];
        }
      }
    }
    tc::fence_before_thread_sync();
    tc::fence_proxy_async_smem();
    __syncthreads();
    if (w_u < C && tc::elect_one()) {  // reduce-scatter: my partials for owner w's units -> its slot [buf^1][my rank]
      const uint32_t d = w_u;
      const uint32_t src = tc::smem_u32(pst + (size_t)d * NB * 32);
      const uint32_t dst_local = tc::smem_u32(ps + ((size_t)((SM::BIG ? 0 : (buf ^ 1)) * C + rank) * NB) * 32);
      if (SM::BIG && p.xchg) {
        // through L2 (profiles/r02_xchg_bench.txt): store my partials for owner d, wait for the writes, then a bulk load
        // "multicast" to that single CTA: it lands at the same CTA-relative offset in d and completes d's mbarrier
        unsigned char* g = p.xchg + ((((size_t)(blockIdx.x / C) * 2 + (it & 1)) * C + rank) * C + d) * (size_t)(NB * 128);
        tc::bulk_store_s2g(g, src, slot_bytes);
        tc::bulk_commit_wait_all();
        tc::bulk_copy_g2s_multicast(dst_local, g, slot_bytes, tc::smem_u32(&ps_full[buf ^ 1]), (uint16_t)(1u << d));
      } else {
        tc::bulk_copy_to_cluster(tc::mapa(dst_local, d), src, slot_bytes, tc::mapa(tc::smem_u32(&ps_full[buf ^ 1]), d));
      }
    }
    }   // !BIG
#pragma unroll
    for (int j = 0; j < NT; ++j) {   // rotate the pipeline registers
#pragma unroll
      for (int q = 0; q < 4; ++q) pg[j][q] = ng[j][q];
      pc_new[j] = pc_prev[j];
      pc_prev[j] = nc[j];
      phead[j] = nh[j];
    }
    if (rep == 0) { rep = p.repeat - 1; --t; } else --rep;
  }
  tc::fence_before_thread_sync();
  cluster.sync();
  if (p.dbias) {   // CTA-level reduction over the 16 warps (same lane -> unit map), then one atomic per (gate, unit)
    float* red = ps;       // [warp | row][4][32] <= 16 KB over ps; all exchange traffic is complete after the cluster barrier
    constexpr int RED_N = PAIR ? 32 : TC_WARPS;   // partial sums per (gate, unit): one per row (PAIR) or per warp
    if constexpr (PAIR) {
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) red[((tid >> 4) * 4 + q) * 32 + cell_unit(j)] = bsum[j][q];
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) red[(w * 4 + q) * 32 + lane] = bsum[0][q];
    }
    __syncthreads();
    if (tid < 128) {
      const int q = tid >> 5;
      float t = 0.f;
#pragma unroll
      for (int ww = 0; ww < RED_N; ++ww) t += red[(ww * 4 + q) * 32 + lane];
      atomicAdd(p.dbias + q * H + ug, t);
      if (p.dbias2) atomicAdd(p.dbias2 + q * H + ug, t);
    }
  }
  if (w == 1) { __syncwarp(); tc::tmem_dealloc(tmem_base, SM::TM_COLS); }
}

// ------------------------------------------------------------------------------------------------
// forward, H = 512: cluster of 16 CTAs, up to 80 batch rows per cluster as two ping-pong sub-tiles of <= 40 rows.
//
// What differs from the kernels above (measured reasons in profiles/r02_*):
//  * only 7 clusters of 16 are resident on a B200 (GPC geometry), so 512 rows are spread as 7 x 74 in ONE wave;
//  * the h_t all-gather goes THROUGH L2: the CTA's slice of a row group (1 KB: 32 units x 8 rows x hi/lo) is bulk-stored
//    to a global scratch line and re-loaded by one MULTICAST bulk copy that lands in all 16 CTAs and completes
//    transaction bytes on each CTA's mbarrier (12 -> ~95 B/clk/SM against shared->remote-shared copies);
//  * the h operand of a sub-tile (40 rows x 512 x hi/lo = 80 KB) is single-buffered: a source may overwrite it only
//    after every CTA of the cluster has retired the MMAs that read it (buf_free: 16 remote arrivals per step);
//  * gate rows are PERMUTED in tensor memory (lane = 4 * unit + gate inside a lane quarter), so the four gates of a
//    cell sit in four adjacent lanes of one warp: the accumulator readback is transposed with eight warp shuffles -
//    no shared-memory tile, no block barrier between readback and cell math;
//  * dedicated exchange warps (one per row group) own the store -> wait -> multicast-load chain; cell warps only
//    arrive on a named barrier; a dedicated warp issues the MMAs (96 per sub-tile step: K = 512, three passes, the
//    last 12 k-steps of the W_hh lo plane come from shared memory).
// ------------------------------------------------------------------------------------------------
constexpr int BIG_CELL_WARPS = 20, BIG_THREADS = (BIG_CELL_WARPS + 1) * 32;   // 672: 5 row groups x 4 lane quarters + MMA warp

struct BigFwdSmem {
  static constexpr int H = 512, C = 16, KC = H / 8, KS = H / 16;
  static constexpr int SLICE = 1024, RG_BYTES = C * SLICE;
  static constexpr int MAX_RG = 5, MAX_ROWS = 8 * MAX_RG;          // per sub-tile
  static constexpr int SUB_BYTES = MAX_RG * RG_BYTES;              // 80 KB
  static constexpr int NCOL = 48;                                  // accumulator columns per sub-tile (N <= 48)
  static constexpr int TM_A_HI = 2 * NCOL, TM_A_LO = TM_A_HI + H / 2, TM_COLS = 512;
  static constexpr int KS_TM_LO = (TM_COLS - TM_A_LO) / 8, KS_TAIL = KS - KS_TM_LO;   // 20 / 12
  static constexpr int OFF_HB = 0;                                 // [sub][row group][slice][plane][4 chunks][8][16 B]
  static constexpr int OFF_WTAIL = OFF_HB + 2 * SUB_BYTES;         // [k-step][2 k-chunks][16 row groups][8][16 B]
  static constexpr int OFF_HSTAGE = OFF_WTAIL + KS_TAIL * 4096;    // [sub][row group][SLICE]
  static constexpr int OFF_BAR = OFF_HSTAGE + 2 * MAX_RG * SLICE;  // h_full[2], mma_done[2], buf_free[2], tmem slot, dead
  static constexpr int BYTES = OFF_BAR + 128;
  static constexpr int XCHG_PER_CLUSTER = 2 * 2 * C * MAX_RG * SLICE;   // [step parity][sub][rank][row group][1 KB]
  static_assert(BYTES <= 232448, "H = 512 forward scan does not fit in shared memory");
};

#define BIG_STAMP(cond, slot) do { if (TRACE && (cond)) p.trace[(((size_t)blockIdx.x * S + s) * 2 + sub) * 8 + (slot)] = gtime(); } while (0)

// two activations with ONE reciprocal: 1/(1+ea) and 1/(1+eb) from rcp((1+ea)(1+eb)); the MUFU pipe (one warp
// instruction per 8 clocks and scheduler) and the issue slots bound the cell phase of this kernel, not the FP32 math.
// x <= 0 arguments are clamped at -30 / scale so that the product of two denominators stays finite.
__device__ __forceinline__ void sigmoid_pair(float xa, float xb, float neg_scale_log2e, float& sa, float& sb) {
  const float ea = tc::ex2_approx(fminf(xa * neg_scale_log2e, 43.f)), eb = tc::ex2_approx(fminf(xb * neg_scale_log2e, 43.f));
  const float da = 1.f + ea, db = 1.f + eb;
  const float r = tc::rcp_approx(da * db);
  sa = r * db;
  sb = r * da;
}

template <bool TRACE>
__global__ void __launch_bounds__(BIG_THREADS, 1) lstm_scan_fwd_big_kernel(ScanFwdParams p, int* err) {
  using SM = BigFwdSmem;
  constexpr int H = SM::H, C = SM::C, KC = SM::KC, KS = SM::KS;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int cl = blockIdx.x / C;
  const int b0 = cl * p.rows_per_cluster;
  const int b_end = min(p.B, b0 + p.rows_per_cluster);
  const int n_rows = b_end - b0;                                   // 1..80
  const int n_sub = n_rows > 8 ? 2 : 1;
  const int rows0 = n_sub == 2 ? (n_rows + 1) / 2 : n_rows;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int w_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int B = p.B, S = p.T * p.repeat;

  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* hb = smem + SM::OFF_HB;
  unsigned char* hstage = smem + SM::OFF_HSTAGE;
  uint64_t* h_full = reinterpret_cast<uint64_t*>(smem + SM::OFF_BAR);   // [sub]
  uint64_t* mma_done = h_full + 2;                                      // [sub]
  uint64_t* buf_free = mma_done + 2;                                    // [sub]: C arrivals per step
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(buf_free + 2);
  volatile int* dead = reinterpret_cast<volatile int*>(tmem_slot + 1);

  const int rows_of[2] = {rows0, n_rows - rows0};
  const int row0_of[2] = {0, rows0};
  const int rgv_of[2] = {(rows0 + 7) >> 3, (n_rows - rows0 + 7) >> 3};

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&h_full[i], 1); tc::mbar_init(&mma_done[i], 1); tc::mbar_init(&buf_free[i], C); }
    tc::fence_mbar_init_cluster();
    *dead = 0;
  }
  if (w == 1) { __syncwarp(); tc::tmem_alloc(tmem_slot, SM::TM_COLS); }
  // ---- initial h tiles (all 512 units of my cluster's rows; zeros where no row exists) -> operand buffers
  for (int idx = tid; idx < 2 * SM::MAX_ROWS * KC; idx += BIG_THREADS) {
    const int sub = idx / (SM::MAX_ROWS * KC), rem = idx % (SM::MAX_ROWS * KC);
    const int n = rem % SM::MAX_ROWS, kc = rem / SM::MAX_ROWS;
    float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
    if (sub < n_sub && n < rows_of[sub] && p.h0) {
      const float* src = p.h0 + (size_t)(b0 + row0_of[sub] + n) * H + kc * 8;
      v0 = __ldg(reinterpret_cast<const float4*>(src));
      v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
    }
    unsigned char* dst = hb + sub * SM::SUB_BYTES + (n >> 3) * SM::RG_BYTES + (kc >> 2) * SM::SLICE + (kc & 3) * 128 + (n & 7) * 16;
    split8_store(v0, v1, dst, dst + 512);
  }
  tc::fence_proxy_async_smem();
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  // ---- W_hh slice -> tensor memory.  Lane L of quarter k = L / 32: unit = 8 k + (L % 32) / 4, gate = L % 4.
  if (w < BIG_CELL_WARPS) {
    const int k = w & 3;
    const int unit = k * 8 + (lane >> 2), gate = lane & 3;
    const float* wrow = p.whh + (size_t)(gate * H + rank * 32 + unit) * H;
    const uint32_t lane_base = tmem_base + ((uint32_t)(k * 32) << 16);
    __syncwarp();
#pragma unroll 1
    for (int ks = (w >> 2); ks < KS; ks += BIG_CELL_WARPS / 4) {
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(wrow + ks * 16 + i * 4));
        split_pack2(v.x, v.y, hi[2 * i], lo[2 * i]);
        split_pack2(v.z, v.w, hi[2 * i + 1], lo[2 * i + 1]);
      }
      tc::tmem_st_32x32b_x8(lane_base + SM::TM_A_HI + ks * 8, hi);
      if (ks < SM::KS_TM_LO) {
        tc::tmem_st_32x32b_x8(lane_base + SM::TM_A_LO + ks * 8, lo);
      } else {
        unsigned char* d = smem + SM::OFF_WTAIL + (ks - SM::KS_TM_LO) * 4096 + (k * 4 + (lane >> 3)) * 128 + (lane & 7) * 16;
        *reinterpret_cast<uint4*>(d) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        *reinterpret_cast<uint4*>(d + 2048) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
      }
    }
    tc::tmem_wait_st();
  }
  tc::fence_proxy_async_smem();
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  cluster.sync();

  const uint32_t hb_addr = tc::smem_u32(hb);
  const size_t gstride = (size_t)4 * H;

  if (w_u == BIG_CELL_WARPS) {
    // ================= MMA warp =================
    const uint64_t db0 = tc::make_smem_desc(hb_addr, 128, SM::RG_BYTES);
    const uint64_t wtail_desc0 = tc::make_smem_desc(tc::smem_u32(smem + SM::OFF_WTAIL), 2048, 128);
    for (int s = 0; s < S; ++s) {
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        if (sub >= n_sub) break;
        BIG_STAMP(lane == 0, 0);
        if (s > 0 && !*dead) {
          if (!tc::mbar_wait(&h_full[sub], (s - 1) & 1)) { *dead = 1; atomicExch(err, 8); }
        }
        __syncwarp();
        BIG_STAMP(lane == 0, 1);
        tc::fence_after_thread_sync();
        if (tc::elect_one()) {
          if (s + 1 < S) tc::mbar_arrive_expect_tx(&h_full[sub], (uint32_t)(C * rgv_of[sub] * SM::SLICE));   // h_s of all 16 CTAs
          const uint32_t idesc = tc::make_idesc_bf16_f32(128, 16 * ((rows_of[sub] + 15) >> 4));
          const uint64_t db_sub = db0 + (uint64_t)((sub * SM::SUB_BYTES) >> 4);
          const uint32_t d = tmem_base + sub * SM::NCOL;
#pragma unroll
          for (int ks = 0; ks < KS; ++ks) {
            const uint32_t ta_hi = tmem_base + SM::TM_A_HI + ks * 8, ta_lo = tmem_base + SM::TM_A_LO + ks * 8;
            const uint64_t db_hi = db_sub + (uint64_t)(((ks >> 1) * SM::SLICE + (ks & 1) * 256) >> 4);
            const uint64_t db_lo = db_hi + (uint64_t)(512 >> 4);
            if (ks < SM::KS_TM_LO) tc::mma_bf16_ts(d, ta_lo, db_hi, idesc, ks != 0);
            else tc::mma_bf16_ss(d, wtail_desc0 + (uint64_t)(((ks - SM::KS_TM_LO) * 4096) >> 4), db_hi, idesc, true);
            tc::mma_bf16_ts(d, ta_hi, db_lo, idesc, true);
            tc::mma_bf16_ts(d, ta_hi, db_hi, idesc, true);
          }
          tc::mma_commit(&mma_done[sub]);
        }
        __syncwarp();
        BIG_STAMP(lane == 0, 2);
      }
    }
  } else {
    // ================= cell warps: row group j = w / 4, lane quarter k = w % 4 (units 8k..8k+7 of this CTA) ============
    // lane = 4 * unit + gate: the thread activates ITS gate for the 8 rows of the group, then the four lanes of a unit
    // swap 2-row blocks (8 shuffles) and each finishes the cells of rows 2 pq, 2 pq + 1
    const int k = w & 3, j = w >> 2;
    const int u8 = lane >> 2, pq = lane & 3;
    const int ug = rank * 32 + k * 8 + u8;          // global hidden unit
    const bool hiq = (pq & 2) != 0, odd = (pq & 1) != 0;
    const float sc = pq == 2 ? 2.f : 1.f;           // gate 2 is tanh(x) = 2 sigmoid(2x) - 1
    const float nsl = -1.4426950408889634f * sc, off = 1.f - sc;
    unsigned char* xbase = p.xchg + (size_t)cl * SM::XCHG_PER_CLUSTER;
    float cst[2][2];
    bool act_of[2];
    const float* gin_ptr[2];      // gin of (row j*8 + 0, gate pq, unit) at input row t
    float* gate_ptr[2];           // gates of the same element at step s
    float* hs_ptr[2];             // hs of (row j*8 + 2 pq, unit) at slot s + 1
    float* head_ptr[2];
#pragma unroll
    for (int sub = 0; sub < 2; ++sub) {
      act_of[sub] = sub < n_sub && j < rgv_of[sub];
      const size_t brow = (size_t)(b0 + row0_of[sub] + j * 8);
      gin_ptr[sub] = p.gin + brow * gstride + pq * H + ug;
      gate_ptr[sub] = p.gates + brow * gstride + pq * H + ug;
      hs_ptr[sub] = p.hs + ((size_t)B + brow + 2 * pq) * H + ug;
      head_ptr[sub] = p.head_in ? p.head_in + (brow + 2 * pq) * H + ug : nullptr;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int n = j * 8 + 2 * pq + i;
        cst[sub][i] = 0.f;
        if (act_of[sub] && n < rows_of[sub]) {
          const size_t b = (size_t)(b0 + row0_of[sub] + n);
          const float hv = p.h0 ? __ldg(p.h0 + b * H + ug) : 0.f;
          const float cv = p.c0 ? __ldg(p.c0 + b * H + ug) : 0.f;
          p.hs[b * H + ug] = hv;
          p.cs[b * H + ug] = cv;
          cst[sub][i] = cv;
        }
      }
    }
    const ptrdiff_t cs_off = p.cs - p.hs;
    const size_t gate_step = (size_t)B * gstride, h_step = (size_t)B * H;
    int rep = 0;
    for (int s = 0; s < S; ++s) {
      const bool last_rep = rep == p.repeat - 1;
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        if (!act_of[sub]) continue;
        const int nrow = rows_of[sub] - j * 8;      // rows of this group that exist (>= 1)
        // input projection of this gate for the 8 rows: issued before the wait, the MMAs take longer than the loads
        float x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = (i < nrow && !(TRACE && (p.dbg & 2))) ? gin_ptr[sub][(size_t)i * gstride] : 0.f;   // plain loads: gates may alias gin
        if (!*dead) {
          if (!tc::mbar_wait(&mma_done[sub], s & 1)) { *dead = 1; atomicExch(err, 10); }
        }
        BIG_STAMP(tid == 0, 3);
        if (w_u == 0 && lane < C) tc::mbar_arrive_remote_relaxed(&buf_free[sub], (uint32_t)lane);   // this CTA's MMAs of (s, sub) have retired
        tc::fence_after_thread_sync();
        __syncwarp();
        {
          float v[8];
          tc::tmem_ld_32x32b_x8(tmem_base + ((uint32_t)(k * 32) << 16) + (uint32_t)(sub * SM::NCOL + j * 8), v);
#pragma unroll
          for (int i = 0; i < 8; ++i) x[i] += v[i];
        }
#pragma unroll
        for (int i = 0; i < 8; i += 2) {
          float sa, sb;
          sigmoid_pair(x[i], x[i + 1], nsl, sa, sb);
          x[i] = fmaf(sc, sa, off);
          x[i + 1] = fmaf(sc, sb, off);
        }
        // 4 x 4 transpose of 2-row blocks among the four lanes of a unit: lane pq ends up with all gates of rows 2pq, 2pq+1
        float kk[4], rc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float snd = hiq ? x[i] : x[4 + i];
          kk[i] = hiq ? x[4 + i] : x[i];
          rc[i] = __shfl_xor_sync(0xffffffffu, snd, 2);            // gate pq^2, rows 4*(pq>>1) + i
        }
        float cn[2], hn[2];
        unsigned char* hs_buf = hstage + (sub * SM::MAX_RG + j) * SM::SLICE;
        float a0[2], a1[2], a2[2], a3[2];                          // gates pq, pq^2, pq^1, pq^3 of rows 2pq + i
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const float s1 = odd ? kk[i] : kk[2 + i];
          const float s2 = odd ? rc[i] : rc[2 + i];
          a0[i] = odd ? kk[2 + i] : kk[i];
          a1[i] = odd ? rc[2 + i] : rc[i];
          a2[i] = __shfl_xor_sync(0xffffffffu, s1, 1);
          a3[i] = __shfl_xor_sync(0xffffffffu, s2, 1);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          // lane 0: [i g f o], 1: [f o i g], 2: [g i o f], 3: [o f g i]  ->  i*g = u*v, (f, o) = (xx, yy) swapped on lanes 2, 3
          const float u = odd ? a2[i] : a0[i], vv = odd ? a3[i] : a1[i];
          const float xx = odd ? a0[i] : a2[i], yy = odd ? a1[i] : a3[i];
          const float fg = hiq ? yy : xx, og = hiq ? xx : yy;
          cn[i] = fmaf(fg, cst[sub][i], u * vv);
          cst[sub][i] = cn[i];
          hn[i] = og;
        }
        {
          float ta, tb;                                            // tanh(c) = 2 sigmoid(2c) - 1
          sigmoid_pair(cn[0], cn[1], -2.8853900817779268f, ta, tb);
          hn[0] *= fmaf(2.f, ta, -1.f);
          hn[1] *= fmaf(2.f, tb, -1.f);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          __nv_bfloat16 hi = __float2bfloat16_rn(0.f), lo = hi;
          if (2 * pq + i < nrow) split_bf16(hn[i], hi, lo);
          unsigned char* dst = hs_buf + k * 128 + (2 * pq + i) * 16 + u8 * 2;   // [plane][chunk = k][row][unit % 8]
          *reinterpret_cast<__nv_bfloat16*>(dst) = hi;
          *reinterpret_cast<__nv_bfloat16*>(dst + 512) = lo;
        }
        BIG_STAMP(tid == 0, 4);
        if (s + 1 < S) {
          tc::fence_proxy_async_smem();
          const int bar_id = 1 + sub * SM::MAX_RG + j;
          if (k == 0) {   // this warp hands the row group's slice to the cluster: store -> L2 -> multicast load into all 16 CTAs
            asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
            if (tc::elect_one()) {
              unsigned char* g = xbase + ((size_t)(((s & 1) * 2 + sub) * C + rank) * SM::MAX_RG + j) * SM::SLICE;
              tc::bulk_store_s2g(g, tc::smem_u32(hs_buf), SM::SLICE);
              tc::bulk_commit_wait_all();
              BIG_STAMP(j == 0, 6);
              if (!*dead) {   // every CTA of the cluster has retired the MMAs of step s that read this sub-tile's operand buffer
                if (!tc::mbar_wait(&buf_free[sub], s & 1)) { *dead = 1; atomicExch(err, 9); }
              }
              tc::bulk_copy_g2s_multicast(hb_addr + sub * SM::SUB_BYTES + j * SM::RG_BYTES + rank * SM::SLICE, g, SM::SLICE,
                                          tc::smem_u32(&h_full[sub]), (uint16_t)0xFFFF);
              BIG_STAMP(j == 0, 7);
            }
            __syncwarp();
          } else {
            asm volatile("bar.arrive %0, 128;" ::"r"(bar_id) : "memory");
          }
        }
        // ---- saved activations: off the serial chain
        if (!(TRACE && (p.dbg & 1))) {
          if (!p.no_save) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (i < nrow) gate_ptr[sub][(size_t)i * gstride] = x[i];
          }
#pragma unroll
          for (int i = 0; i < 2; ++i)
            if (2 * pq + i < nrow) {
              float* ho = hs_ptr[sub] + (size_t)i * H;
              ho[0] = hn[i];
              if (!p.no_save) ho[cs_off] = cn[i];
              if (head_ptr[sub] && last_rep) head_ptr[sub][(size_t)i * H] = fast_tanh(hn[i]);
            }
        }
        gate_ptr[sub] += gate_step;
        hs_ptr[sub] += h_step;
        if (last_rep) {
          gin_ptr[sub] += gate_step;
          if (head_ptr[sub]) head_ptr[sub] += h_step;
        }
      }
      rep = last_rep ? 0 : rep + 1;
    }
  }
  tc::fence_before_thread_sync();
  cluster.sync();
  if (w == 1) { __syncwarp(); tc::tmem_dealloc(tmem_base, SM::TM_COLS); }
}

bool scan_pingpong_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("R2D2_SCAN_PINGPONG"); v = (e && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

template <typename Kern, typename Params>
int launch_cluster_tc(Kern kern, const Params& p, int cluster_size, int n_clusters, int smem_bytes, cudaStream_t stream,
                      int threads = TC_THREADS) {
  R2D2_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  if (cluster_size > 8) R2D2_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cluster_size * n_clusters);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster_size;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int* err = scan_error_flag();
  R2D2_REQUIRE(err != nullptr, "scan error flag allocation failed");
  R2D2_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, p, err));
  count_launch();
  return R2D2_OK;
}

// how many clusters of this kernel the device can keep resident at once (GPC geometry decides, not just SM count)
template <typename Kern>
int max_active_clusters(Kern kern, int cluster_size, int smem_bytes, int threads = TC_THREADS) {
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  if (cluster_size > 8) cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cluster_size * 64);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster_size;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return -1; }
  return n;
}

// Tiling of the batch over clusters.  The chain is a serial dependency, so every cluster must be RESIDENT at once
// (a cluster that waits for a free GPC slot doubles the chain's latency): ask the driver how many clusters of this
// kernel fit (15 clusters of 8 on a B200, not 148/8 = 18: clusters cannot straddle GPCs) and, when 16-row tiles
// would need more than that, spread the rows evenly over the resident clusters with the 32-column MMA tile.
struct Tiling { int nb, rows_per_cluster, n_clusters; };

template <int H, typename K16, typename K32>
Tiling pick_tiling(int B, K16 k16, int smem16, K32 k32, int smem32) {
  static int max16 = -2, max32 = -2;
  if (max16 == -2) max16 = max_active_clusters(k16, H / 32, smem16);
  if (max32 == -2) max32 = max_active_clusters(k32, H / 32, smem32);
  const int fit16 = max16 > 0 ? max16 : 148 / (H / 32), fit32 = max32 > 0 ? max32 : 148 / (H / 32);
  if (ceil_div(B, 16) <= fit16) return {16, 16, ceil_div(B, 16)};
  int n = fit32;
  if (ceil_div(B, n) > 32) n = ceil_div(B, 32);  // more rows than one wave can hold: full 32-row tiles, several waves
  const int rows = ceil_div(B, n);
  return {32, rows, ceil_div(B, rows)};
}

// the H = 512 kernels exchange through L2 (env R2D2_SCAN_L2XCHG=0: shared->remote-shared copies, the A/B fallback)
bool scan_l2_exchange_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("R2D2_SCAN_L2XCHG"); v = (e && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

int fwd_big(const ScanFwdParams& p_in, cudaStream_t stream, bool* handled) {
  *handled = false;
  if (!scan_l2_exchange_enabled()) return R2D2_OK;
  static int fit = -2;
  if (fit == -2) fit = max_active_clusters(lstm_scan_fwd_big_kernel<false>, 16, BigFwdSmem::BYTES, BIG_THREADS);
  const int resident = fit > 0 ? fit : 7;
  const int max_rows = 2 * BigFwdSmem::MAX_ROWS;
  int rows = ceil_div(p_in.B, resident);
  if (rows > max_rows) rows = ceil_div(p_in.B, ceil_div(p_in.B, max_rows));   // several waves of full clusters
  const int n_clusters = ceil_div(p_in.B, rows);
  size_t cap = 0;
  unsigned char* scratch = scan_xchg_scratch(&cap);
  if (!scratch || (size_t)n_clusters * BigFwdSmem::XCHG_PER_CLUSTER > cap) return R2D2_OK;
  ScanFwdParams p = p_in;
  p.rows_per_cluster = rows;
  p.xchg = scratch;
  if (const char* e = getenv("R2D2_SCAN_DBG")) p.dbg = atoi(e);
  *handled = true;
  return p.trace ? launch_cluster_tc(lstm_scan_fwd_big_kernel<true>, p, 16, n_clusters, BigFwdSmem::BYTES, stream, BIG_THREADS)
                 : launch_cluster_tc(lstm_scan_fwd_big_kernel<false>, p, 16, n_clusters, BigFwdSmem::BYTES, stream, BIG_THREADS);
}

template <int H>
int fwd_tc(const ScanFwdParams& p_in, cudaStream_t stream) {
  if constexpr (H == 512) {
    bool handled = false;
    R2D2_TRY(fwd_big(p_in, stream, &handled));
    if (handled) return R2D2_OK;
  }
  ScanFwdParams p = p_in;
  const Tiling t = pick_tiling<H>(p.B, lstm_scan_fwd_tc_kernel<H, 16>, TcFwdSmem<H, 16>::BYTES,
                                  lstm_scan_fwd_tc_kernel<H, 32>, TcFwdSmem<H, 32>::BYTES);
  p.rows_per_cluster = t.rows_per_cluster;
  if (t.nb == 16)
    return launch_cluster_tc(lstm_scan_fwd_tc_kernel<H, 16>, p, H / 32, t.n_clusters, TcFwdSmem<H, 16>::BYTES, stream);
  if constexpr (H <= 256) {
    if (scan_pingpong_enabled())
      return p.trace ? launch_cluster_tc(lstm_scan_fwd_pp_kernel<H, true>, p, H / 32, t.n_clusters, PpFwdSmem<H>::BYTES, stream, PP_THREADS)
                     : launch_cluster_tc(lstm_scan_fwd_pp_kernel<H, false>, p, H / 32, t.n_clusters, PpFwdSmem<H>::BYTES, stream, PP_THREADS);
  }
  return launch_cluster_tc(lstm_scan_fwd_tc_kernel<H, 32>, p, H / 32, t.n_clusters, TcFwdSmem<H, 32>::BYTES, stream);
}
template <int H>
int bwd_tc(const ScanBwdParams& p_in, cudaStream_t stream) {
  ScanBwdParams p = p_in;
  R2D2_REQUIRE(!p.skip_fp32 || (p.img_k && (p.repeat == 1 || p.img_mn_gin || !p.img_mn_dg)), "skip_fp32 without operand images");
  {  // rows of the last tile that no batch row maps to must read as zeros in the GEMMs
    const size_t rows_g = (size_t)p.T * p.B, rows_d = (size_t)p.T * p.repeat * p.B;
    const size_t mn_tiles = 4 * H / 128 > 0 ? 4 * H / 128 : 1;
    if (p.img_k && rows_g % 128 != 0)
      R2D2_CUDA_TRY(cudaMemsetAsync(p.img_k + (rows_g / 128) * (size_t)(4 * H / 32) * 16384, 0, (size_t)(4 * H / 32) * 16384, stream));
    if (p.img_mn_dg && rows_d % 32 != 0) {
      const size_t kt = (rows_d + 31) / 32;
      R2D2_CUDA_TRY(cudaMemset2DAsync(p.img_mn_dg + (kt - 1) * 16384, kt * 16384, 0, 16384, mn_tiles, stream));
    }
    if (p.img_mn_gin && p.img_mn_gin != p.img_mn_dg && rows_g % 32 != 0) {
      const size_t kt = (rows_g + 31) / 32;
      R2D2_CUDA_TRY(cudaMemset2DAsync(p.img_mn_gin + (kt - 1) * 16384, kt * 16384, 0, 16384, mn_tiles, stream));
    }
  }
  const Tiling t = pick_tiling<H>(p.B, lstm_scan_bwd_tc_kernel<H, 16>, TcBwdSmem<H, 16>::BYTES,
                                  lstm_scan_bwd_tc_kernel<H, 32>, TcBwdSmem<H, 32>::BYTES);
  p.rows_per_cluster = t.rows_per_cluster;
  if (const char* e = getenv("R2D2_SCAN_DBG")) p.dbg = atoi(e);
  if constexpr (H == 512) {
    size_t cap = 0;
    unsigned char* scratch = scan_l2_exchange_enabled() ? scan_xchg_scratch(&cap) : nullptr;
    if (scratch && (size_t)t.n_clusters * 2 * 16 * 16 * (size_t)(t.nb * 128) <= cap) p.xchg = scratch;
  }
  if (t.nb == 16)
    return launch_cluster_tc(lstm_scan_bwd_tc_kernel<H, 16>, p, H / 32, t.n_clusters, TcBwdSmem<H, 16>::BYTES, stream);
  if constexpr (H == 512) {
    // Waves: only `fit` (7) clusters of 16 are resident and a wave of 32-row clusters costs the same ~3.9 us per step
    // whether 7 or 2 clusters run in it.  512 rows as 16 clusters = waves of 7 + 7 + 2; instead the full waves run as
    // 32-row clusters and the remainder as 16-row clusters (shorter MMA and cell phases) in ONE extra wave of a second launch.
    static int fit32 = -2;
    if (fit32 == -2) fit32 = max_active_clusters(lstm_scan_bwd_tc_kernel<H, 32>, H / 32, TcBwdSmem<H, 32>::BYTES);
    const int fit = fit32 > 0 ? fit32 : 7;
    const int full = (t.n_clusters / fit) * fit;                  // clusters of 32 rows in full waves
    const int rest_rows = p.B - full * 32;
    if (t.rows_per_cluster == 32 && full > 0 && rest_rows > 0 && ceil_div(rest_rows, 16) <= fit) {
      ScanBwdParams a = p, b = p;
      a.row_begin = 0; a.row_end = full * 32;
      b.row_begin = full * 32; b.row_end = p.B; b.rows_per_cluster = 16;
      R2D2_TRY(launch_cluster_tc(lstm_scan_bwd_tc_kernel<H, 32>, a, H / 32, full, TcBwdSmem<H, 32>::BYTES, stream));
      return launch_cluster_tc(lstm_scan_bwd_tc_kernel<H, 16>, b, H / 32, ceil_div(rest_rows, 16), TcBwdSmem<H, 16>::BYTES, stream);
    }
  }
  return launch_cluster_tc(lstm_scan_bwd_tc_kernel<H, 32>, p, H / 32, t.n_clusters, TcBwdSmem<H, 32>::BYTES, stream);
}

}  // namespace

int* scan_error_flag() {   // one flag per device (a process may drive several GPUs through separate handles)
  static std::mutex mu;
  static std::map<int, int*> flags;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  auto it = flags.find(dev);
  if (it != flags.end()) return it->second;
  int* flag = nullptr;
  if (cudaMalloc(&flag, sizeof(int)) != cudaSuccess) return nullptr;
  cudaMemset(flag, 0, sizeof(int));
  flags[dev] = flag;
  return flag;
}

// One scratch block per device: the scans of a device are stream-ordered behind each other (one learner stream); the
// exchange lines are double-buffered by step parity inside a launch and every launch rewrites what it reads.
unsigned char* scan_xchg_scratch(size_t* bytes) {
  static std::mutex mu;
  static std::map<int, unsigned char*> bufs;
  constexpr size_t BYTES = (size_t)80 << 20;
  if (bytes) *bytes = BYTES;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  auto it = bufs.find(dev);
  if (it != bufs.end()) return it->second;
  unsigned char* b = nullptr;
  if (cudaMalloc(&b, BYTES) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  cudaMemset(b, 0, BYTES);
  bufs[dev] = b;
  return b;
}

int lstm_scan_error_status(int* out, cudaStream_t stream) {
  int* flag = scan_error_flag();
  R2D2_REQUIRE(flag && out, "flag");
  R2D2_CUDA_TRY(cudaMemcpyAsync(out, flag, sizeof(int), cudaMemcpyDeviceToHost, stream));
  R2D2_CUDA_TRY(cudaStreamSynchronize(stream));
  return R2D2_OK;
}

// the same queries pick_tiling, bwd_tc and fwd_big make, so that tests can predict the tiling of a batch size
template <int H>
int max_active_clusters_tc(int nb, int backward) {
  if (nb == 16) return backward ? max_active_clusters(lstm_scan_bwd_tc_kernel<H, 16>, H / 32, TcBwdSmem<H, 16>::BYTES)
                                : max_active_clusters(lstm_scan_fwd_tc_kernel<H, 16>, H / 32, TcFwdSmem<H, 16>::BYTES);
  if (nb == 32) return backward ? max_active_clusters(lstm_scan_bwd_tc_kernel<H, 32>, H / 32, TcBwdSmem<H, 32>::BYTES)
                                : max_active_clusters(lstm_scan_fwd_tc_kernel<H, 32>, H / 32, TcFwdSmem<H, 32>::BYTES);
  return -1;
}

int lstm_scan_max_active_clusters(int H, int nb, int backward) {
  if (H == 512 && nb == 80 && !backward)
    return max_active_clusters(lstm_scan_fwd_big_kernel<false>, 16, BigFwdSmem::BYTES, BIG_THREADS);
  switch (H) {
    case 32: return max_active_clusters_tc<32>(nb, backward);
    case 64: return max_active_clusters_tc<64>(nb, backward);
    case 128: return max_active_clusters_tc<128>(nb, backward);
    case 256: return max_active_clusters_tc<256>(nb, backward);
    case 512: return max_active_clusters_tc<512>(nb, backward);
    default: return -1;
  }
}

int lstm_scan_forward_tc(const ScanFwdParams& p, cudaStream_t stream) {
  switch (p.H) {
    case 32: return fwd_tc<32>(p, stream);
    case 64: return fwd_tc<64>(p, stream);
    case 128: return fwd_tc<128>(p, stream);
    case 256: return fwd_tc<256>(p, stream);
    case 512: return fwd_tc<512>(p, stream);
    default: break;
  }
  set_last_error("tcgen05 scan: unsupported hidden size");
  return R2D2_ERR_UNSUPPORTED;
}

int lstm_scan_backward_tc(const ScanBwdParams& p, cudaStream_t stream) {
  switch (p.H) {
    case 32: return bwd_tc<32>(p, stream);
    case 64: return bwd_tc<64>(p, stream);
    case 128: return bwd_tc<128>(p, stream);
    case 256: return bwd_tc<256>(p, stream);
    case 512: return bwd_tc<512>(p, stream);
    default: break;
  }
  set_last_error("tcgen05 scan: unsupported hidden size");
  return R2D2_ERR_UNSUPPORTED;
}

}  // namespace r2d2
