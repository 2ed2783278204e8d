// One acting step of the four nets over B environments (actor.py:136-148 of the reference, batched):
//
//   actor:          z = tanh(W1 x + b1);        (h,c) <- LSTMCell(z, (h,c));  mu   = tanh(W3 tanh(h) + b3)
//   target_actor:   the same with its own weights                             mu_t
//   critic:         z = tanh(W1 [x; mu] + b1);  (h,c) <- LSTMCell(z, (h,c))   (head output discarded, actor.py:143)
//   target_critic:  z = tanh(W1 [x; mu_t] + b1);(h,c) <- LSTMCell(z, (h,c))   (actor.py:144)
//
// Four stream-ordered launches, no host synchronisation:
//   1. act_l1_kernel      l1 of the two actors -> z; obs half of the two critics' l1 -> pre; all four h_in rows.
//                         z and h_in leave as the bf16 hi/lo K-major operand image of [z | h] (gemm_tc.cu format).
//   2. act_gate_kernel    gates = [z | h] [W_ih | W_hh]^T + (b_ih + b_hh) on tcgen05 (bf16x3) with the LSTM cell in
//                         the epilogue, for actor and target actor as one grid.
//   3. act_bridge_kernel  mu and mu_t (row-local heads), then the action half of the critics' l1 and its tanh -> image.
//   4. act_gate_kernel    the same for critic and target critic.
//
// The gate product is swapped for small batches: the weights are the M = 128 operand (32 hidden units x 4 gates per
// tile, rows permuted so that TMEM lane = 4 * unit + gate, as in lstm_scan_fwd_big_kernel), the batch is N (<= 128
// per MMA, two B tiles per CTA).  The weight images are packed once per r2d2_act_load (H^2 * 32 bytes per net,
// 8 MB at H = 512) and stay L2-resident across steps.  Only the live batch rows of an activation tile are copied
// (the K-major image keeps rows 0..n-1 of a plane in its first n * 64 bytes).  The cell update is CTA-local: the
// four gates of a unit sit in four adjacent lanes of one warp, so no gates tensor is written.
#include <stdlib.h>

#include "act.cuh"
#include "tc05.cuh"

namespace r2d2 {

struct Act {
  int O = 0, A = 0, H = 0, max_batch = 0;
  int KT = 0, MT = 0, NT = 0;          // k tiles (32) of K = 2H, m tiles (128 permuted gate rows) per net, n tiles (128)
  bool loaded = false;
  unsigned char* w_img = nullptr;      // [4 nets][MT][KT][16 KB]   [W_ih | W_hh], gate rows permuted
  unsigned char* x_img = nullptr;      // [4 nets][NT][KT][16 KB]   [z | h_in] of the current step
  float* w1t = nullptr;                // [4][O][H]   l1 weight, observation columns, transposed
  float* w1a = nullptr;                // [2][A][H]   critics' l1 weight, action columns, transposed
  float* b1 = nullptr;                 // [4][H]
  float* bg = nullptr;                 // [4][4H]     b_ih + b_hh
  float* w3 = nullptr;                 // [2][A][H]   actor heads
  float* b3 = nullptr;                 // [2][A]
  float* pre = nullptr;                // [2][max_batch][H] obs half of the critics' l1 pre-activation (+ b1)
  int* err = nullptr;                  // != 0: a bounded mbarrier wait expired
};

namespace {

constexpr int TBK = 32;
constexpr int PLANE_BYTES = 128 * TBK * 2;     // one bf16 plane of a 128 x 32 operand tile
constexpr int TILE_BYTES = 2 * PLANE_BYTES;    // hi + lo plane
constexpr int GATE_THREADS = 320;              // warp 0 producer, warp 1 MMA, warps 2..9 cell epilogue
constexpr int GATE_STAGES = 4;
constexpr int GATE_STAGE_BYTES = 3 * TILE_BYTES;   // weight tile + two batch tiles
constexpr int GATE_OFF_BARS = GATE_STAGES * GATE_STAGE_BYTES;
constexpr int GATE_SMEM = GATE_OFF_BARS + 128;
constexpr int GATE_TM_COLS = 256;

// byte offset of the 16-byte group (row, k..k+7) inside a K-major image [row tiles][k_tiles][16 KB] (k % 8 == 0)
__host__ __device__ __forceinline__ size_t img_offset(int row, int k, int k_tiles) {
  return ((size_t)(row >> 7) * k_tiles + (k >> 5)) * TILE_BYTES +
         (size_t)((((row & 127) >> 3) * 32) + ((k & 31) >> 3) * 8 + (row & 7)) * 16;
}

__device__ __forceinline__ void img_store8(unsigned char* img, int row, int k, int k_tiles, const float (&v)[8]) {
  uint4 h, l;
  split_pack2(v[0], v[1], h.x, l.x);
  split_pack2(v[2], v[3], h.y, l.y);
  split_pack2(v[4], v[5], h.z, l.z);
  split_pack2(v[6], v[7], h.w, l.w);
  unsigned char* d = img + img_offset(row, k, k_tiles);
  *reinterpret_cast<uint4*>(d) = h;
  *reinterpret_cast<uint4*>(d + PLANE_BYTES) = l;
}

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.f / (1.f + __expf(-x)); }

struct NetPtrs { const float* p[4]; };

// flat parameter block offsets (include/r2d2_b200.h): l1.weight[H,I], l1.bias[H], w_ih[4H,H], w_hh[4H,H], b_ih[4H],
// b_hh[4H], l3.weight[A,H], l3.bias[A]
__host__ __device__ __forceinline__ size_t off_b1(int H, int I) { return (size_t)H * I; }
__host__ __device__ __forceinline__ size_t off_wih(int H, int I) { return (size_t)H * I + H; }
__host__ __device__ __forceinline__ size_t off_whh(int H, int I) { return off_wih(H, I) + (size_t)4 * H * H; }
__host__ __device__ __forceinline__ size_t off_bih(int H, int I) { return off_whh(H, I) + (size_t)4 * H * H; }
__host__ __device__ __forceinline__ size_t off_w3(int H, int I) { return off_bih(H, I) + (size_t)8 * H; }

// [W_ih | W_hh] of net blockIdx.z -> tile (blockIdx.y, blockIdx.x) of its image; image row r of m tile mt is gate
// r % 4 of hidden unit 32 mt + r / 4
__global__ void __launch_bounds__(256) act_pack_w_kernel(NetPtrs nets, int O, int A, int H, int MT, int KT,
                                                         unsigned char* __restrict__ w_img) {
  const int e = blockIdx.z, mt = blockIdx.y, kt = blockIdx.x;
  const int I = O + (e >= 2 ? A : 0);
  const float* wih = nets.p[e] + off_wih(H, I);
  const float* whh = nets.p[e] + off_whh(H, I);
  unsigned char* img = w_img + (size_t)e * MT * KT * TILE_BYTES;
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const int id = threadIdx.x + g * 256;
    const int r = 8 * (id >> 5) + (id & 7), k = kt * TBK + 8 * ((id >> 3) & 3);
    const int src_row = (r & 3) * H + mt * 32 + (r >> 2);
    const float* src = k < H ? wih + (size_t)src_row * H + k : whh + (size_t)src_row * H + (k - H);
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __ldg(src + i);      // H % 32 == 0: a group never straddles W_ih / W_hh
    img_store8(img, mt * 128 + r, k, KT, v);
  }
}

// the small per-net tensors in the layouts the step kernels read
__global__ void act_prep_kernel(NetPtrs nets, int O, int A, int H, float* __restrict__ w1t, float* __restrict__ w1a,
                                float* __restrict__ b1, float* __restrict__ bg, float* __restrict__ w3,
                                float* __restrict__ b3) {
  const int e = blockIdx.y;
  const int I = O + (e >= 2 ? A : 0);
  const float* p = nets.p[e];
  const long long n_w1 = (long long)H * I, n_bg = 4LL * H, n_w3 = (e < 2) ? (long long)A * H : 0;
  const long long total = n_w1 + H + n_bg + n_w3 + (e < 2 ? A : 0);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long j = i;
    if (j < n_w1) {                       // l1.weight[k][c] -> w1t[e][c][k] or w1a[e-2][c-O][k]
      const int k = (int)(j / I), c = (int)(j % I);
      const float v = p[j];
      if (c < O) w1t[((size_t)e * O + c) * H + k] = v;
      else w1a[((size_t)(e - 2) * A + (c - O)) * H + k] = v;
      continue;
    }
    j -= n_w1;
    if (j < H) { b1[(size_t)e * H + j] = p[off_b1(H, I) + j]; continue; }
    j -= H;
    if (j < n_bg) { bg[(size_t)e * 4 * H + j] = p[off_bih(H, I) + j] + p[off_bih(H, I) + 4 * H + j]; continue; }
    j -= n_bg;
    if (j < n_w3) { w3[(size_t)e * A * H + j] = p[off_w3(H, I) + j]; continue; }
    j -= n_w3;
    b3[(size_t)e * A + j] = p[off_w3(H, I) + (size_t)A * H + j];
  }
}

// launch 1: 32 rows x 32 outputs of net blockIdx.z per CTA; thread = (row, 8 consecutive outputs)
__global__ void __launch_bounds__(128) act_l1_kernel(const float* __restrict__ x, const float* __restrict__ state_in,
                                                     const float* __restrict__ w1t, const float* __restrict__ b1,
                                                     unsigned char* __restrict__ x_img, float* __restrict__ pre,
                                                     int B, int O, int H, int NT, int KT) {
  const int e = blockIdx.z;
  const int n = blockIdx.y * 32 + (threadIdx.x >> 2);
  const int k0 = blockIdx.x * 32 + (threadIdx.x & 3) * 8;
  if (n >= B) return;
  const float* w = w1t + (size_t)e * O * H + k0;
  float acc[8];
  {
    const float4 a = __ldg(reinterpret_cast<const float4*>(b1 + (size_t)e * H + k0));
    const float4 b = __ldg(reinterpret_cast<const float4*>(b1 + (size_t)e * H + k0 + 4));
    acc[0] = a.x; acc[1] = a.y; acc[2] = a.z; acc[3] = a.w; acc[4] = b.x; acc[5] = b.y; acc[6] = b.z; acc[7] = b.w;
  }
  const float* xr = x + (size_t)n * O;
#pragma unroll 4
  for (int o = 0; o < O; ++o) {
    const float xv = __ldg(xr + o);
    const float4 a = __ldg(reinterpret_cast<const float4*>(w + (size_t)o * H));
    const float4 b = __ldg(reinterpret_cast<const float4*>(w + (size_t)o * H + 4));
    acc[0] = fmaf(xv, a.x, acc[0]); acc[1] = fmaf(xv, a.y, acc[1]); acc[2] = fmaf(xv, a.z, acc[2]); acc[3] = fmaf(xv, a.w, acc[3]);
    acc[4] = fmaf(xv, b.x, acc[4]); acc[5] = fmaf(xv, b.y, acc[5]); acc[6] = fmaf(xv, b.z, acc[6]); acc[7] = fmaf(xv, b.w, acc[7]);
  }
  unsigned char* img = x_img + (size_t)e * NT * KT * TILE_BYTES;
  if (e < 2) {
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = tanhf(acc[i]);
    img_store8(img, n, k0, KT, acc);
  } else {
    float* d = pre + ((size_t)(e - 2) * B + n) * H + k0;
    *reinterpret_cast<float4*>(d) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    *reinterpret_cast<float4*>(d + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
  const float* h = state_in + ((size_t)(e * 2) * B + n) * H + k0;   // h_in of net e, [4,2,B,H]
  const float4 a = __ldg(reinterpret_cast<const float4*>(h)), b = __ldg(reinterpret_cast<const float4*>(h + 4));
  const float hv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  img_store8(img, n, H + k0, KT, hv);
}

struct GateParams {
  const unsigned char* w_img;   // first net of the pair: [2][MT][KT][16 KB]
  const unsigned char* x_img;   // [2][NT][KT][16 KB]
  const float* bg;              // [2][4H]
  const float* state_in;        // [4,2,B,H]
  float* state_out;
  int e0;                       // state index of the first net of the pair (0: actors, 2: critics)
  int B, H, MT, NT, KT;
  int* err;
};

__global__ void __launch_bounds__(GATE_THREADS, 1) act_gate_kernel(GateParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + GATE_OFF_BARS);   // [stage] bytes landed
  uint64_t* empty = full + GATE_STAGES;                                 // [stage] MMAs retired
  uint64_t* accum_full = empty + GATE_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_full + 1);
  volatile int* dead = reinterpret_cast<volatile int*>(tmem_slot + 1);

  const int tid = threadIdx.x, lane = tid & 31;
  const int w_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int n_blk = blockIdx.x, mt = blockIdx.y, net = blockIdx.z;
  const int n0 = n_blk * 256, KT = p.KT, H = p.H, B = p.B;
  int n_eff[2], nb_live = 0;                // rows of each batch tile rounded up to the MMA granule of 16
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int e = min(128, B - n0 - j * 128);
    n_eff[j] = e > 0 ? ((e + 15) & ~15) : 0;
    if (e > 0) nb_live = j + 1;
  }

  if (tid == 0) {
    for (int s = 0; s < GATE_STAGES; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
    tc::mbar_init(accum_full, 1);
    tc::fence_mbar_init_cluster();
    *dead = 0;
  }
  if (w_u == 1) { __syncwarp(); tc::tmem_alloc(tmem_slot, GATE_TM_COLS); }
  tc::fence_before_thread_sync();
  __syncthreads();
  tc::fence_after_thread_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (w_u == 0) {
    // ================= producer: the weight tile and the live rows of the batch tiles, per k tile =================
    if (tc::elect_one()) {
      const unsigned char* a_src = p.w_img + ((size_t)net * p.MT + mt) * KT * TILE_BYTES;
      const unsigned char* b_src = p.x_img + ((size_t)net * p.NT + n_blk * 2) * KT * TILE_BYTES;
      const uint32_t smem_base = tc::smem_u32(smem);
      uint32_t tx = TILE_BYTES;
#pragma unroll
      for (int j = 0; j < 2; ++j) tx += 2u * (uint32_t)n_eff[j] * 64u;
      for (int i = 0; i < KT; ++i) {
        const int s = i % GATE_STAGES;
        if (!*dead && !tc::mbar_wait(&empty[s], ((i / GATE_STAGES) & 1) ^ 1)) { *dead = 1; atomicExch(p.err, 1); }
        const uint32_t bar = tc::smem_u32(&full[s]);
        tc::mbar_arrive_expect_tx(&full[s], tx);
        tc::bulk_copy_g2s(smem_base + s * GATE_STAGE_BYTES, a_src + (size_t)i * TILE_BYTES, TILE_BYTES, bar);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (j >= nb_live) continue;
          const unsigned char* src = b_src + ((size_t)j * KT + i) * TILE_BYTES;
          const uint32_t dst = smem_base + s * GATE_STAGE_BYTES + (1 + j) * TILE_BYTES;
          const uint32_t bytes = (uint32_t)n_eff[j] * 64u;   // rows 0..n_eff-1 of a K-major plane
          tc::bulk_copy_g2s(dst, src, bytes, bar);
          tc::bulk_copy_g2s(dst + PLANE_BYTES, src + PLANE_BYTES, bytes, bar);
        }
      }
    }
    __syncwarp();
  } else if (w_u == 1) {
    // ================= MMA issuer: D[128 gate rows, batch] += W . X^T, three bf16 passes =================
    const uint64_t d0 = tc::make_smem_desc(tc::smem_u32(smem), 128, 512);
    for (int i = 0; i < KT; ++i) {
      const int s = i % GATE_STAGES;
      if (!*dead && !tc::mbar_wait(&full[s], (i / GATE_STAGES) & 1)) { *dead = 1; atomicExch(p.err, 2); }
      __syncwarp();
      tc::fence_after_thread_sync();
      if (tc::elect_one()) {
        const uint64_t dsa = d0 + (uint64_t)((s * GATE_STAGE_BYTES) >> 4);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (j >= nb_live) continue;
          const uint32_t idesc = tc::make_idesc_bf16_f32(128, n_eff[j]);
          const uint64_t dsb = d0 + (uint64_t)((s * GATE_STAGE_BYTES + (1 + j) * TILE_BYTES) >> 4);
          const uint32_t d = tmem_base + j * 128;
#pragma unroll
          for (int ks = 0; ks < TBK / 16; ++ks) {
            const uint64_t a_hi = dsa + (uint64_t)((ks * 256) >> 4), a_lo = a_hi + (uint64_t)(PLANE_BYTES >> 4);
            const uint64_t b_hi = dsb + (uint64_t)((ks * 256) >> 4), b_lo = b_hi + (uint64_t)(PLANE_BYTES >> 4);
            tc::mma_bf16_ss(d, a_lo, b_hi, idesc, (i | ks) != 0);
            tc::mma_bf16_ss(d, a_hi, b_lo, idesc, true);
            tc::mma_bf16_ss(d, a_hi, b_hi, idesc, true);
          }
        }
        tc::mma_commit(&empty[s]);
        if (i + 1 == KT) tc::mma_commit(accum_full);
      }
      __syncwarp();
    }
  } else {
    // ================= cell epilogue: warp -> lane quarter q (8 units x 4 gates), batch tile `half` ==============
    if (!*dead && !tc::mbar_wait(accum_full, 0)) { *dead = 1; atomicExch(p.err, 3); }
    __syncwarp();
    tc::fence_after_thread_sync();
    const int q = w_u & 3, half = (w_u - 2) >> 2;
    if (half < nb_live) {
      const int gate = lane & 3, unit = mt * 32 + q * 8 + (lane >> 2);
      const int grp = lane & ~3;
      const int e = p.e0 + net;
      const float bias = __ldg(p.bg + (size_t)net * 4 * H + gate * H + unit);
      const float* c_in = p.state_in + ((size_t)(e * 2 + 1) * B) * H + unit;
      float* h_out = p.state_out + ((size_t)(e * 2) * B) * H + unit;
      float* c_out = p.state_out + ((size_t)(e * 2 + 1) * B) * H + unit;
      const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 128);
      const int col0 = n0 + half * 128, n_cols = half == 0 ? n_eff[0] : n_eff[1];
      for (int c0 = 0; c0 < n_cols; c0 += 8) {
        float v[8];
        tc::tmem_ld_32x32b_x8(lane_base + (uint32_t)c0, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float x = v[j] + bias;
          v[j] = gate == 2 ? tanhf(x) : sigmoid_acc(x);
        }
        // the four lanes of a unit swap gates; lane `gate` finishes the cells of columns 2 gate, 2 gate + 1
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float gi = __shfl_sync(0xffffffffu, v[j], grp | 0);
          const float gf = __shfl_sync(0xffffffffu, v[j], grp | 1);
          const float gg = __shfl_sync(0xffffffffu, v[j], grp | 2);
          const float go = __shfl_sync(0xffffffffu, v[j], grp | 3);
          const int col = col0 + c0 + j;
          if ((j >> 1) == gate && col < B) {
            const float cn = fmaf(gf, __ldg(c_in + (size_t)col * H), gi * gg);
            c_out[(size_t)col * H] = cn;
            h_out[(size_t)col * H] = go * tanhf(cn);
          }
        }
      }
    }
    tc::fence_before_thread_sync();
  }
  __syncthreads();
  if (w_u == 1) { __syncwarp(); tc::tmem_dealloc(tmem_base, GATE_TM_COLS); }
}

// launch 3: one CTA per (row, actor net): mu = tanh(W3 tanh(h') + b3), then the critic's l1 on [x; mu] -> image
__global__ void __launch_bounds__(128) act_bridge_kernel(const float* __restrict__ state_out, const float* __restrict__ w3,
                                                         const float* __restrict__ b3, const float* __restrict__ w1a,
                                                         const float* __restrict__ pre, unsigned char* __restrict__ x_img,
                                                         float* __restrict__ mu, int B, int A, int H, int NT, int KT) {
  __shared__ float th[512];
  __shared__ float mu_s[32];
  const int n = blockIdx.x, e = blockIdx.y, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const float* h = state_out + ((size_t)(e * 2) * B + n) * H;
  for (int k = tid; k < H; k += 128) th[k] = tanhf(h[k]);
  __syncthreads();
  for (int a = w; a < A; a += 4) {
    const float* wr = w3 + ((size_t)e * A + a) * H;
    float s = 0.f;
    for (int k = lane; k < H; k += 32) s = fmaf(__ldg(wr + k), th[k], s);
    s = warp_sum(s);
    if (lane == 0) {
      const float m = tanhf(s + __ldg(b3 + (size_t)e * A + a));
      mu_s[a] = m;
      if (e == 0) mu[(size_t)n * A + a] = m;
    }
  }
  __syncthreads();
  unsigned char* img = x_img + (size_t)(2 + e) * NT * KT * TILE_BYTES;
  for (int k0 = tid * 8; k0 < H; k0 += 128 * 8) {
    float acc[8];
    const float* pr = pre + ((size_t)e * B + n) * H + k0;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = pr[i];
    for (int a = 0; a < A; ++a) {
      const float m = mu_s[a];
      const float* wr = w1a + ((size_t)e * A + a) * H + k0;
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = fmaf(__ldg(wr + i), m, acc[i]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = tanhf(acc[i]);
    img_store8(img, n, k0, KT, acc);
  }
}

int unsupported(const std::string& msg) {
  set_last_error("unsupported: " + msg);
  return R2D2_ERR_UNSUPPORTED;
}

}  // namespace

int act_create(Act** out, int obs, int act, int hidden, int max_batch) {
  R2D2_REQUIRE(out, "null handle pointer");
  *out = nullptr;
  if (hidden < 32 || hidden > 512 || hidden % 32 != 0)
    return unsupported("hidden size " + std::to_string(hidden) + ": the act kernels take H a multiple of 32 in [32, 512]");
  if (act < 1 || act > 32) return unsupported("n_actions " + std::to_string(act) + ": the act kernels take 1 <= A <= 32");
  R2D2_REQUIRE(obs >= 1, "obs_size >= 1");
  R2D2_REQUIRE(max_batch >= 1 && max_batch <= (1 << 20), "1 <= max_batch <= 2^20");
  Act* a = new Act();
  a->O = obs; a->A = act; a->H = hidden; a->max_batch = max_batch;
  a->KT = 2 * hidden / TBK; a->MT = hidden / 32; a->NT = ceil_div(max_batch, 128);
  const size_t w_bytes = (size_t)4 * a->MT * a->KT * TILE_BYTES, x_bytes = (size_t)4 * a->NT * a->KT * TILE_BYTES;
  const size_t H = hidden, O = obs, A = act;
  // segments of the small-tensor block, each rounded up to 64 floats: the step kernels use 16-byte vector accesses
  auto seg = [](size_t n) { return (n + 63) & ~(size_t)63; };
  const size_t s_w1t = seg(4 * O * H), s_w1a = seg(2 * A * H), s_b1 = seg(4 * H), s_bg = seg(16 * H), s_w3 = seg(2 * A * H),
               s_b3 = seg(2 * A);
  const size_t floats = s_w1t + s_w1a + s_b1 + s_bg + s_w3 + s_b3 + seg(2 * (size_t)max_batch * H);
  auto fail = [&](int rc) { act_destroy(a); return rc; };
  if (cudaMalloc(&a->w_img, w_bytes) != cudaSuccess || cudaMalloc(&a->x_img, x_bytes) != cudaSuccess ||
      cudaMalloc(&a->w1t, floats * sizeof(float)) != cudaSuccess || cudaMalloc(&a->err, sizeof(int)) != cudaSuccess) {
    set_last_error("r2d2_act_create: cudaMalloc failed");
    return fail(R2D2_ERR_CUDA);
  }
  a->w1a = a->w1t + s_w1t;
  a->b1 = a->w1a + s_w1a;
  a->bg = a->b1 + s_b1;
  a->w3 = a->bg + s_bg;
  a->b3 = a->w3 + s_w3;
  a->pre = a->b3 + s_b3;
  // batch rows past B of the last tile are read by the MMA (N rounded up to 16) and never written: keep them finite
  if (cudaMemset(a->x_img, 0, x_bytes) != cudaSuccess || cudaMemset(a->err, 0, sizeof(int)) != cudaSuccess ||
      cudaDeviceSynchronize() != cudaSuccess) {
    set_last_error("r2d2_act_create: cudaMemset failed");
    return fail(R2D2_ERR_CUDA);
  }
  *out = a;
  return R2D2_OK;
}

int act_destroy(Act* a) {
  if (!a) return R2D2_OK;
  cudaFree(a->w_img);
  cudaFree(a->x_img);
  cudaFree(a->w1t);
  cudaFree(a->err);
  delete a;
  return R2D2_OK;
}

int act_load(Act* a, const float* const params[4], cudaStream_t stream) {
  R2D2_REQUIRE(a, "null handle");
  for (int e = 0; e < 4; ++e) R2D2_REQUIRE(params[e], "four parameter blocks");
  NetPtrs np;
  for (int e = 0; e < 4; ++e) np.p[e] = params[e];
  act_pack_w_kernel<<<dim3(a->KT, a->MT, 4), 256, 0, stream>>>(np, a->O, a->A, a->H, a->MT, a->KT, a->w_img);
  R2D2_CUDA_TRY(cudaGetLastError());
  act_prep_kernel<<<dim3(64, 4), 256, 0, stream>>>(np, a->O, a->A, a->H, a->w1t, a->w1a, a->b1, a->bg, a->w3, a->b3);
  R2D2_CUDA_TRY(cudaGetLastError());
  count_launch(2);
  a->loaded = true;
  return R2D2_OK;
}

int act_step(Act* a, const float* obs, const float* state_in, float* state_out, float* mu, int B, cudaStream_t stream) {
  R2D2_REQUIRE(a, "null handle");
  R2D2_REQUIRE(obs && state_in && state_out && mu, "null tensor");
  R2D2_REQUIRE(B >= 1 && B <= a->max_batch, "1 <= B <= max_batch");
  const size_t st_bytes = (size_t)8 * B * a->H * sizeof(float);
  const char *si = reinterpret_cast<const char*>(state_in), *so = reinterpret_cast<const char*>(state_out);
  R2D2_REQUIRE(so + st_bytes <= si || si + st_bytes <= so, "state_out must not alias state_in");
  R2D2_REQUIRE(((reinterpret_cast<uintptr_t>(state_in) | reinterpret_cast<uintptr_t>(state_out)) & 15) == 0,
               "16-byte aligned state buffers");
  if (!a->loaded) {
    set_last_error("r2d2_act_step: no weights loaded (r2d2_act_load)");
    return R2D2_ERR_STATE;
  }
  static PerDeviceOnce once;
  if (once.need()) R2D2_CUDA_TRY(cudaFuncSetAttribute(act_gate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GATE_SMEM));
  const int H = a->H, KT = a->KT, NT = a->NT;
  act_l1_kernel<<<dim3(H / 32, ceil_div(B, 32), 4), 128, 0, stream>>>(obs, state_in, a->w1t, a->b1, a->x_img, a->pre, B,
                                                                      a->O, H, NT, KT);
  R2D2_CUDA_TRY(cudaGetLastError());
  GateParams g;
  g.w_img = a->w_img; g.x_img = a->x_img; g.bg = a->bg; g.state_in = state_in; g.state_out = state_out; g.e0 = 0;
  g.B = B; g.H = H; g.MT = a->MT; g.NT = NT; g.KT = KT; g.err = a->err;
  const dim3 grid(ceil_div(B, 256), a->MT, 2);
  act_gate_kernel<<<grid, GATE_THREADS, GATE_SMEM, stream>>>(g);
  R2D2_CUDA_TRY(cudaGetLastError());
  act_bridge_kernel<<<dim3(B, 2), 128, 0, stream>>>(state_out, a->w3, a->b3, a->w1a, a->pre, a->x_img, mu, B, a->A, H,
                                                    NT, KT);
  R2D2_CUDA_TRY(cudaGetLastError());
  g.w_img = a->w_img + (size_t)2 * a->MT * KT * TILE_BYTES;
  g.x_img = a->x_img + (size_t)2 * NT * KT * TILE_BYTES;
  g.bg = a->bg + (size_t)2 * 4 * H;
  g.e0 = 2;
  act_gate_kernel<<<grid, GATE_THREADS, GATE_SMEM, stream>>>(g);
  R2D2_CUDA_TRY(cudaGetLastError());
  count_launch(4);
  return R2D2_OK;
}

int act_status(Act* a, int* status, cudaStream_t stream) {
  R2D2_REQUIRE(a && status, "null");
  R2D2_CUDA_TRY(cudaStreamSynchronize(stream));
  R2D2_CUDA_TRY(cudaMemcpy(status, a->err, sizeof(int), cudaMemcpyDeviceToHost));
  return R2D2_OK;
}

}  // namespace r2d2
