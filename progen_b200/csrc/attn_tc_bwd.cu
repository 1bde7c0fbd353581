// Sliding-window attention BACKWARD on tcgen05 tensor cores (sm_100a), bf16, dim_head 64, window % 128 == 0.
// Two kernels without atomics, both built like the forward (attn_tc.cu): TMA-staged operand tiles, tcgen05.mma into
// double-buffered TMEM tiles, element-wise work by threads that own a (row, half-of-the-columns) slice, results kept in
// TMEM across the inner loop.
//
//   dQ  kernel: one work item = 128 query rows.  For every visible 64-key tile j:
//        S  = Q K_j^T            (128 x 64 x 64)      dP = dO V_j^T          (128 x 64 x 64)      -> TMEM
//        dS = exp2(S c - lse) o (dP - delta) / sqrt(dh)                       threads -> bf16 K-major smem tile
//        dQ += dS K_j            (128 x 64 x 64, K_j read MN-major from the same smem tile)       -> TMEM, whole item
//      prologue: delta = rowsum(dO o O) (also written out for the dK/dV kernel); epilogue: rotary backward fused.
//   dKV kernel: one work item = 128 key rows.  For every 64-query tile j that can see them:
//        S^T = K Q_j^T, dP^T = V dO_j^T -> TMEM;  P^T, dS^T -> two bf16 smem tiles
//        dV += P^T dO_j,  dK += dS^T Q_j   (Q_j / dO_j read MN-major from the tiles already in smem)  -> TMEM, whole item
#include "tc_ptx.cuh"
#include "../../include/progen_b200.h"

int attn_bwd_ts_launch(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta,
                       const float* rot_sin, const float* rot_cos, const float* rot_sin_t, const float* rot_cos_t, int B,
                       int seq_len, int window, int heads, int mode, cudaStream_t s);

namespace {

using namespace tc;

constexpr int DH = 64;
constexpr int RB = 128;               // rows owned by a work item (queries for dQ, keys for dKV)
constexpr int CT = 64;                // columns streamed per step (keys for dQ, queries for dKV)
constexpr int ROW_TILE_BYTES = RB * DH * 2;    // 16 KiB
constexpr int COL_TILE_BYTES = CT * DH * 2;    // 8 KiB
constexpr int ES_BYTES = RB * CT * 2;          // 16 KiB element-wise result tile [128 x 64] bf16, K-major
constexpr int TMEM_COLS = 512;
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void named_bar_256() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

struct BwdDev {
  int B, n, w, h;
  const bf16* out;       // [T, I]   (dQ kernel: delta)
  const bf16* dout;      // [T, I]
  const float* lse;      // [T, h]
  float* delta;          // [T, h]   written by the dQ kernel, read by the dKV kernel
  bf16* dqkv;            // [T, 3I]
  const float* rot_sin;  // [n, 32] or null
  const float* rot_cos;
};

// store 32 fp32 gradient values of one row (channels ch0..ch0+31 of one head) as bf16, un-rotating pairs when tables given
__device__ __forceinline__ void store_grad_row(const BwdDev& a, bf16* dst, int pos, int ch0, const float (&v)[32]) {
  float o[32];
  if (a.rot_sin) {
    const float* sp = a.rot_sin + pos * (DH / 2) + (ch0 >> 1);
    const float* cp = a.rot_cos + pos * (DH / 2) + (ch0 >> 1);
    float s[16], c[16];
    load_vec<16>(sp, s);
    load_vec<16>(cp, c);
#pragma unroll
    for (int i = 0; i < 16; ++i) {                       // d/d(x0,x1) of (x0 c - x1 s, x1 c + x0 s)
      o[2 * i] = v[2 * i] * c[i] + v[2 * i + 1] * s[i];
      o[2 * i + 1] = v[2 * i + 1] * c[i] - v[2 * i] * s[i];
    }
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i) o[i] = v[i];
  }
  store_vec<32>(dst, o);
}

// write 32 consecutive columns (col0 = half * 32) of row `row` into a [128 x 64] K-major 128B-swizzled bf16 tile
__device__ __forceinline__ void write_es_row(uint8_t* tile, int row, int half, const float (&v)[32]) {
  uint8_t* prow = tile + row * 128;
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) {
    uint4 t;
    t.x = pack_bf16x2(v[8 * ch], v[8 * ch + 1]); t.y = pack_bf16x2(v[8 * ch + 2], v[8 * ch + 3]);
    t.z = pack_bf16x2(v[8 * ch + 4], v[8 * ch + 5]); t.w = pack_bf16x2(v[8 * ch + 6], v[8 * ch + 7]);
    *reinterpret_cast<uint4*>(prow + (((half * 4 + ch) ^ (row & 7)) << 4)) = t;
  }
}

// ===================================================================================================== dQ
namespace dq {
constexpr int KV_STAGES = 4;
constexpr int KV_BYTES = 2 * COL_TILE_BYTES;                                   // K_j then V_j
constexpr int OFF_Q = 0, OFF_DO = ROW_TILE_BYTES, OFF_KV = 2 * ROW_TILE_BYTES;
constexpr int OFF_DS = OFF_KV + KV_STAGES * KV_BYTES;
constexpr int OFF_BAR = OFF_DS + 2 * ES_BYTES;
constexpr int BAR_BYTES = 256 + 2 * RB * 4;                                    // barriers + delta exchange [2][128]
constexpr int SMEM_BYTES = OFF_BAR + BAR_BYTES + 1024;
}  // namespace dq

struct QItem { int b, hh, q0, win, i0, nprev, ntiles; };
__device__ __forceinline__ bool decode_qitem(const BwdDev& a, int wi, QItem& it) {
  const int qtiles = a.n / RB;
  if (wi >= a.B * a.h * qtiles) return false;
  const int qt = wi % qtiles, r = wi / qtiles;
  it.hh = r % a.h; it.b = r / a.h;
  it.q0 = qt * RB; it.win = it.q0 / a.w; it.i0 = it.q0 % a.w;
  it.nprev = it.win > 0 ? a.w / CT : 0;                  // zero look-back keys of window 0 carry no gradient (K == 0)
  it.ntiles = it.nprev + (it.i0 + RB) / CT;
  return true;
}

__global__ void __launch_bounds__(384, 1) attn_bwd_dq_tc_kernel(const __grid_constant__ CUtensorMap tmap_qkv,
                                                               const __grid_constant__ CUtensorMap tmap_kv,
                                                               const __grid_constant__ CUtensorMap tmap_do, const BwdDev a) {
  using namespace dq;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sQ = base + OFF_Q, sDO = base + OFF_DO, sKV = base + OFF_KV, sDS = base + OFF_DS, bars = base + OFF_BAR;
  const uint32_t qdo_full = bars, qdo_empty = bars + 8, dq_full = bars + 16, dq_empty = bars + 24;
  auto kv_full = [&](int s) { return bars + 32 + 8 * s; };
  auto kv_empty = [&](int s) { return bars + 64 + 8 * s; };
  auto sd_full = [&](int i) { return bars + 96 + 8 * i; };
  auto sd_empty = [&](int i) { return bars + 112 + 8 * i; };
  auto ds_full = [&](int i) { return bars + 128 + 8 * i; };
  auto ds_empty = [&](int i) { return bars + 144 + 8 * i; };
  const uint32_t tmem_slot = bars + 160;
  float* xd = reinterpret_cast<float*>(gen + OFF_BAR + 256);                   // delta exchange [2][128]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int I = a.h * DH;

  if (warp == 0 && lane == 0) { prefetch_tensormap(&tmap_qkv); prefetch_tensormap(&tmap_kv); prefetch_tensormap(&tmap_do); }
  if (warp == 1 && lane == 0) {
    mbar_init(qdo_full, 1); mbar_init(qdo_empty, 1); mbar_init(dq_full, 1); mbar_init(dq_empty, 8);
    for (int s = 0; s < KV_STAGES; ++s) { mbar_init(kv_full(s), 1); mbar_init(kv_empty(s), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(sd_full(i), 1); mbar_init(sd_empty(i), 8); mbar_init(ds_full(i), 8); mbar_init(ds_empty(i), 1); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + OFF_BAR + 160);
  // TMEM: step buffer b: S at b*128, dP at b*128 + 64;  dQ at 256
  auto key_pos = [&](const QItem& it, int kt) { return kt < it.nprev ? (it.win - 1) * a.w + kt * CT : it.win * a.w + (kt - it.nprev) * CT; };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t kv_phase = 0, q_phase = 0;
      QItem it;
      for (int wi = blockIdx.x; decode_qitem(a, wi, it); wi += gridDim.x) {
        const int row0 = it.b * a.n;
        mbar_wait(qdo_empty, q_phase ^ 1);
        mbar_expect_tx(qdo_full, 2 * ROW_TILE_BYTES);
        tma_load_2d(sQ, &tmap_qkv, qdo_full, it.hh * DH, row0 + it.q0);
        tma_load_2d(sDO, &tmap_do, qdo_full, it.hh * DH, row0 + it.q0);
        q_phase ^= 1;
        for (int kt = 0; kt < it.ntiles; ++kt) {
          mbar_wait(kv_empty(stage), kv_phase ^ 1);
          const uint32_t dst = sKV + stage * KV_BYTES;
          const int kp = row0 + key_pos(it, kt);
          mbar_expect_tx(kv_full(stage), KV_BYTES);
          tma_load_2d(dst, &tmap_kv, kv_full(stage), I + it.hh * DH, kp);                       // 64-row boxes
          tma_load_2d(dst + COL_TILE_BYTES, &tmap_kv, kv_full(stage), 2 * I + it.hh * DH, kp);
          if (++stage == KV_STAGES) { stage = 0; kv_phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc(RB, CT, false, false);      // [128 x 64] = A (K-major) x B^T (K-major), K = dh
      constexpr uint32_t idesc_a = make_idesc(RB, DH, false, true);       // [128 x 64] += dS (K-major, K = keys) x K_j (MN-major)
      int stage = 0;
      uint32_t kv_phase = 0, q_phase = 0, g = 0, item = 0;
      QItem it;
      auto issue_s = [&](int st, uint32_t gi) {
        const uint32_t buf = gi & 1;
        if (gi >= 2) mbar_wait(sd_empty(buf), ((gi - 2) >> 1) & 1);
        tcgen05_fence_after();
        const uint64_t qd = make_smem_desc<false>(sQ), dod = make_smem_desc<false>(sDO);
        const uint64_t kd = make_smem_desc<false>(sKV + st * KV_BYTES), vd = make_smem_desc<false>(sKV + st * KV_BYTES + COL_TILE_BYTES);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) umma_bf16(tmem_base + buf * 128, qd + 2 * k, kd + 2 * k, idesc_s, k > 0);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) umma_bf16(tmem_base + buf * 128 + 64, dod + 2 * k, vd + 2 * k, idesc_s, k > 0);
        tcgen05_commit(sd_full(buf));
      };
      for (int wi = blockIdx.x; decode_qitem(a, wi, it); wi += gridDim.x, ++item) {
        mbar_wait(qdo_full, q_phase);
        q_phase ^= 1;
        int s_stage = stage;
        uint32_t s_phase = kv_phase;
        mbar_wait(kv_full(s_stage), s_phase);
        issue_s(s_stage, g);
        if (++s_stage == KV_STAGES) { s_stage = 0; s_phase ^= 1; }
        for (int j = 0; j < it.ntiles; ++j) {
          if (j + 1 < it.ntiles) {
            mbar_wait(kv_full(s_stage), s_phase);
            issue_s(s_stage, g + j + 1);
            if (++s_stage == KV_STAGES) { s_stage = 0; s_phase ^= 1; }
          } else {
            tcgen05_commit(qdo_empty);                                     // Q / dO tiles no longer needed by any pending MMA
          }
          const uint32_t gj = g + j, buf = gj & 1;
          mbar_wait(ds_full(buf), (gj >> 1) & 1);
          if (j == 0 && item > 0) mbar_wait(dq_empty, (item - 1) & 1);     // previous item's dQ has been read out
          tcgen05_fence_after();
          const uint64_t dsd = make_smem_desc<false>(sDS + buf * ES_BYTES);
          const uint64_t kmn = make_smem_desc<true>(sKV + stage * KV_BYTES);
#pragma unroll
          for (int k = 0; k < CT / 16; ++k)
            umma_bf16(tmem_base + 256, dsd + 2 * k, kmn + (uint64_t)(k * (2048 >> 4)), idesc_a, (j > 0 || k > 0) ? 1u : 0u);
          tcgen05_commit(kv_empty(stage));
          tcgen05_commit(ds_empty(buf));
          if (++stage == KV_STAGES) { stage = 0; kv_phase ^= 1; }
        }
        tcgen05_commit(dq_full);
        g += it.ntiles;
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3, half = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float scale = 0.125f, sc = 0.125f * LOG2E;
    uint32_t g = 0, item = 0;
    QItem it;
    for (int wi = blockIdx.x; decode_qitem(a, wi, it); wi += gridDim.x, ++item) {
      const long long t = (long long)it.b * a.n + it.q0 + row;
      // delta = rowsum(dO o O): each half sums 32 channels, exchanged through smem
      float dpart = 0.f;
      {
        float o[32], d[32];
        load_vec<32>(a.out + t * I + it.hh * DH + half * 32, o);
        load_vec<32>(a.dout + t * I + it.hh * DH + half * 32, d);
#pragma unroll
        for (int i = 0; i < 32; ++i) dpart = fmaf(o[i], d[i], dpart);
      }
      xd[half * RB + row] = dpart;
      named_bar_256();
      const float D = dpart + xd[(half ^ 1) * RB + row];
      named_bar_256();                                                     // xd may be rewritten by the next item
      if (half == 0) a.delta[t * a.h + it.hh] = D;
      const float L2 = a.lse[t * a.h + it.hh] * LOG2E;
      const int qi = it.i0 + row;
      for (int j = 0; j < it.ntiles; ++j) {
        const uint32_t gj = g + j, buf = gj & 1;
        const bool own = j >= it.nprev;
        const int c0 = (j - it.nprev) * CT + half * 32;                    // in-window offset of this thread's first key column
        mbar_wait(sd_full(buf), (gj >> 1) & 1);
        tcgen05_fence_after();
        float s[32], dp[32];
        tmem_ld32(tmem_base + buf * 128 + half * 32 + lane_addr, s);
        tmem_ld32(tmem_base + buf * 128 + 64 + half * 32 + lane_addr, dp);
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(sd_empty(buf));
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float p = ex2_approx(s[i] * sc - L2);
          if (own && c0 + i > qi) p = 0.f;
          s[i] = p * (dp[i] - D) * scale;
        }
        if (gj >= 2) mbar_wait(ds_empty(buf), ((gj - 2) >> 1) & 1);        // MMA finished reading the tile of step gj-2
        write_es_row(gen + OFF_DS + buf * ES_BYTES, row, half, s);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(ds_full(buf));
      }
      g += it.ntiles;
      mbar_wait(dq_full, item & 1);
      tcgen05_fence_after();
      float dqv[32];
      tmem_ld32(tmem_base + 256 + half * 32 + lane_addr, dqv);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(dq_empty);
      store_grad_row(a, a.dqkv + t * (3LL * I) + it.hh * DH + half * 32, it.q0 + row, half * 32, dqv);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) { tcgen05_fence_after(); tmem_dealloc<TMEM_COLS>(tmem_base); }
}

// ===================================================================================================== dK, dV
namespace dkv {
constexpr int Q_STAGES = 3;
constexpr int QS_BYTES = 2 * COL_TILE_BYTES;                                   // Q_j then dO_j
constexpr int OFF_K = 0, OFF_V = ROW_TILE_BYTES, OFF_QS = 2 * ROW_TILE_BYTES;
constexpr int OFF_ES = OFF_QS + Q_STAGES * QS_BYTES;                           // [2 bufs][P^T | dS^T]
constexpr int OFF_BAR = OFF_ES + 4 * ES_BYTES;
constexpr int BAR_BYTES = 256 + 2 * 2 * CT * 4;                                // barriers + [2 bufs][lse*log2e | delta][64]
constexpr int SMEM_BYTES = OFF_BAR + BAR_BYTES + 1024;
}  // namespace dkv

struct KItem { int b, hh, k0, win, j0, nown, ntiles; };
__device__ __forceinline__ bool decode_kitem(const BwdDev& a, int wi, KItem& it) {
  const int ktiles = a.n / RB;
  if (wi >= a.B * a.h * ktiles) return false;
  const int kt = wi % ktiles, r = wi / ktiles;
  it.hh = r % a.h; it.b = r / a.h;
  it.k0 = kt * RB; it.win = it.k0 / a.w; it.j0 = it.k0 % a.w;
  it.nown = (a.w - it.j0) / CT;                                                // query tiles of the own window from the diagonal on
  it.ntiles = it.nown + ((it.win + 1 < a.n / a.w) ? a.w / CT : 0);            // + the whole next window
  return true;
}

__global__ void __launch_bounds__(384, 1) attn_bwd_dkv_tc_kernel(const __grid_constant__ CUtensorMap tmap_qkv_row,
                                                                const __grid_constant__ CUtensorMap tmap_qkv_col,
                                                                const __grid_constant__ CUtensorMap tmap_do_col, const BwdDev a) {
  using namespace dkv;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sK = base + OFF_K, sV = base + OFF_V, sQS = base + OFF_QS, sES = base + OFF_ES, bars = base + OFF_BAR;
  const uint32_t kvi_full = bars, kvi_empty = bars + 8, acc_full = bars + 16, acc_empty = bars + 24;
  auto qs_full = [&](int s) { return bars + 32 + 8 * s; };
  auto qs_empty = [&](int s) { return bars + 56 + 8 * s; };
  auto st_full = [&](int i) { return bars + 80 + 8 * i; };
  auto st_empty = [&](int i) { return bars + 96 + 8 * i; };
  auto es_full = [&](int i) { return bars + 112 + 8 * i; };
  auto es_empty = [&](int i) { return bars + 128 + 8 * i; };
  const uint32_t tmem_slot = bars + 144;
  float* xq = reinterpret_cast<float*>(gen + OFF_BAR + 256);                   // [2 bufs][2][64]: lse*log2e, delta of the query columns

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int I = a.h * DH;

  if (warp == 0 && lane == 0) { prefetch_tensormap(&tmap_qkv_row); prefetch_tensormap(&tmap_qkv_col); prefetch_tensormap(&tmap_do_col); }
  if (warp == 1 && lane == 0) {
    mbar_init(kvi_full, 1); mbar_init(kvi_empty, 1); mbar_init(acc_full, 1); mbar_init(acc_empty, 8);
    for (int s = 0; s < Q_STAGES; ++s) { mbar_init(qs_full(s), 1); mbar_init(qs_empty(s), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(st_full(i), 1); mbar_init(st_empty(i), 8); mbar_init(es_full(i), 8); mbar_init(es_empty(i), 1); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + OFF_BAR + 144);
  // TMEM: step buffer b: S^T at b*128, dP^T at b*128 + 64;  dK at 256, dV at 320
  auto q_pos = [&](const KItem& it, int qt) { return qt < it.nown ? it.win * a.w + it.j0 + qt * CT : (it.win + 1) * a.w + (qt - it.nown) * CT; };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t q_phase = 0, kv_phase = 0;
      KItem it;
      for (int wi = blockIdx.x; decode_kitem(a, wi, it); wi += gridDim.x) {
        const int row0 = it.b * a.n;
        mbar_wait(kvi_empty, kv_phase ^ 1);
        mbar_expect_tx(kvi_full, 2 * ROW_TILE_BYTES);
        tma_load_2d(sK, &tmap_qkv_row, kvi_full, I + it.hh * DH, row0 + it.k0);
        tma_load_2d(sV, &tmap_qkv_row, kvi_full, 2 * I + it.hh * DH, row0 + it.k0);
        kv_phase ^= 1;
        for (int qt = 0; qt < it.ntiles; ++qt) {
          mbar_wait(qs_empty(stage), q_phase ^ 1);
          const uint32_t dst = sQS + stage * QS_BYTES;
          const int qp = row0 + q_pos(it, qt);
          mbar_expect_tx(qs_full(stage), QS_BYTES);
          tma_load_2d(dst, &tmap_qkv_col, qs_full(stage), it.hh * DH, qp);
          tma_load_2d(dst + COL_TILE_BYTES, &tmap_do_col, qs_full(stage), it.hh * DH, qp);
          if (++stage == Q_STAGES) { stage = 0; q_phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc(RB, CT, false, false);      // S^T / dP^T [128 keys x 64 queries], K = dh
      constexpr uint32_t idesc_a = make_idesc(RB, DH, false, true);       // dV / dK [128 keys x 64 dh], K = queries, B MN-major
      int stage = 0;
      uint32_t q_phase = 0, kv_phase = 0, g = 0, item = 0;
      KItem it;
      auto issue_s = [&](int st, uint32_t gi) {
        const uint32_t buf = gi & 1;
        if (gi >= 2) mbar_wait(st_empty(buf), ((gi - 2) >> 1) & 1);
        tcgen05_fence_after();
        const uint64_t kd = make_smem_desc<false>(sK), vd = make_smem_desc<false>(sV);
        const uint64_t qd = make_smem_desc<false>(sQS + st * QS_BYTES), dod = make_smem_desc<false>(sQS + st * QS_BYTES + COL_TILE_BYTES);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) umma_bf16(tmem_base + buf * 128, kd + 2 * k, qd + 2 * k, idesc_s, k > 0);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) umma_bf16(tmem_base + buf * 128 + 64, vd + 2 * k, dod + 2 * k, idesc_s, k > 0);
        tcgen05_commit(st_full(buf));
      };
      for (int wi = blockIdx.x; decode_kitem(a, wi, it); wi += gridDim.x, ++item) {
        mbar_wait(kvi_full, kv_phase);
        kv_phase ^= 1;
        int s_stage = stage;
        uint32_t s_phase = q_phase;
        mbar_wait(qs_full(s_stage), s_phase);
        issue_s(s_stage, g);
        if (++s_stage == Q_STAGES) { s_stage = 0; s_phase ^= 1; }
        for (int j = 0; j < it.ntiles; ++j) {
          if (j + 1 < it.ntiles) {
            mbar_wait(qs_full(s_stage), s_phase);
            issue_s(s_stage, g + j + 1);
            if (++s_stage == Q_STAGES) { s_stage = 0; s_phase ^= 1; }
          } else {
            tcgen05_commit(kvi_empty);                                     // K / V row tiles free for the next item
          }
          const uint32_t gj = g + j, buf = gj & 1;
          mbar_wait(es_full(buf), (gj >> 1) & 1);
          if (j == 0 && item > 0) mbar_wait(acc_empty, (item - 1) & 1);
          tcgen05_fence_after();
          const uint64_t ptd = make_smem_desc<false>(sES + (2 * buf) * ES_BYTES);
          const uint64_t dsd = make_smem_desc<false>(sES + (2 * buf + 1) * ES_BYTES);
          const uint64_t qmn = make_smem_desc<true>(sQS + stage * QS_BYTES);
          const uint64_t domn = make_smem_desc<true>(sQS + stage * QS_BYTES + COL_TILE_BYTES);
          const uint32_t acc = (j > 0) ? 1u : 0u;
#pragma unroll
          for (int k = 0; k < CT / 16; ++k)                                // dV += P^T dO_j
            umma_bf16(tmem_base + 320, ptd + 2 * k, domn + (uint64_t)(k * (2048 >> 4)), idesc_a, (acc || k > 0) ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < CT / 16; ++k)                                // dK += dS^T Q_j
            umma_bf16(tmem_base + 256, dsd + 2 * k, qmn + (uint64_t)(k * (2048 >> 4)), idesc_a, (acc || k > 0) ? 1u : 0u);
          tcgen05_commit(qs_empty(stage));
          tcgen05_commit(es_empty(buf));
          if (++stage == Q_STAGES) { stage = 0; q_phase ^= 1; }
        }
        tcgen05_commit(acc_full);
        g += it.ntiles;
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3, half = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const int cidx = threadIdx.x - 128;                                        // 0..255 among the compute threads
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float scale = 0.125f, sc = 0.125f * LOG2E;
    uint32_t g = 0, item = 0;
    KItem it;
    for (int wi = blockIdx.x; decode_kitem(a, wi, it); wi += gridDim.x, ++item) {
      const long long row0 = (long long)it.b * a.n;
      const int kj = it.j0 + row;                                              // in-window offset of this thread's key row
      for (int j = 0; j < it.ntiles; ++j) {
        const uint32_t gj = g + j, buf = gj & 1;
        const bool own = j < it.nown;
        const int qp = q_pos(it, j);
        // per-column constants of this query tile: 64 threads fetch lse*log2e, 64 fetch delta
        float* xl = xq + buf * 2 * CT;
        if (cidx < CT) xl[cidx] = a.lse[(row0 + qp + cidx) * a.h + it.hh] * LOG2E;
        else if (cidx < 2 * CT) xl[cidx] = a.delta[(row0 + qp + cidx - CT) * a.h + it.hh];
        named_bar_256();
        mbar_wait(st_full(buf), (gj >> 1) & 1);
        tcgen05_fence_after();
        float s[32], dp[32];
        tmem_ld32(tmem_base + buf * 128 + half * 32 + lane_addr, s);
        tmem_ld32(tmem_base + buf * 128 + 64 + half * 32 + lane_addr, dp);
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(st_empty(buf));
        const int c0 = it.j0 + j * CT + half * 32;                             // in-window offset of this thread's first query column (own window)
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float p = ex2_approx(s[i] * sc - xl[half * 32 + i]);
          if (own && kj > c0 + i) p = 0.f;                                     // key after query: masked
          dp[i] = p * (dp[i] - xl[CT + half * 32 + i]) * scale;                // dS^T
          s[i] = p;                                                            // P^T
        }
        if (gj >= 2) mbar_wait(es_empty(buf), ((gj - 2) >> 1) & 1);
        write_es_row(gen + OFF_ES + (2 * buf) * ES_BYTES, row, half, s);
        write_es_row(gen + OFF_ES + (2 * buf + 1) * ES_BYTES, row, half, dp);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(es_full(buf));
      }
      g += it.ntiles;
      mbar_wait(acc_full, item & 1);
      tcgen05_fence_after();
      float dk[32], dv[32];
      tmem_ld32(tmem_base + 256 + half * 32 + lane_addr, dk);
      tmem_ld32(tmem_base + 320 + half * 32 + lane_addr, dv);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      const long long t = row0 + it.k0 + row;
      bf16* dst = a.dqkv + t * (3LL * I) + I + it.hh * DH + half * 32;
      store_grad_row(a, dst, it.k0 + row, half * 32, dk);
      store_grad_row(a, dst + I, it.k0 + row, half * 32, dv);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) { tcgen05_fence_after(); tmem_dealloc<TMEM_COLS>(tmem_base); }
}

#include "attn_tc_bwd_pair.cuh"

}  // namespace

extern "C" {

// tcgen05 backward; same contract as progen_local_attn_bwd (delta is produced by the dQ kernel), window % 128 == 0.
int progen_local_attn_bwd_tc_ex(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta,
                                const float* rot_sin, const float* rot_cos, const float* rot_sin_t, const float* rot_cos_t, int B,
                                int seq_len, int window, int heads, int dim_head, int mode, void* stream) {
  PG_CHECK_ARG(B > 0 && heads > 0 && dim_head == DH && window % 128 == 0 && seq_len % window == 0);
  PG_CHECK_ARG(!rot_sin == !rot_cos && !rot_sin_t == !rot_cos_t && (rot_sin || !rot_sin_t));
  // round-2 kernels (element-wise results in tensor memory, alternating groups; attn_bwd_ts.cu)
  const int rc_ts = attn_bwd_ts_launch(qkv, out, dout, lse, dqkv, delta, rot_sin, rot_cos, rot_sin_t, rot_cos_t, B, seq_len,
                                       window, heads, mode, (cudaStream_t)stream);
  if (rc_ts <= 0) return rc_ts;
  const long long T = (long long)B * seq_len;
  const int I = heads * DH;
  CUtensorMap tq_row, tq_col, tdo_row, tdo_col;
  int rc = pg_tensor_map_2d_bf16(qkv, 3ull * I, (uint64_t)T, 3ull * I, DH, RB, &tq_row);
  if (rc) return rc;
  rc = pg_tensor_map_2d_bf16(qkv, 3ull * I, (uint64_t)T, 3ull * I, DH, CT, &tq_col);
  if (rc) return rc;
  rc = pg_tensor_map_2d_bf16(dout, (uint64_t)I, (uint64_t)T, (uint64_t)I, DH, RB, &tdo_row);
  if (rc) return rc;
  rc = pg_tensor_map_2d_bf16(dout, (uint64_t)I, (uint64_t)T, (uint64_t)I, DH, CT, &tdo_col);
  if (rc) return rc;
  static bool once = false;
  if (!once) {
    PG_CUDA(cudaFuncSetAttribute(attn_bwd_dq_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dq::SMEM_BYTES));
    PG_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dkv::SMEM_BYTES));
    once = true;
  }
  BwdDev a{B, seq_len, window, heads, (const bf16*)out, (const bf16*)dout, lse, delta, (bf16*)dqkv, rot_sin, rot_cos};
  cudaStream_t s = (cudaStream_t)stream;
  static int pair_enabled = [] { const char* e = getenv("PROGEN_ATTN_PAIR"); return e ? atoi(e) : 1; }();
  if (pair_enabled && window % (2 * RB) == 0) {
    // two 128-row work items per CTA, one element-wise warp group each (attn_tc_bwd_pair.cuh)
    static bool once_pair = false;
    if (!once_pair) {
      PG_CUDA(cudaFuncSetAttribute(attn_bwd_dq_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dqp::SMEM_BYTES));
      PG_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dkvp::SMEM_BYTES));
      once_pair = true;
    }
    const long long pitems = (long long)B * heads * (seq_len / (2 * RB));
    const int pgrid = (int)(pitems < pg_num_sms() ? pitems : pg_num_sms());
    attn_bwd_dq_pair_kernel<<<pgrid, 384, dqp::SMEM_BYTES, s>>>(tq_row, tq_col, tdo_row, a);
    PG_LAUNCH_CHECK();
    attn_bwd_dkv_pair_kernel<<<pgrid, 384, dkvp::SMEM_BYTES, s>>>(tq_row, tq_col, tdo_col, a);
    PG_LAUNCH_CHECK();
    return PROGEN_OK;
  }
  const long long items = (long long)B * heads * (seq_len / RB);
  const int grid = (int)(items < pg_num_sms() ? items : pg_num_sms());
  // dQ: K/V column tiles are 64 rows of the qkv tensor, Q / dO row tiles 128 rows
  attn_bwd_dq_tc_kernel<<<grid, 384, dq::SMEM_BYTES, s>>>(tq_row, tq_col, tdo_row, a);
  PG_LAUNCH_CHECK();
  attn_bwd_dkv_tc_kernel<<<grid, 384, dkv::SMEM_BYTES, s>>>(tq_row, tq_col, tdo_col, a);
  PG_LAUNCH_CHECK();
  return PROGEN_OK;
}

int progen_local_attn_bwd_tc(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta,
                             const float* rot_sin, const float* rot_cos, int B, int seq_len, int window, int heads, int dim_head,
                             void* stream) {
  return progen_local_attn_bwd_tc_ex(qkv, out, dout, lse, dqkv, delta, rot_sin, rot_cos, nullptr, nullptr, B, seq_len, window,
                                     heads, dim_head, -1, stream);
}

}  // extern "C"
