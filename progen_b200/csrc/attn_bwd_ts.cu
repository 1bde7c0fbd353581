// Sliding-window attention BACKWARD, round-2 kernels (window % 128 == 0, dim_head 64): gradient of reference
// progen.py:88-102 with respect to the rotated q | k | v (the rotary backward is fused into the stores).
//
// Round 1 (attn_tc_bwd_pair.cuh) ran both kernels at 20-22 % tensor pipe / 37-40 % issue slots: each 64-column step of a
// group was a chain  S,dP MMAs -> TMEM read -> exp2 / dS -> bf16 tiles in SHARED memory -> proxy fence -> accumulate MMAs
// with TMEM completely allocated (two groups x (S | dP | accumulators)), so a group's next scores could not be computed
// while its current ones were still in use.  Here, for both kernels:
//
//   * a CTA owns ONE 128-row work item at a time (128 keys for dK/dV, 128 queries for dQ) with ONE set of accumulators
//     in TMEM, and its two element-wise warp groups take ALTERNATE 64-column steps of the reduction, each with its own
//     score buffer: TMEM = 3 x (S 64 | dP 64) + accumulators (2 x 64 for dK/dV, 64 for dQ) — three buffers for two groups, so
//     the scores of a group's NEXT step are already there when it finishes the current one (with two buffers both groups
//     exponentiated at the same time and then both waited for the MMAs: XU and tensor pipe took turns);
//   * the element-wise results never touch shared memory: P^T / dS^T (resp. dS) are written back over the score columns
//     as packed bf16 (tcgen05.st) and the accumulate MMAs read their A operand from tensor memory;
//   * one MMA thread walks the step sequence twice, three steps apart: "ahead" issues S / dP of step x+3 into the buffer
//     whose results step x has just consumed, so the tensor pipe works on later scores and earlier accumulations while
//     the groups exponentiate;
//   * packed fp32x2 arithmetic, the 1/sqrt(dh) factor applied once to the accumulators instead of per element, next
//     item's row tiles prefetched (double-buffered), work items ordered heaviest first.
//
//   dQ  kernel (runs first; also writes delta = rowsum(dO o O) for the dK/dV kernel):
//        S = Q K_j^T, dP = dO V_j^T (128 x 64 x 64)  ->  dS = exp2(S c - lse) o (dP - delta)  ->  dQ += dS K_j
//   dKV kernel:  S^T = K Q_j^T, dP^T = V dO_j^T  ->  P^T, dS^T  ->  dV += P^T dO_j,  dK += dS^T Q_j
//
// Gradient stores (template flag TMA_ST, mode 3).  Without it every element-wise thread un-rotates and writes its own
// row (store_grad_row): 128 B per thread with rows 3 KiB apart in dqkv, and the [n, 32] rotary tables read 64 B per thread
// from 32 different lines per warp.  With it, each group stages its half of the finished tiles in shared memory (bf16,
// 64-byte TMA swizzle: conflict-free 16-byte row writes) and one thread of the group writes them with a TMA store; the
// rotary tables are read transposed ([32, n]: a warp's 32 consecutive positions are one 128-byte line per pair index).
// Each group owns its own staging slot and issues its own boxes (128 rows x 32 channels): the two groups run a step
// apart, and a shared 64-channel box would make the earlier group wait for the later one at every item.  In the dK/dV
// kernel group g stores channels [32 g, 32 g + 32) of both dK and dV (one TMEM read-out of 2 x 32 columns per thread, as
// with one whole 64-channel gradient per group).
#include "tc_ptx.cuh"
#include "../../include/progen_b200.h"

namespace {

using namespace tc;

constexpr int DH = 64;
constexpr int RB = 128;               // rows owned by a work item (queries for dQ, keys for dKV)
constexpr int CT = 64;                // columns streamed per step (keys for dQ, queries for dKV)
constexpr int ROW_TILE_BYTES = RB * DH * 2;    // 16 KiB
constexpr int COL_TILE_BYTES = CT * DH * 2;    // 8 KiB
constexpr int NS = 6;                 // column-tile stages
constexpr int NB = 3;                 // score buffers (S | dP, 128 TMEM columns each): step x uses buffer x % 3, group x & 1
constexpr int STAGE_BYTES = 2 * COL_TILE_BYTES;
constexpr int TMEM_COLS = 512;
constexpr float LOG2E = 1.4426950408889634f;
constexpr float SCALE = 0.125f;       // 1/sqrt(dim_head)

struct BwdDev {
  int B, n, w, h;
  const bf16* out;       // [T, I]   (dQ kernel: delta)
  const bf16* dout;      // [T, I]
  const float* lse;      // [T, h]
  float* delta;          // [T, h]   written by the dQ kernel, read by the dKV kernel
  bf16* dqkv;            // [T, 3I]
  const float* rot_sin;  // entry (position p, pair j) at [p * rot_ld_pos + j * rot_ld_pair], or null
  const float* rot_cos;
  int rot_ld_pos, rot_ld_pair;   // [n, 32]: 32, 1;  transposed [32, n]: 1, n
};

// store 32 fp32 gradient values of one row (channels ch0..ch0+31 of one head) as bf16, un-rotating pairs when tables given
// (row-major [n, 32] tables: the launcher gives these kernels no other layout)
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

// ---------------------------------------------------------------------------------------- TMA-store epilogue (TMA_ST)
constexpr int ST_BOX_BYTES = RB * 32 * 2;      // 8 KiB: 128 rows x 32 bf16 channels, 64-byte rows

// un-rotate 32 fp32 values of one row (channels ch0..ch0+31 of one head, position pos) in place when tables are given
__device__ __forceinline__ void unrotate32(const BwdDev& a, int pos, int ch0, float (&v)[32]) {
  if (!a.rot_sin) return;
  const long long e0 = (long long)pos * a.rot_ld_pos + (long long)(ch0 >> 1) * a.rot_ld_pair;
  float s[16], c[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    s[i] = __ldg(a.rot_sin + e0 + (long long)i * a.rot_ld_pair);
    c[i] = __ldg(a.rot_cos + e0 + (long long)i * a.rot_ld_pair);
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {                         // d/d(x0,x1) of (x0 c - x1 s, x1 c + x0 s)
    const float x0 = v[2 * i], x1 = v[2 * i + 1];
    v[2 * i] = x0 * c[i] + x1 * s[i];
    v[2 * i + 1] = x1 * c[i] - x0 * s[i];
  }
}

// row `row` of a [128 x 32] bf16 staging box in the 64-byte TMA swizzle (16-byte chunk c of row r at chunk
// c ^ ((r >> 1) & 3); the box is 1024-byte aligned): 8 consecutive rows cover all 32 banks
__device__ __forceinline__ void stage_row32(uint32_t box, int row, const float (&v)[32]) {
#pragma unroll
  for (int c = 0; c < 4; ++c)
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(box + row * 64 + ((c ^ ((row >> 1) & 3)) << 4)), "r"(pack_bf16x2(v[8 * c], v[8 * c + 1])),
                   "r"(pack_bf16x2(v[8 * c + 2], v[8 * c + 3])), "r"(pack_bf16x2(v[8 * c + 4], v[8 * c + 5])),
                   "r"(pack_bf16x2(v[8 * c + 6], v[8 * c + 7])) : "memory");
}

// the 128 threads of element-wise group g (warps 4 + 4 g .. 7 + 4 g)
__device__ __forceinline__ void group_bar(int g) {
  if (g == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
  else asm volatile("bar.sync 2, 128;" ::: "memory");
}

// ===================================================================================================== dK, dV
namespace dkv {
constexpr int OFF_KV = 0;                                                      // [kvb]: K tile, V tile (128 rows each)
constexpr int OFF_QS = 4 * ROW_TILE_BYTES;                                     // [stage]: Q_t, dO_t (64 rows each)
constexpr int OFF_STAT = OFF_QS + NS * STAGE_BYTES;                            // [stage][lse*log2e | delta][64]
constexpr int STAT_BYTES = 2 * CT * 4;
constexpr int OFF_BAR = OFF_STAT + NS * STAT_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
constexpr int OFF_ST = (OFF_BAR + 256 + 1023) / 1024 * 1024;                   // TMA_ST: [group]: dK box, dV box
constexpr int SMEM_BYTES_ST = OFF_ST + 2 * 2 * ST_BOX_BYTES + 1024;            // 196 KiB with NS = 6
static_assert(SMEM_BYTES_ST <= 227 * 1024, "dK/dV staging slots do not fit");
}  // namespace dkv

// one work item = (batch, head, 128-key tile); its steps are the 64-query tiles that can see those keys: own window
// from the tile's diagonal on, then the whole next window.  Heaviest first: windows before the last by key tile, then the
// last window (no next window: at most half the steps).
struct KItem { int b, hh, k0, win, j0, nown, nT; };
__device__ __forceinline__ bool decode_kitem(const BwdDev& a, int wi, KItem& it) {
  const int nk = a.w / RB, W = a.n / a.w, bh = a.B * a.h;
  if (wi >= bh * nk * W) return false;
  const int nl = bh * (W - 1);
  int kt, r;
  if (wi < nl * nk) { kt = wi / nl; const int v = wi % nl; it.win = v % (W - 1); r = v / (W - 1); }
  else { const int v = wi - nl * nk; kt = v / bh; r = v % bh; it.win = W - 1; }
  it.hh = r % a.h; it.b = r / a.h;
  it.j0 = kt * RB; it.k0 = it.win * a.w + it.j0;
  it.nown = (a.w - it.j0) / CT;
  it.nT = it.nown + (it.win + 1 < W ? a.w / CT : 0);
  return true;
}

template <bool TMA_ST>
__global__ void __launch_bounds__(384, 1) attn_bwd_dkv_ts_kernel(const __grid_constant__ CUtensorMap tmap_qkv_row,
                                                                const __grid_constant__ CUtensorMap tmap_qkv_col,
                                                                const __grid_constant__ CUtensorMap tmap_do_col,
                                                                const __grid_constant__ CUtensorMap tmap_dqkv_st, const BwdDev a) {
  using namespace dkv;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sKV = base + OFF_KV, sQS = base + OFF_QS, bars = base + OFF_BAR;
  auto kv_full = [&](int b) { return bars + 8 * b; };
  auto kv_empty = [&](int b) { return bars + 16 + 8 * b; };
  auto qs_full = [&](int s) { return bars + 32 + 8 * s; };
  auto qs_empty = [&](int s) { return bars + 80 + 8 * s; };
  auto s_full = [&](int b) { return bars + 128 + 8 * b; };
  auto p_full = [&](int b) { return bars + 152 + 8 * b; };
  const uint32_t acc_full = bars + 176, acc_empty = bars + 184, tmem_slot = bars + 192;
  float* stats = reinterpret_cast<float*>(gen + OFF_STAT);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int I = a.h * DH;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmap_qkv_row); prefetch_tensormap(&tmap_qkv_col); prefetch_tensormap(&tmap_do_col);
    if (TMA_ST) prefetch_tensormap(&tmap_dqkv_st);
  }
  if (warp == 1 && lane == 0) {
    for (int b = 0; b < 2; ++b) { mbar_init(kv_full(b), 1); mbar_init(kv_empty(b), 1); }
    for (int s = 0; s < NS; ++s) { mbar_init(qs_full(s), 2); mbar_init(qs_empty(s), 1); }   // full: TMA bytes + the stats warp
    for (int b = 0; b < NB; ++b) { mbar_init(s_full(b), 1); mbar_init(p_full(b), 4); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 8);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + OFF_BAR + 192);
  auto q_pos = [&](const KItem& it, int t) { return t < it.nown ? it.win * a.w + it.j0 + t * CT : (it.win + 1) * a.w + (t - it.nown) * CT; };

  if (warp < 4) {
    setmaxnreg_dec<72>();
    if (warp == 0) {
      // ------------------------------------------------------------------------------------------ TMA producer
      {                                                       // whole warp, one elected lane issues (uniform operands)
        uint32_t x = 0, item = 0;
        KItem it;
        for (int wi = blockIdx.x; decode_kitem(a, wi, it); wi += gridDim.x, ++item) {
          const int row0 = it.b * a.n, kvb = item & 1;
          mbar_wait(kv_empty(kvb), ((item >> 1) & 1) ^ 1);
          if (elect_one()) {
            mbar_expect_tx(kv_full(kvb), 2 * ROW_TILE_BYTES);
            tma_load_2d(sKV + (2 * kvb) * ROW_TILE_BYTES, &tmap_qkv_row, kv_full(kvb), I + it.hh * DH, row0 + it.k0);
            tma_load_2d(sKV + (2 * kvb + 1) * ROW_TILE_BYTES, &tmap_qkv_row, kv_full(kvb), 2 * I + it.hh * DH, row0 + it.k0);
          }
          __syncwarp();
          for (int t = 0; t < it.nT; ++t, ++x) {
            const int st = x % NS;
            mbar_wait(qs_empty(st), ((x / NS) & 1) ^ 1);
            const uint32_t dst = sQS + st * STAGE_BYTES;
            const int qp = row0 + q_pos(it, t);
            if (elect_one()) {
              mbar_expect_tx(qs_full(st), STAGE_BYTES);
              tma_load_2d(dst, &tmap_qkv_col, qs_full(st), it.hh * DH, qp);
              tma_load_2d(dst + COL_TILE_BYTES, &tmap_do_col, qs_full(st), it.hh * DH, qp);
            }
            __syncwarp();
          }
        }
      }
    } else if (warp == 3) {
      // ------------------------------------------------------------------------------------------ per-query constants of a stage
      uint32_t x = 0;
      KItem it;
      for (int wi = blockIdx.x; decode_kitem(a, wi, it); wi += gridDim.x) {
        const long long row0 = (long long)it.b * a.n;
        for (int t = 0; t < it.nT; ++t, ++x) {
          const int st = x % NS;
          mbar_wait(qs_empty(st), ((x / NS) & 1) ^ 1);
          float* xl = stats + st * (2 * CT);
          const long long qp = row0 + q_pos(it, t);
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const long long idx = (qp + r * 32 + lane) * a.h + it.hh;
            xl[r * 32 + lane] = -a.lse[idx] * LOG2E;
            xl[CT + r * 32 + lane] = -a.delta[idx];
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(qs_full(st));
        }
      }
    } else if (warp == 1) {
      // ------------------------------------------------------------------------------------------ MMA issuer
      // (whole warp: descriptors stay in uniform registers — see tc::elect_one; one elected lane issues tcgen05)
      {
        constexpr uint32_t idesc_s = make_idesc(RB, CT, false, false);      // S^T / dP^T [128 keys x 64 queries], K = dh
        constexpr uint32_t idesc_a = make_idesc(RB, DH, false, true);       // dV / dK [128 keys x 64 dh], K = queries, B MN-major
        struct Cur { int wi; uint32_t item; int t; KItem it; bool valid; };
        Cur ahead, cur;
        ahead.wi = blockIdx.x; ahead.item = 0; ahead.t = 0; ahead.valid = decode_kitem(a, ahead.wi, ahead.it);
        cur = ahead;
        auto advance = [&](Cur& c) {
          if (++c.t == c.it.nT) { c.t = 0; c.wi += gridDim.x; ++c.item; c.valid = decode_kitem(a, c.wi, c.it); }
        };
        uint32_t xa = 0;
        auto issue_ahead = [&]() {
          if (!ahead.valid) return;
          const int kvb = ahead.item & 1, st = xa % NS, buf = xa % NB;
          if (ahead.t == 0) mbar_wait(kv_full(kvb), (ahead.item >> 1) & 1);
          mbar_wait(qs_full(st), (xa / NS) & 1);
          tcgen05_fence_after();
          const uint64_t kd = make_smem_desc<false>(sKV + (2 * kvb) * ROW_TILE_BYTES);
          const uint64_t vd = make_smem_desc<false>(sKV + (2 * kvb + 1) * ROW_TILE_BYTES);
          const uint64_t qd = make_smem_desc<false>(sQS + st * STAGE_BYTES), dod = make_smem_desc<false>(sQS + st * STAGE_BYTES + COL_TILE_BYTES);
          const uint32_t tm = tmem_base + buf * 128;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < DH / 16; ++k) umma_bf16(tm, kd + 2 * k, qd + 2 * k, idesc_s, k > 0);
#pragma unroll
            for (int k = 0; k < DH / 16; ++k) umma_bf16(tm + 64, vd + 2 * k, dod + 2 * k, idesc_s, k > 0);
            tcgen05_commit(s_full(buf));
            if (ahead.t == ahead.it.nT - 1) tcgen05_commit(kv_empty(kvb));   // the item's K / V tiles have had their last reader
          }
          __syncwarp();
          advance(ahead);
          ++xa;
        };
        for (int i = 0; i < NB; ++i) issue_ahead();
        for (uint32_t x = 0; cur.valid; ++x) {
          const int st = x % NS, buf = x % NB;
          mbar_wait(p_full(buf), (x / NB) & 1);                              // P^T / dS^T of step x are in tensor memory
          if (cur.t == 0 && cur.item > 0) mbar_wait(acc_empty, (cur.item - 1) & 1);   // previous item's dK / dV have been read out
          tcgen05_fence_after();
          const uint64_t qmn = make_smem_desc<true>(sQS + st * STAGE_BYTES);
          const uint64_t domn = make_smem_desc<true>(sQS + st * STAGE_BYTES + COL_TILE_BYTES);
          const uint32_t tm = tmem_base + buf * 128;
          const uint32_t acc = cur.t > 0 ? 1u : 0u;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < CT / 16; ++k)                                // dV += P^T dO_t
              umma_bf16_ts(tmem_base + 448, tm + 8 * k, domn + (uint64_t)(k * (2048 >> 4)), idesc_a, (acc || k > 0) ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < CT / 16; ++k)                                // dK += dS^T Q_t
              umma_bf16_ts(tmem_base + 384, tm + 64 + 8 * k, qmn + (uint64_t)(k * (2048 >> 4)), idesc_a, (acc || k > 0) ? 1u : 0u);
            tcgen05_commit(qs_empty(st));
            if (cur.t == cur.it.nT - 1) tcgen05_commit(acc_full);
          }
          __syncwarp();
          advance(cur);
          issue_ahead();                                                     // step x+3 into the buffer step x has just released
        }
      }
    }
  } else {
    // -------------------------------------------------------------------------------------------- element-wise groups
    setmaxnreg_inc<216>();
    const int q = warp & 3, g = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float sc = SCALE * LOG2E;
    const float2 sc2 = make_float2(sc, sc);
    uint32_t x = 0, item = 0;
    KItem it;
    // The item's accumulators are read out ONE OWN STEP LATE: after its last step a group goes straight on to the next
    // item (whose scores are already there) and stores the previous item's dK / dV only after that step's P^T / dS^T have
    // been published.  Waiting for the accumulate MMAs of the last step + the epilogue at every item boundary cost 21-28 %
    // of the element-wise warps' time (ncu on the first version of this kernel).
    bool pending = false;
    int pend_b = 0, pend_hh = 0, pend_k0 = 0;
    uint32_t pend_item = 0;
    auto epilogue = [&]() {     // group 0 stores dK (x 1/sqrt(dh)), group 1 stores dV
      if constexpr (TMA_ST) {   // group g: channels [32 g, 32 g + 32) of dK (x 1/sqrt(dh)) and of dV, both un-rotated
        const uint32_t slot = base + OFF_ST + g * (2 * ST_BOX_BYTES);
        mbar_wait(acc_full, pend_item & 1);
        tcgen05_fence_after();
        uint32_t rk[32], rv[32];
        tmem_ld32_issue(tmem_base + lane_addr + 384 + 32 * g, rk);
        tmem_ld32_issue(tmem_base + lane_addr + 448 + 32 * g, rv);
        tmem_ld32_wait(rk);
        tmem_ld32_wait(rv);
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty);
        float vk[32], vv[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) { vk[i] = __uint_as_float(rk[i]) * SCALE; vv[i] = __uint_as_float(rv[i]); }
        unrotate32(a, pend_k0 + row, 32 * g, vk);
        unrotate32(a, pend_k0 + row, 32 * g, vv);                            // v is rotated too (progen.py:36-41)
        if (row == 0) bulk_wait_group_read<0>();                             // the previous item's boxes have left the slot
        group_bar(g);
        stage_row32(slot, row, vk);
        stage_row32(slot + ST_BOX_BYTES, row, vv);
        fence_proxy_async();                                                 // my slot writes -> visible to the TMA store
        group_bar(g);
        if (row == 0) {
          const int r0 = pend_b * a.n + pend_k0, c0 = pend_hh * DH + 32 * g;
          tma_store_2d(&tmap_dqkv_st, slot, I + c0, r0);
          tma_store_2d(&tmap_dqkv_st, slot + ST_BOX_BYTES, 2 * I + c0, r0);
          bulk_commit_group();
        }
        pending = false;
        return;
      }
      mbar_wait(acc_full, pend_item & 1);
      tcgen05_fence_after();
      const long long tr = (long long)pend_b * a.n + pend_k0 + row;
      bf16* out = a.dqkv + tr * (3LL * I) + (g == 0 ? I : 2 * I) + pend_hh * DH;
      const uint32_t src = tmem_base + lane_addr + (g == 0 ? 384 : 448);
      const float mul = g == 0 ? SCALE : 1.f;
      uint32_t r0[32], r1[32];
      tmem_ld32_issue(src, r0);
      tmem_ld32_issue(src + 32, r1);
      tmem_ld32_wait(r0);
      tmem_ld32_wait(r1);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      float v0[32], v1[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) { v0[i] = __uint_as_float(r0[i]) * mul; v1[i] = __uint_as_float(r1[i]) * mul; }
      store_grad_row(a, out, pend_k0 + row, 0, v0);
      store_grad_row(a, out + 32, pend_k0 + row, 32, v1);
      pending = false;
    };
    for (int wi = blockIdx.x; decode_kitem(a, wi, it); wi += gridDim.x, ++item) {
      const int kj = it.j0 + row;                                            // in-window offset of this thread's key row
      for (int t = 0; t < it.nT; ++t, ++x) {
        if ((int)(x & 1) != g) continue;
        const int st = x % NS;
        const uint32_t tm = tmem_base + (x % NB) * 128 + lane_addr;
        mbar_wait(qs_full(st), (x / NS) & 1);                                // the stage's lse / delta columns are visible
        const float* xl = stats + st * (2 * CT);
        mbar_wait(s_full(x % NB), (x / NB) & 1);
        tcgen05_fence_after();
        const bool masked = t < it.nown && t * CT < RB;                      // query tiles on the key tile's diagonal
        const int c0 = it.j0 + t * CT;                                       // in-window offset of the step's first query
        uint32_t pk[32], dk[32];
        uint32_t s[2][32], dp[2][32];
        tmem_ld32_issue(tm, s[0]);
        tmem_ld32_issue(tm + 64, dp[0]);
        tmem_ld32_issue(tm + 32, s[1]);
        tmem_ld32_issue(tm + 96, dp[1]);
        tmem_ld32_wait(s[0]);
        tmem_ld32_wait(dp[0]);
        tmem_ld32_wait(s[1]);
        tmem_ld32_wait(dp[1]);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float2 nl = *reinterpret_cast<const float2*>(xl + half * 32 + i);        // -lse * log2e of queries i, i+1
            const float2 nd = *reinterpret_cast<const float2*>(xl + CT + half * 32 + i);   // -delta
            float2 e = ffma2(make_float2(__uint_as_float(s[half][i]), __uint_as_float(s[half][i + 1])), sc2, nl);
            e.x = ex2f(e.x);
            e.y = ex2f(e.y);
            if (masked) {                                                    // key after query: masked
              if (kj > c0 + half * 32 + i) e.x = 0.f;
              if (kj > c0 + half * 32 + i + 1) e.y = 0.f;
            }
            const float2 dd = fmul2(e, fadd2(make_float2(__uint_as_float(dp[half][i]), __uint_as_float(dp[half][i + 1])), nd));
            pk[half * 16 + i / 2] = pack_bf16x2(e.x, e.y);                   // P^T
            dk[half * 16 + i / 2] = pack_bf16x2(dd.x, dd.y);                 // dS^T (without the 1/sqrt(dh): applied to dK once)
          }
        }
        tmem_st<32>(tm, pk);                                                 // over S^T[0, 32): 64 queries as bf16 pairs
        tmem_st<32>(tm + 64, dk);                                            // over dP^T[0, 32)
        tmem_st_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full(x % NB));
        if (pending) epilogue();                                             // the PREVIOUS item's dK / dV (see above)
      }
      pend_b = it.b; pend_hh = it.hh; pend_k0 = it.k0; pend_item = item; pending = true;
    }
    if (pending) epilogue();
    if (TMA_ST && row == 0) bulk_wait_group<0>();                            // every store has completed before smem goes away
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) { tcgen05_fence_after(); tmem_dealloc<TMEM_COLS>(tmem_base); }
}

// ===================================================================================================== dQ
namespace dq {
constexpr int OFF_QD = 0;                                                      // [qb]: Q tile, dO tile (128 rows each)
constexpr int OFF_KV = 4 * ROW_TILE_BYTES;                                     // [stage]: K_j, V_j (64 rows each)
constexpr int OFF_BAR = OFF_KV + NS * STAGE_BYTES;
constexpr int OFF_RC = OFF_BAR + 256;                                          // [qb][-delta | -lse*log2e][128] row constants
constexpr int SMEM_BYTES = OFF_RC + 2 * 2 * RB * 4 + 1024;
constexpr int OFF_ST = (OFF_RC + 2 * 2 * RB * 4 + 1023) / 1024 * 1024;        // TMA_ST: [group]: dQ box
constexpr int SMEM_BYTES_ST = OFF_ST + 2 * ST_BOX_BYTES + 1024;
static_assert(SMEM_BYTES_ST <= 227 * 1024, "dQ staging slots do not fit");
}  // namespace dq

// one work item = (batch, head, 128-query tile); steps = the visible 64-key tiles (look-back window, then own window up to
// the diagonal).  Window 0's zero look-back keys carry no gradient (K == V == 0 there).  Heaviest first.
struct QItem { int b, hh, q0, win, i0, nprev, nT; };
__device__ __forceinline__ bool decode_qitem(const BwdDev& a, int wi, QItem& it) {
  const int nq = a.w / RB, W = a.n / a.w, bh = a.B * a.h;
  if (wi >= bh * nq * W) return false;
  const int nl = bh * (W - 1);                                                // items per query-tile class outside window 0
  int qt, r;
  if (wi < nl * nq) { qt = nq - 1 - wi / nl; const int v = wi % nl; it.win = 1 + v % (W - 1); r = v / (W - 1); }
  else { const int v = wi - nl * nq; qt = nq - 1 - v / bh; r = v % bh; it.win = 0; }
  it.hh = r % a.h; it.b = r / a.h;
  it.i0 = qt * RB; it.q0 = it.win * a.w + it.i0;
  it.nprev = it.win > 0 ? a.w / CT : 0;
  it.nT = it.nprev + (it.i0 + RB) / CT;
  return true;
}

template <bool POLY, bool TMA_ST>
__global__ void __launch_bounds__(384, 1) attn_bwd_dq_ts_kernel(const __grid_constant__ CUtensorMap tmap_qkv_row,
                                                               const __grid_constant__ CUtensorMap tmap_qkv_col,
                                                               const __grid_constant__ CUtensorMap tmap_do_row,
                                                               const __grid_constant__ CUtensorMap tmap_dqkv_st, const BwdDev a) {
  using namespace dq;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sQD = base + OFF_QD, sKV = base + OFF_KV, bars = base + OFF_BAR;
  auto qd_full = [&](int b) { return bars + 8 * b; };
  auto qd_empty = [&](int b) { return bars + 16 + 8 * b; };
  auto kv_full = [&](int s) { return bars + 32 + 8 * s; };
  auto kv_empty = [&](int s) { return bars + 80 + 8 * s; };
  auto s_full = [&](int b) { return bars + 128 + 8 * b; };
  auto p_full = [&](int b) { return bars + 152 + 8 * b; };
  const uint32_t acc_full = bars + 176, acc_empty = bars + 184, tmem_slot = bars + 192;
  auto rc_full = [&](int b) { return bars + 200 + 8 * b; };
  auto rc_empty = [&](int b) { return bars + 216 + 8 * b; };
  float* rcs = reinterpret_cast<float*>(gen + OFF_RC);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int I = a.h * DH;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmap_qkv_row); prefetch_tensormap(&tmap_qkv_col); prefetch_tensormap(&tmap_do_row);
    if (TMA_ST) prefetch_tensormap(&tmap_dqkv_st);
  }
  if (warp == 1 && lane == 0) {
    for (int b = 0; b < 2; ++b) { mbar_init(qd_full(b), 1); mbar_init(qd_empty(b), 1); }
    for (int s = 0; s < NS; ++s) { mbar_init(kv_full(s), 1); mbar_init(kv_empty(s), 1); }
    for (int b = 0; b < NB; ++b) { mbar_init(s_full(b), 1); mbar_init(p_full(b), 4); }
    for (int b = 0; b < 2; ++b) { mbar_init(rc_full(b), 2); mbar_init(rc_empty(b), 8); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 8);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + OFF_BAR + 192);
  auto key_pos = [&](const QItem& it, int j) { return j < it.nprev ? (it.win - 1) * a.w + j * CT : it.win * a.w + (j - it.nprev) * CT; };

  if (warp < 4) {
    setmaxnreg_dec<72>();
    if (warp == 0) {
      {                                                       // whole warp, one elected lane issues (uniform operands)
        uint32_t x = 0, item = 0;
        QItem it;
        for (int wi = blockIdx.x; decode_qitem(a, wi, it); wi += gridDim.x, ++item) {
          const int row0 = it.b * a.n, qb = item & 1;
          mbar_wait(qd_empty(qb), ((item >> 1) & 1) ^ 1);
          if (elect_one()) {
            mbar_expect_tx(qd_full(qb), 2 * ROW_TILE_BYTES);
            tma_load_2d(sQD + (2 * qb) * ROW_TILE_BYTES, &tmap_qkv_row, qd_full(qb), it.hh * DH, row0 + it.q0);
            tma_load_2d(sQD + (2 * qb + 1) * ROW_TILE_BYTES, &tmap_do_row, qd_full(qb), it.hh * DH, row0 + it.q0);
          }
          __syncwarp();
          for (int j = 0; j < it.nT; ++j, ++x) {
            const int st = x % NS;
            mbar_wait(kv_empty(st), ((x / NS) & 1) ^ 1);
            const uint32_t dst = sKV + st * STAGE_BYTES;
            const int kp = row0 + key_pos(it, j);
            if (elect_one()) {
              mbar_expect_tx(kv_full(st), STAGE_BYTES);
              tma_load_2d(dst, &tmap_qkv_col, kv_full(st), I + it.hh * DH, kp);
              tma_load_2d(dst + COL_TILE_BYTES, &tmap_qkv_col, kv_full(st), 2 * I + it.hh * DH, kp);
            }
            __syncwarp();
          }
        }
      }
    } else if (warp == 1) {
      {                                                       // whole warp, one elected lane issues (uniform operands)
        constexpr uint32_t idesc_s = make_idesc(RB, CT, false, false);      // S / dP [128 q x 64 keys], K = dh
        constexpr uint32_t idesc_a = make_idesc(RB, DH, false, true);       // dQ [128 q x 64 dh] += dS (TMEM, K = keys) x K_j (MN-major)
        struct Cur { int wi; uint32_t item; int t; QItem it; bool valid; };
        Cur ahead, cur;
        ahead.wi = blockIdx.x; ahead.item = 0; ahead.t = 0; ahead.valid = decode_qitem(a, ahead.wi, ahead.it);
        cur = ahead;
        auto advance = [&](Cur& c) {
          if (++c.t == c.it.nT) { c.t = 0; c.wi += gridDim.x; ++c.item; c.valid = decode_qitem(a, c.wi, c.it); }
        };
        uint32_t xa = 0;
        auto issue_ahead = [&]() {
          if (!ahead.valid) return;
          const int qb = ahead.item & 1, st = xa % NS, buf = xa % NB;
          if (ahead.t == 0) {
            // the item's Q and dO tiles go to tensor memory ONCE (tcgen05.cp, behind every MMA of the previous item): S and dP
            // then read their A operand there — an SS MMA spends ~32 cycles per K step just fetching 128 x 16 of A from
            // shared memory (ubench: 83 vs 50 cycles per 128 x 64 x 16 instruction)
            mbar_wait(qd_full(qb), (ahead.item >> 1) & 1);
            tcgen05_fence_after();
            const uint64_t qd = make_smem_desc<false>(sQD + (2 * qb) * ROW_TILE_BYTES);
            const uint64_t dod = make_smem_desc<false>(sQD + (2 * qb + 1) * ROW_TILE_BYTES);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < DH / 16; ++k) tmem_cp_128x256b(tmem_base + 448 + 8 * k, qd + 2 * k);
#pragma unroll
              for (int k = 0; k < DH / 16; ++k) tmem_cp_128x256b(tmem_base + 480 + 8 * k, dod + 2 * k);
              tcgen05_commit(qd_empty(qb));                                  // the shared-memory tiles are free once copied
            }
            __syncwarp();
          }
          mbar_wait(kv_full(st), (xa / NS) & 1);
          tcgen05_fence_after();
          const uint64_t kd = make_smem_desc<false>(sKV + st * STAGE_BYTES), vd = make_smem_desc<false>(sKV + st * STAGE_BYTES + COL_TILE_BYTES);
          const uint32_t tm = tmem_base + buf * 128;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < DH / 16; ++k) umma_bf16_ts(tm, tmem_base + 448 + 8 * k, kd + 2 * k, idesc_s, k > 0);
#pragma unroll
            for (int k = 0; k < DH / 16; ++k) umma_bf16_ts(tm + 64, tmem_base + 480 + 8 * k, vd + 2 * k, idesc_s, k > 0);
            tcgen05_commit(s_full(buf));
          }
          __syncwarp();
          advance(ahead);
          ++xa;
        };
        for (int i = 0; i < NB; ++i) issue_ahead();
        for (uint32_t x = 0; cur.valid; ++x) {
          const int st = x % NS, buf = x % NB;
          mbar_wait(p_full(buf), (x / NB) & 1);                              // dS of step x is in tensor memory
          if (cur.t == 0 && cur.item > 0) mbar_wait(acc_empty, (cur.item - 1) & 1);
          tcgen05_fence_after();
          const uint64_t kmn = make_smem_desc<true>(sKV + st * STAGE_BYTES);
          const uint32_t tm = tmem_base + buf * 128;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < CT / 16; ++k)                                // dQ += dS K_j
              umma_bf16_ts(tmem_base + 384, tm + 64 + 8 * k, kmn + (uint64_t)(k * (2048 >> 4)), idesc_a, (cur.t > 0 || k > 0) ? 1u : 0u);
            tcgen05_commit(kv_empty(st));
            if (cur.t == cur.it.nT - 1) tcgen05_commit(acc_full);
          }
          __syncwarp();
          advance(cur);
          issue_ahead();
        }
      }
    } else {
      // ------------------------------------------------------------------------------------------ row constants (warps 2, 3)
      // delta = rowsum(dO o O) (also written out for the dK/dV kernel) and lse in log2 units of the NEXT items' 128 query
      // rows, two rows per thread, published through shared memory: the element-wise groups never wait for these loads
      uint32_t item = 0;
      QItem it;
      for (int wi = blockIdx.x; decode_qitem(a, wi, it); wi += gridDim.x, ++item) {
        const int rb = item & 1;
        mbar_wait(rc_empty(rb), ((item >> 1) & 1) ^ 1);
        float* dst = rcs + rb * (2 * RB);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const int row = (warp - 2) * 64 + r * 32 + lane;
          const long long t = (long long)it.b * a.n + it.q0 + row;
          float D = 0.f;
#pragma unroll
          for (int hc = 0; hc < 4; ++hc) {
            float o[16], d[16];
            load_vec<16>(a.out + t * I + it.hh * DH + hc * 16, o);
            load_vec<16>(a.dout + t * I + it.hh * DH + hc * 16, d);
#pragma unroll
            for (int i = 0; i < 16; ++i) D = fmaf(o[i], d[i], D);
          }
          a.delta[t * a.h + it.hh] = D;
          dst[row] = -D;
          dst[RB + row] = -a.lse[t * a.h + it.hh] * LOG2E;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(rc_full(rb));
      }
    }
  } else {
    setmaxnreg_inc<216>();
    const int q = warp & 3, g = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float sc = SCALE * LOG2E;
    const float2 sc2 = make_float2(sc, sc);
    uint32_t x = 0, item = 0;
    QItem it;
    // the item's dQ is read out one own step late (see the dK/dV kernel): group g stores channels [32 g, 32 g + 32)
    bool pending = false;
    int pend_b = 0, pend_hh = 0, pend_q0 = 0;
    uint32_t pend_item = 0;
    auto epilogue = [&]() {
      mbar_wait(acc_full, pend_item & 1);
      tcgen05_fence_after();
      uint32_t r0[32];
      tmem_ld32_issue(tmem_base + lane_addr + 384 + g * 32, r0);
      tmem_ld32_wait(r0);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      float v0[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) v0[i] = __uint_as_float(r0[i]) * SCALE;
      if constexpr (TMA_ST) {
        const uint32_t slot = base + OFF_ST + g * ST_BOX_BYTES;
        unrotate32(a, pend_q0 + row, g * 32, v0);
        if (row == 0) bulk_wait_group_read<0>();                             // the previous item's box has left the slot
        group_bar(g);
        stage_row32(slot, row, v0);
        fence_proxy_async();
        group_bar(g);
        if (row == 0) {
          tma_store_2d(&tmap_dqkv_st, slot, pend_hh * DH + g * 32, pend_b * a.n + pend_q0);
          bulk_commit_group();
        }
      } else {
        const long long t = (long long)pend_b * a.n + pend_q0 + row;
        store_grad_row(a, a.dqkv + t * (3LL * I) + pend_hh * DH + g * 32, pend_q0 + row, g * 32, v0);
      }
      pending = false;
    };
    for (int wi = blockIdx.x; decode_qitem(a, wi, it); wi += gridDim.x, ++item) {
      const int qi = it.i0 + row;                                            // in-window offset of this thread's query row
      const int rb = item & 1;
      mbar_wait(rc_full(rb), (item >> 1) & 1);
      const float nD = rcs[rb * (2 * RB) + row], nL2 = rcs[rb * (2 * RB) + RB + row];
      __syncwarp();
      if (lane == 0) mbar_arrive(rc_empty(rb));
      const float2 nl2 = make_float2(nL2, nL2), nd2 = make_float2(nD, nD);
      for (int j = 0; j < it.nT; ++j, ++x) {
        if ((int)(x & 1) != g) continue;
        const uint32_t tm = tmem_base + (x % NB) * 128 + lane_addr;
        mbar_wait(s_full(x % NB), (x / NB) & 1);
        tcgen05_fence_after();
        const int c0 = (j - it.nprev) * CT;                                  // in-window offset of the tile's first key (own window)
        const bool masked = j >= it.nprev && c0 + CT - 1 > it.i0;            // own-window tiles that reach past the tile's first query
        uint32_t dk[32];
        uint32_t s[2][32], dp[2][32];
        tmem_ld32_issue(tm, s[0]);
        tmem_ld32_issue(tm + 64, dp[0]);
        tmem_ld32_issue(tm + 32, s[1]);
        tmem_ld32_issue(tm + 96, dp[1]);
        tmem_ld32_wait(s[0]);
        tmem_ld32_wait(dp[0]);
        tmem_ld32_wait(s[1]);
        tmem_ld32_wait(dp[1]);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float2 e = ffma2(make_float2(__uint_as_float(s[half][i]), __uint_as_float(s[half][i + 1])), sc2, nl2);
            e.x = ex2f(e.x);
            e.y = (POLY && (i & 2)) ? ex2_poly(e.y) : ex2f(e.y);
            if (masked) {                                                    // key after query: masked
              if (c0 + half * 32 + i > qi) e.x = 0.f;
              if (c0 + half * 32 + i + 1 > qi) e.y = 0.f;
            }
            const float2 dd = fmul2(e, fadd2(make_float2(__uint_as_float(dp[half][i]), __uint_as_float(dp[half][i + 1])), nd2));
            dk[half * 16 + i / 2] = pack_bf16x2(dd.x, dd.y);                 // dS (without the 1/sqrt(dh): applied to dQ once)
          }
        }
        tmem_st<32>(tm + 64, dk);                                            // over dP[0, 32): 64 keys as bf16 pairs
        tmem_st_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full(x % NB));
        if (pending) epilogue();                                             // the PREVIOUS item's dQ
      }
      pend_b = it.b; pend_hh = it.hh; pend_q0 = it.q0; pend_item = item; pending = true;
    }
    if (pending) epilogue();
    if (TMA_ST && row == 0) bulk_wait_group<0>();
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) { tcgen05_fence_after(); tmem_dealloc<TMEM_COLS>(tmem_base); }
}

}  // namespace

// Round-2 backward (both kernels); returns 1 when disabled so the caller falls back to the round-1 kernels.
// mode: 0 off, 1 MUFU only, 2 + FMA-pipe exp2 in dQ, 3 = 2 + gradient tiles stored through TMA (see the file header);
// -1 reads PROGEN_ATTN_BWD_TS (once per process; default 3).  Rotary tables: row-major [n, 32] (rot_sin / rot_cos) and/or
// transposed [32, n] (rot_sin_t / rot_cos_t); modes 1 and 2 read the row-major ones, mode 3 the transposed ones when given.
int attn_bwd_ts_launch(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, float* delta,
                       const float* rot_sin, const float* rot_cos, const float* rot_sin_t, const float* rot_cos_t, int B,
                       int seq_len, int window, int heads, int mode, cudaStream_t s) {
  static const int env_mode = [] { const char* e = getenv("PROGEN_ATTN_BWD_TS"); return e ? atoi(e) : 3; }();
  if (mode < 0) mode = env_mode;
  if (!mode || window % RB != 0) return 1;
  PG_CHECK_ARG(mode <= 3);
  const bool tma_st = mode == 3;
  PG_CHECK_ARG(tma_st || rot_sin || !rot_sin_t);      // modes 1 and 2 have no transposed-table path
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
  CUtensorMap tst;                                      // dqkv, 128 rows x 32 channels per box, 64-byte swizzle
  if (tma_st) {
    rc = pg_tensor_map_2d(dqkv, 2, 3ull * I, (uint64_t)T, 3ull * I, 32, RB, 64, &tst);
    if (rc) return rc;
  } else {
    tst = tq_row;                                       // not read
  }
  static bool once = false;
  if (!once) {
    PG_CUDA(cudaFuncSetAttribute(attn_bwd_dq_ts_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dq::SMEM_BYTES));
    PG_CUDA(cudaFuncSetAttribute(attn_bwd_dq_ts_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dq::SMEM_BYTES));
    PG_CUDA(cudaFuncSetAttribute(attn_bwd_dq_ts_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dq::SMEM_BYTES_ST));
    PG_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_ts_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dkv::SMEM_BYTES));
    PG_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_ts_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dkv::SMEM_BYTES_ST));
    once = true;
  }
  BwdDev a{B, seq_len, window, heads, (const bf16*)out, (const bf16*)dout, lse, delta, (bf16*)dqkv, rot_sin, rot_cos, DH / 2, 1};
  if (tma_st && rot_sin_t) { a.rot_sin = rot_sin_t; a.rot_cos = rot_cos_t; a.rot_ld_pos = 1; a.rot_ld_pair = seq_len; }
  const long long items = (long long)B * heads * (seq_len / RB);
  const int grid = (int)(items < pg_num_sms() ? items : pg_num_sms());
  if (tma_st) attn_bwd_dq_ts_kernel<true, true><<<grid, 384, dq::SMEM_BYTES_ST, s>>>(tq_row, tq_col, tdo_row, tst, a);
  else if (mode == 2) attn_bwd_dq_ts_kernel<true, false><<<grid, 384, dq::SMEM_BYTES, s>>>(tq_row, tq_col, tdo_row, tst, a);
  else attn_bwd_dq_ts_kernel<false, false><<<grid, 384, dq::SMEM_BYTES, s>>>(tq_row, tq_col, tdo_row, tst, a);
  PG_LAUNCH_CHECK();
  if (tma_st) attn_bwd_dkv_ts_kernel<true><<<grid, 384, dkv::SMEM_BYTES_ST, s>>>(tq_row, tq_col, tdo_col, tst, a);
  else attn_bwd_dkv_ts_kernel<false><<<grid, 384, dkv::SMEM_BYTES, s>>>(tq_row, tq_col, tdo_col, tst, a);
  PG_LAUNCH_CHECK();
  return PROGEN_OK;
}
