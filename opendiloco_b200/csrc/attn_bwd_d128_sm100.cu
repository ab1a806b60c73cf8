// Causal flash-attention BACKWARD for head_dim 128 on tcgen05 / TMEM / TMA (sm_100a), bf16, MHA + GQA.
//
// The fused head_dim-64 kernel (attn_bwd_sm100.cu) keeps S^T, dP^T, dV, dK and dQ in tensor memory: at D = 128 that is
// 640 columns against 512.  The backward is therefore split into two kernels that each fit:
//
//   dK / dV kernel (key-stationary, the head_dim-64 design without its dQ role): one CTA per (batch, kv-head, pair of
//     128-key tiles {x, nq-1-x}), walking the query heads of its GQA group and the query tiles kb .. nq-1 (MASKED:
//     kb .. q_hi[b, kb]).  Per query tile
//       S^T  = K  Q^T    A = K  (smem, K-major)   B = Q  (smem, K-major)   N = 128, K = 128 (8 steps over two boxes)
//       dP^T = V  dO^T   A = V  (smem, K-major)   B = dO (smem, K-major)
//       dV  += P^T  dO   A = P^T  (TMEM, bf16)    B = dO (smem, MN-major, the two 64-column boxes one LBO apart)
//       dK  += dS^T Q    A = dS^T (TMEM, bf16)    B = Q  (smem, MN-major)
//     TMEM: S^T [0,128)  dP^T -> P^T | dS^T [128,256)  dV [256,384)  dK [384,512).  Shared memory: K, V and two stages of
//     (Q, dO) = 192 KB.  dK / dV leave through registers (bf16, RoPE transpose applied to dK on the way).
//
//   dQ kernel (query-stationary, laid out like the forward): one CTA per (batch, q-head, pair of 128-query tiles), walking
//     key tiles 0 .. qt (MASKED: kv_lo[b, qt] .. qt).  Per key tile
//       S  = Q K^T , dP = dO V^T                  (SS, N = 128)
//       P  = exp2(S*c - lse2), dS = P (dP - D) scale, written back as bf16 into this thread's own dP columns
//       dQ += dS K                                (TS: A = dS from TMEM, B = K read MN-major)
//     TMEM: S [0,128)  dP -> dS [128,256)  dQ [256,384).  Shared memory: Q, dO and two stages of (K, V) = 192 KB.  dQ is
//     written once, as bf16 (RoPE transpose on the way): no fp32 accumulator and no reduce-adds, so the whole D = 128
//     backward is bitwise deterministic.
//
// Both kernels: warp 0 TMA, warp 1 MMA, 8 element-wise warps with two threads per TMEM lane (64 score columns each).
// The pre-pass writes the per-query statistics block (-lse*log2(e), -D*scale, and lo when MASKED) of the head_dim-64
// kernel.  MASKED: allowed(s, t) = t == s || (lo[s] <= t < s && valid[t]), see odb_attn_mask_prep in attn_sm100.cu.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "packed_math.cuh"

using namespace odb;
using namespace sm100;
using namespace packed_math;

namespace attn_bwd128 {

constexpr int BQ = 128, BKV = 128, D = 128;
constexpr int BOX = 128 * 128;                   // bytes of a [128 x 64] bf16 box (128-byte swizzled rows)
constexpr int OP = 2 * BOX;                      // a [128 x 128] bf16 operand = two boxes
constexpr int BOX16 = BOX >> 4;                  // one box in descriptor units (16 bytes)
constexpr int EW_WARP0 = 2, EW_WARPS = 8;
constexpr int THREADS = 32 * (EW_WARP0 + EW_WARPS);
constexpr int QST = 2;                           // dK/dV kernel: (Q, dO, stats) stages - three do not fit
constexpr int STAT_BYTES = 2 * 128 * 4, MASKED_STAT_BYTES = 3 * 128 * 4;
template <bool MASKED> struct DkvCfg {
  static constexpr int SB = MASKED ? MASKED_STAT_BYTES : STAT_BYTES;
  static constexpr int SMEM_BYTES = 2 * OP + 2 * QST * OP + QST * SB + 256 + 1024;
};
constexpr int DQ_SMEM_BYTES = 2 * OP + 2 * 2 * OP + 256 + 1024;
constexpr uint32_t TMEM_COLS = 512;

struct Params {
  int B, S, Hq, Hkv;
  float scale, scale_log2;
  const float* stats;      // [B, Hq, S/128, 2 or 3, 128] written by the pre-pass
  const float* cos_t;      // [S, 64] RoPE tables (nullptr: no rotation)
  const float* sin_t;
  __nv_bfloat16* dq;       // row stride ld_dq
  __nv_bfloat16* dk;       // dk / dv row stride ld_dkv
  __nv_bfloat16* dv;
  long long ld_dq, ld_dkv;
  // MASKED only (odb_attn_mask_prep outputs)
  const int* lo;           // [B*S]
  const uint32_t* vbits;   // [B, S/32]
  const int* kv_lo;        // [B, S/128]
  const int* q_hi;         // [B, S/128]
  const int* lo_hi;        // [B, S/128]
};

__device__ __forceinline__ void lds_2x64(uint32_t addr, uint64_t& a, uint64_t& b) {
  asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}
__device__ __forceinline__ uint32_t mul_bf16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}

// One thread's share of a [128 x 128] fp32 accumulator row: columns [32*part, +32) and [64 + 32*part, +32), i.e. both
// members of 32 rotation pairs (j, j+64).  Optionally rotated by -theta (the transpose of the forward RoPE), then stored
// as bf16 into dst (the row's 128 columns).
__device__ __forceinline__ void store_row_pairs(uint32_t taddr, int part, __nv_bfloat16* dst, const float* cos_row,
                                                const float* sin_row) {
  uint32_t a[32], b[32];
  tmem_ld_32x32b_x32(taddr + 32 * part, a);
  tmem_ld_32x32b_x32(taddr + 64 + 32 * part, b);
  tmem_ld_wait();
  if (cos_row != nullptr) {
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 c = ld_f4(cos_row + 32 * part + i), s = ld_f4(sin_row + 32 * part + i);
      const float cs[4] = {c.x, c.y, c.z, c.w}, sn[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float x = __uint_as_float(a[i + u]), y = __uint_as_float(b[i + u]);
        a[i + u] = __float_as_uint(x * cs[u] + y * sn[u]);
        b[i + u] = __float_as_uint(y * cs[u] - x * sn[u]);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    float f[8], g[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { f[i] = __uint_as_float(a[u * 8 + i]); g[i] = __uint_as_float(b[u * 8 + i]); }
    st_v4(dst + 32 * part + 8 * u, pack8(f));
    st_v4(dst + 64 + 32 * part + 8 * u, pack8(g));
  }
}

// ===================================================================================================== dK / dV
template <bool MASKED>
__global__ void __launch_bounds__(THREADS, 1)
attn_bwd_dkv_d128_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_do, Params p) {
  constexpr int SB = DkvCfg<MASKED>::SB, SF = SB / 4;
  constexpr int NQ = 64;                         // queries (score columns) per element-wise thread
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = sK + OP;
  uint8_t* sQ = sV + OP;                   // QST stages
  uint8_t* sdO = sQ + QST * OP;            // QST stages
  float* sStat = reinterpret_cast<float*>(sdO + QST * OP);
  uint64_t* kv_full = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sStat) + QST * SB);
  uint64_t* kv_empty = kv_full + 1;
  uint64_t* q_full = kv_empty + 1;         // [QST]
  uint64_t* q_empty = q_full + QST;        // [QST]
  uint64_t* s_full = q_empty + QST;        // S^T ready
  uint64_t* dp_full = s_full + 1;          // dP^T ready (and every earlier MMA retired)
  uint64_t* s_free = dp_full + 1;          // S^T in registers (8 warps)
  uint64_t* pds_full = s_free + 1;         // P^T / dS^T in tensor memory (8 warps)
  uint64_t* mma_done = pds_full + 1;       // dV / dK MMAs of this iteration retired
  uint64_t* dkv_empty = mma_done + 1;      // dK / dV accumulators read by the epilogue (8 warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dkv_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = p.S / BQ;
  pdl_launch_dependents();
  const int kb_first = (int)blockIdx.x, kb_second = nq - 1 - (int)blockIdx.x;
  const int nitems = kb_first != kb_second ? 2 : 1;
  const int hk = blockIdx.y, b = blockIdx.z;
  const int group = p.Hq / p.Hkv;
  const int col_k = (p.Hq + hk) * D, col_v = (p.Hq + p.Hkv + hk) * D;
  auto q_end = [&](int kb) { return MASKED ? p.q_hi[b * nq + kb] + 1 : nq; };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    mbar_init(kv_full, 1);
    mbar_init(kv_empty, 1);
    for (int i = 0; i < QST; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
    mbar_init(s_full, 1);
    mbar_init(dp_full, 1);
    mbar_init(s_free, EW_WARPS);
    mbar_init(pds_full, EW_WARPS);
    mbar_init(mma_done, 1);
    mbar_init(dkv_empty, EW_WARPS);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tb = *tmem_slot;
  const uint32_t tS = tb, tdP = tb + 128, tdV = tb + 256, tdK = tb + 384;
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      int st = 0, ph = 0;
      for (int w = 0; w < nitems; ++w) {
        const int kb = w ? kb_second : kb_first;
        mbar_wait(kv_empty, (w & 1) ^ 1);
        mbar_arrive_expect_tx(kv_full, 2 * OP);
        for (int c = 0; c < 2; ++c) {
          tma_load_2d(sK + c * BOX, &tmap_qkv, kv_full, col_k + 64 * c, b * p.S + kb * BKV);
          tma_load_2d(sV + c * BOX, &tmap_qkv, kv_full, col_v + 64 * c, b * p.S + kb * BKV);
        }
        for (int hh = 0; hh < group; ++hh) {
          const int h = hk * group + hh;
          for (int qi = kb, qe = q_end(kb); qi < qe; ++qi) {
            mbar_wait(&q_empty[st], ph ^ 1);
            mbar_arrive_expect_tx(&q_full[st], 2 * OP + SB);
            for (int c = 0; c < 2; ++c) {
              tma_load_2d(sQ + st * OP + c * BOX, &tmap_qkv, &q_full[st], h * D + 64 * c, b * p.S + qi * BQ);
              tma_load_2d(sdO + st * OP + c * BOX, &tmap_do, &q_full[st], h * D + 64 * c, b * p.S + qi * BQ);
            }
            bulk_load_1d(sStat + st * SF, p.stats + (((size_t)b * p.Hq + h) * nq + qi) * SF, SB, &q_full[st]);
            if (++st == QST) { st = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t id_s = make_idesc_bf16(128, 128, 0, 0);     // S^T, dP^T
    constexpr uint32_t id_ts = make_idesc_bf16(128, 128, 0, 1);    // dV, dK: A from tensor memory, B MN-major
    const bool leader = elect_one();
    const uint64_t kd = make_smem_desc_sw128(smem_u32(sK), 16, 1024);
    const uint64_t vd = make_smem_desc_sw128(smem_u32(sV), 16, 1024);
    int st = 0, ph = 0;                                  // stage / phase of the NEXT S^T to issue
    // 8 K16 steps over the head dimension: steps 0-3 in the first 64-column box, 4-7 in the second
    auto kstep = [](int k) { return (uint32_t)((k >> 2) * BOX16 + 2 * (k & 3)); };
    auto issue_s = [&]() {
      const uint64_t qd = make_smem_desc_sw128(smem_u32(sQ + st * OP), 16, 1024);
      mbar_wait(&q_full[st], ph);
      tc_fence_after_sync();
      if (leader) {
#pragma unroll
        for (int k = 0; k < 8; ++k) umma_ss(tS, kd + kstep(k), qd + kstep(k), id_s, k > 0);
        umma_commit(s_full);
      }
      __syncwarp();
    };
    auto issue_dp = [&](int stg) {
      const uint64_t dod = make_smem_desc_sw128(smem_u32(sdO + stg * OP), 16, 1024);
      if (leader) {
#pragma unroll
        for (int k = 0; k < 8; ++k) umma_ss(tdP, vd + kstep(k), dod + kstep(k), id_s, k > 0);
        umma_commit(dp_full);
      }
      __syncwarp();
    };
    for (int w = 0, g = 0; w < nitems; ++w) {
      const int kb = w ? kb_second : kb_first;
      const int iters = group * (q_end(kb) - kb);
      mbar_wait(kv_full, w & 1);
      if (g > 0) mbar_wait(s_free, (g - 1) & 1);       // the previous key tile's last S^T has been read
      issue_s();
      int cur = st;
      issue_dp(cur);
      if (++st == QST) { st = 0; ph ^= 1; }
      for (int i = 0; i < iters; ++i) {
        const int it = g + i;
        // MN-major B operands: N = 128 head columns = two 64-element chunks one box (LBO) apart; 16 queries per K step
        const uint64_t qmn = make_smem_desc_sw128(smem_u32(sQ + cur * OP), BOX, 1024);
        const uint64_t domn = make_smem_desc_sw128(smem_u32(sdO + cur * OP), BOX, 1024);
        const int nxt = st;
        if (i + 1 < iters) {
          mbar_wait(s_free, it & 1);
          issue_s();
          if (++st == QST) { st = 0; ph ^= 1; }
        }
        mbar_wait(pds_full, it & 1);                   // P^T, dS^T in tensor memory
        if (i == 0 && w > 0) mbar_wait(dkv_empty, (w - 1) & 1);   // the epilogue read the previous key tile's dK / dV
        tc_fence_after_sync();
        const bool first = (i == 0);
        if (leader) {
          // each element-wise thread's 64 dP^T columns now hold P^T (first 32) and dS^T (last 32) of its 64 queries
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_ts(tdV, tdP + (16 * k / NQ) * NQ + (16 * k % NQ) / 2, domn + 128 * k, id_ts, (first && k == 0) ? 0u : 1u);
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_ts(tdK, tdP + (16 * k / NQ) * NQ + NQ / 2 + (16 * k % NQ) / 2, qmn + 128 * k, id_ts, (first && k == 0) ? 0u : 1u);
          umma_commit(&q_empty[cur]);
          umma_commit(mma_done);
          if (i + 1 == iters) umma_commit(kv_empty);
        }
        __syncwarp();
        // dP^T(it+1) overwrites the columns dV / dK(it) read P^T / dS^T from: the tensor pipe executes in issue order
        if (i + 1 < iters) issue_dp(nxt);
        cur = nxt;
      }
      g += iters;
    }
  } else {
    // ------------------------------------------------------------------ element-wise warps (two threads per KEY row)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int part = (warp - EW_WARP0) >> 2;             // queries [64*part, 64*part + 64) of the query tile
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const float c = p.scale_log2;
    const uint64_t c2 = pack2(c, c), sc2 = pack2(p.scale, p.scale);
    const uint32_t tPD = tdP + lane_off + part * NQ;
    int st = 0, ph = 0;
    for (int w = 0, it = 0; w < nitems; ++w) {
      const int kb = w ? kb_second : kb_first;
      const int key = kb * BKV + row;
      const bool key_valid = MASKED ? (p.vbits[(size_t)b * (p.S / 32) + key / 32] >> (key & 31)) & 1u : true;
      for (int hh = 0; hh < group; ++hh) {
        for (int qi = kb, qe = q_end(kb); qi < qe; ++qi, ++it) {
          const bool diag = (qi == kb);
          const uint32_t stat = smem_u32(sStat + st * SF + part * NQ);
          mbar_wait(&q_full[st], ph);
          mbar_wait(s_full, it & 1);
          tc_fence_after_sync();
          uint32_t pp[NQ / 2];
          {
            uint32_t sr[NQ];
            tmem_ld_32x32b_x32(tS + lane_off + part * NQ, *reinterpret_cast<uint32_t(*)[32]>(&sr[0]));
            tmem_ld_32x32b_x32(tS + lane_off + part * NQ + 32, *reinterpret_cast<uint32_t(*)[32]>(&sr[32]));
            tmem_ld_wait();
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(s_free);
            if constexpr (MASKED) {
              const bool need = diag || !key_valid || key < p.lo_hi[b * nq + qi];
              if (__any_sync(0xffffffffu, need)) {
                const int rel = key - (qi * BQ + part * NQ);
                const int* lo_s = reinterpret_cast<const int*>(sStat + st * SF + 256 + part * NQ);
#pragma unroll
                for (int i = 0; i < NQ; i += 4) {
                  const int4 l4 = *reinterpret_cast<const int4*>(lo_s + i);
                  const int lv[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
                  for (int u = 0; u < 4; ++u)
                    if (!(i + u >= rel && key >= lv[u] && (key_valid || i + u == rel))) sr[i + u] = 0xff800000u;
                }
              }
            } else if (diag) {
#pragma unroll
              for (int i = 0; i < NQ; ++i)
                if (row > part * NQ + i) sr[i] = 0xff800000u;
            }
#pragma unroll
            for (int i = 0; i < NQ; i += 4) {
              uint64_t nla, nlb;
              lds_2x64(stat + i * 4, nla, nlb);
              const uint64_t ya = ffma2(pack2u(sr[i], sr[i + 1]), c2, nla);
              const uint64_t yb = ffma2(pack2u(sr[i + 2], sr[i + 3]), c2, nlb);
              float a0, a1;
              unpack2(ya, a0, a1);
              pp[i / 2] = cvt_bf16x2(pack2(fast_exp2(a0), fast_exp2(a1)));
              pp[i / 2 + 1] = cvt_bf16x2(poly_exp2x2(yb));
            }
          }
          mbar_wait(dp_full, it & 1);
          if (it > 0) mbar_wait(mma_done, (it - 1) & 1);   // (implied by dp_full; keeps this barrier's phases in step)
          tc_fence_after_sync();
          uint32_t ds[NQ / 2];
          {
            uint32_t dr[NQ];
            tmem_ld_32x32b_x32(tPD, *reinterpret_cast<uint32_t(*)[32]>(&dr[0]));
            tmem_ld_32x32b_x32(tPD + 32, *reinterpret_cast<uint32_t(*)[32]>(&dr[32]));
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < NQ; i += 4) {
              uint64_t nda, ndb;
              lds_2x64(stat + 512 + i * 4, nda, ndb);
              ds[i / 2] = mul_bf16x2(pp[i / 2], cvt_bf16x2(ffma2(pack2u(dr[i], dr[i + 1]), sc2, nda)));
              ds[i / 2 + 1] = mul_bf16x2(pp[i / 2 + 1], cvt_bf16x2(ffma2(pack2u(dr[i + 2], dr[i + 3]), sc2, ndb)));
            }
          }
          tmem_st_32x32b_x32(tPD, pp);
          tmem_st_32x32b_x32(tPD + NQ / 2, ds);
          tmem_st_wait();
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(pds_full);
          if (++st == QST) { st = 0; ph ^= 1; }
        }
      }
      // ---- dK / dV of this key tile: this thread's 64 columns -> bf16 -> global (dK rotated back by -theta)
      mbar_wait(mma_done, (it - 1) & 1);
      tc_fence_after_sync();
      const long long t = (long long)b * p.S + key;
      const float* cr = p.cos_t != nullptr ? p.cos_t + (size_t)key * 64 : nullptr;
      const float* sr = p.sin_t != nullptr ? p.sin_t + (size_t)key * 64 : nullptr;
      store_row_pairs(tdK + lane_off, part, p.dk + t * p.ld_dkv + hk * D, cr, sr);
      {
        uint32_t a[32], bb[32];
        tmem_ld_32x32b_x32(tdV + lane_off + 32 * part, a);
        tmem_ld_32x32b_x32(tdV + lane_off + 64 + 32 * part, bb);
        tmem_ld_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(dkv_empty);         // the next key tile may start accumulating
        __nv_bfloat16* dst = p.dv + t * p.ld_dkv + hk * D;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float f[8], g[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) { f[i] = __uint_as_float(a[u * 8 + i]); g[i] = __uint_as_float(bb[u * 8 + i]); }
          st_v4(dst + 32 * part + 8 * u, pack8(f));
          st_v4(dst + 64 + 32 * part + 8 * u, pack8(g));
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tb, TMEM_COLS);
}

// ===================================================================================================== dQ
template <bool MASKED>
__global__ void __launch_bounds__(THREADS, 1)
attn_bwd_dq_d128_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_do, Params p) {
  constexpr int SR = MASKED ? 3 : 2;             // rows of a statistics block
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sdO = sQ + OP;
  uint8_t* sK = sdO + OP;                        // 2 stages
  uint8_t* sV = sK + 2 * OP;                     // 2 stages
  uint64_t* q_full = reinterpret_cast<uint64_t*>(sV + 2 * OP);
  uint64_t* q_empty = q_full + 1;                // every MMA of the current query tile retired: Q / dO may be replaced
  uint64_t* kv_full = q_empty + 1;               // [2]
  uint64_t* kv_empty = kv_full + 2;              // [2]
  uint64_t* s_full = kv_empty + 2;
  uint64_t* dp_full = s_full + 1;
  uint64_t* s_free = dp_full + 1;                // S in registers (8 warps)
  uint64_t* ds_full = s_free + 1;                // dS in tensor memory (8 warps)
  uint64_t* dq_full = ds_full + 1;               // the query tile's last dQ MMA retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dq_full + 1);

  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = p.S / BQ;
  const int qb[2] = {nq - 1 - (int)blockIdx.x, (int)blockIdx.x};   // balanced pair, as in the forward
  const int nitems = qb[0] != qb[1] ? 2 : 1;
  const int h = blockIdx.y, b = blockIdx.z;
  const int hk = h / (p.Hq / p.Hkv);
  const int col_q = h * D, col_k = (p.Hq + hk) * D, col_v = (p.Hq + p.Hkv + hk) * D;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
    mbar_init(s_full, 1);
    mbar_init(dp_full, 1);
    mbar_init(s_free, EW_WARPS);
    mbar_init(ds_full, EW_WARPS);
    mbar_init(dq_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tb = *tmem_slot;
  const uint32_t tS = tb, tdP = tb + 128, tdQ = tb + 256;
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      for (int w = 0, t0 = 0; w < nitems; ++w) {
        const int j0 = MASKED ? p.kv_lo[b * nq + qb[w]] : 0;
        const int nkv = qb[w] + 1 - j0;
        mbar_wait(q_empty, (w & 1) ^ 1);
        mbar_arrive_expect_tx(q_full, 2 * OP);
        for (int c = 0; c < 2; ++c) {
          tma_load_2d(sQ + c * BOX, &tmap_qkv, q_full, col_q + 64 * c, b * p.S + qb[w] * BQ);
          tma_load_2d(sdO + c * BOX, &tmap_do, q_full, col_q + 64 * c, b * p.S + qb[w] * BQ);
        }
        for (int j = 0; j < nkv; ++j) {
          const int tg = t0 + j, st = tg & 1;
          mbar_wait(&kv_empty[st], ((tg >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(&kv_full[st], 2 * OP);
          for (int c = 0; c < 2; ++c) {
            tma_load_2d(sK + st * OP + c * BOX, &tmap_qkv, &kv_full[st], col_k + 64 * c, b * p.S + (j0 + j) * BKV);
            tma_load_2d(sV + st * OP + c * BOX, &tmap_qkv, &kv_full[st], col_v + 64 * c, b * p.S + (j0 + j) * BKV);
          }
        }
        t0 += nkv;
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t id_s = make_idesc_bf16(128, 128, 0, 0);     // S, dP: both operands K-major
    constexpr uint32_t id_dq = make_idesc_bf16(128, 128, 0, 1);    // dQ: A = dS from TMEM, B = K MN-major
    const bool leader = elect_one();
    const uint64_t qd = make_smem_desc_sw128(smem_u32(sQ), 16, 1024);
    const uint64_t dod = make_smem_desc_sw128(smem_u32(sdO), 16, 1024);
    auto kstep = [](int k) { return (uint32_t)((k >> 2) * BOX16 + 2 * (k & 3)); };
    // S(tg) and dP(tg); S is committed on its own so the element-wise warps start the exponentials while dP runs
    auto issue_s = [&](int tg) {
      const int st = tg & 1;
      mbar_wait(&kv_full[st], (tg >> 1) & 1);
      tc_fence_after_sync();
      if (leader) {
        const uint64_t kd = make_smem_desc_sw128(smem_u32(sK + st * OP), 16, 1024);
#pragma unroll
        for (int k = 0; k < 8; ++k) umma_ss(tS, qd + kstep(k), kd + kstep(k), id_s, k > 0);
        umma_commit(s_full);
      }
      __syncwarp();
    };
    auto issue_dp = [&](int tg) {
      const int st = tg & 1;
      if (leader) {
        const uint64_t vd = make_smem_desc_sw128(smem_u32(sV + st * OP), 16, 1024);
#pragma unroll
        for (int k = 0; k < 8; ++k) umma_ss(tdP, dod + kstep(k), vd + kstep(k), id_s, k > 0);
        umma_commit(dp_full);
      }
      __syncwarp();
    };
    for (int w = 0, t0 = 0; w < nitems; ++w) {
      const int nkv = qb[w] + 1 - (MASKED ? p.kv_lo[b * nq + qb[w]] : 0);
      mbar_wait(q_full, w & 1);
      if (w > 0) mbar_wait(s_free, (t0 - 1) & 1);  // the previous query tile's last S has been read
      issue_s(t0);
      issue_dp(t0);                              // after the previous tile's last dQ MMA in issue order
      for (int j = 0; j < nkv; ++j) {
        const int tg = t0 + j, st = tg & 1;
        if (j + 1 < nkv) {
          mbar_wait(s_free, tg & 1);             // S(tg) is in registers: S(tg+1) may overwrite its columns
          issue_s(tg + 1);
        }
        mbar_wait(ds_full, tg & 1);
        tc_fence_after_sync();
        if (leader) {
          // A = dS from tensor memory: thread part x keeps keys [64x, 64x+64) as 32 packed columns at tdP + 64x;
          // B = K_tg read MN-major (its two 64-column boxes one LBO apart), 16 keys per K step
          const uint64_t kmn = make_smem_desc_sw128(smem_u32(sK + st * OP), BOX, 1024);
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_ts(tdQ, tdP + 64 * (k >> 2) + 8 * (k & 3), kmn + 128 * k, id_dq, (j > 0 || k > 0) ? 1u : 0u);
          umma_commit(&kv_empty[st]);
          if (j + 1 == nkv) {
            umma_commit(q_empty);
            umma_commit(dq_full);
          }
        }
        __syncwarp();
        if (j + 1 < nkv) issue_dp(tg + 1);       // overwrites the dS(tg) columns after dQ(tg) read them (issue order)
      }
      t0 += nkv;
    }
  } else {
    // ------------------------------------------------------------------ element-wise warps (two threads per QUERY row)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int half = (warp - EW_WARP0) >> 2;     // keys [64*half, 64*half + 64) of every tile
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const float c = p.scale_log2;
    const uint64_t c2 = pack2(c, c), sc2 = pack2(p.scale, p.scale);
    for (int w = 0, t0 = 0; w < nitems; ++w) {
      const int qblk = qb[w];
      const int j0 = MASKED ? p.kv_lo[b * nq + qblk] : 0;
      const int nkv = qblk + 1 - j0;
      const int qpos = qblk * BQ + row;
      const int lo_q = MASKED ? p.lo[b * p.S + qpos] : 0;
      const float* stb = p.stats + (((size_t)b * p.Hq + h) * nq + qblk) * SR * 128 + row;
      const float nl = stb[0], nd = stb[128];    // -lse * log2(e), -D * scale of this query
      const uint64_t nl2 = pack2(nl, nl), nd2 = pack2(nd, nd);
      for (int j = 0; j < nkv; ++j) {
        const int tg = t0 + j;
        mbar_wait(s_full, tg & 1);
        tc_fence_after_sync();
        uint32_t pp[32];
        {
          uint32_t sr[64];
          tmem_ld_32x32b_x32(tS + lane_off + half * 64, *reinterpret_cast<uint32_t(*)[32]>(&sr[0]));
          tmem_ld_32x32b_x32(tS + lane_off + half * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&sr[32]));
          tmem_ld_wait();
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(s_free);
          if constexpr (MASKED) {
            const int kbase = (j0 + j) * BKV + half * 64;
            const uint32_t* vw = p.vbits + (size_t)b * (p.S / 32) + kbase / 32;
            const uint32_t w0 = vw[0], w1 = vw[1];
            const bool need = kbase + 63 > qpos || lo_q > kbase || (w0 & w1) != 0xffffffffu;
            if (__any_sync(0xffffffffu, need)) {
              const int rel_hi = qpos - kbase, rel_lo = lo_q - kbase;
#pragma unroll
              for (int i = 0; i < 64; ++i) {
                const uint32_t bit = ((i < 32 ? w0 : w1) >> (i & 31)) & 1u;
                if (!(i <= rel_hi && i >= rel_lo && (bit || i == rel_hi))) sr[i] = 0xff800000u;
              }
            }
          } else if (j0 + j == qblk) {
#pragma unroll
            for (int i = 0; i < 64; ++i)
              if (half * 64 + i > row) sr[i] = 0xff800000u;
          }
#pragma unroll
          for (int i = 0; i < 64; i += 4) {
            const uint64_t ya = ffma2(pack2u(sr[i], sr[i + 1]), c2, nl2);
            const uint64_t yb = ffma2(pack2u(sr[i + 2], sr[i + 3]), c2, nl2);
            float a0, a1;
            unpack2(ya, a0, a1);
            pp[i / 2] = cvt_bf16x2(pack2(fast_exp2(a0), fast_exp2(a1)));
            pp[i / 2 + 1] = cvt_bf16x2(poly_exp2x2(yb));
          }
        }
        mbar_wait(dp_full, tg & 1);
        tc_fence_after_sync();
        uint32_t ds[32];
        {
          uint32_t dr[64];
          tmem_ld_32x32b_x32(tdP + lane_off + half * 64, *reinterpret_cast<uint32_t(*)[32]>(&dr[0]));
          tmem_ld_32x32b_x32(tdP + lane_off + half * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&dr[32]));
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 64; i += 4) {
            ds[i / 2] = mul_bf16x2(pp[i / 2], cvt_bf16x2(ffma2(pack2u(dr[i], dr[i + 1]), sc2, nd2)));
            ds[i / 2 + 1] = mul_bf16x2(pp[i / 2 + 1], cvt_bf16x2(ffma2(pack2u(dr[i + 2], dr[i + 3]), sc2, nd2)));
          }
        }
        tmem_st_32x32b_x32(tdP + lane_off + half * 64, ds);
        tmem_st_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(ds_full);
      }
      t0 += nkv;
      // ---- epilogue: dQ (scale already in dS) -> RoPE transpose -> bf16 -> global
      mbar_wait(dq_full, w & 1);
      tc_fence_after_sync();
      const float* cr = p.cos_t != nullptr ? p.cos_t + (size_t)qpos * 64 : nullptr;
      const float* sn = p.sin_t != nullptr ? p.sin_t + (size_t)qpos * 64 : nullptr;
      store_row_pairs(tdQ + lane_off, half, p.dq + ((long long)b * p.S + qpos) * p.ld_dq + h * D, cr, sn);
      tc_fence_before_sync();                    // the next tile's first dQ MMA (ordered behind ds_full) overwrites it
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tb, TMEM_COLS);
}

// Pre-pass: per (token, head) D = sum_d dO * O over 128 columns, stored with the forward's log-sum-exp in the statistics
// layout of the head_dim-64 kernel: stats[b, h, s/128, 0, s%128] = -lse * log2(e), [..., 1, ...] = -D * scale, and
// (MASKED) [..., 2, ...] = lo[s].  Sixteen lanes per (token, head), 16 bytes of dO and O each.
template <bool MASKED>
__global__ void __launch_bounds__(256) attn_dsum_d128_kernel(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ out,
                                                             const float* __restrict__ lse, float* __restrict__ stats, int B, int S,
                                                             int Hq, long long ld, float scale, const int* __restrict__ lo) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)B * S * Hq * 16;
  if (i >= total) return;                                // total is a multiple of 16: whole lane groups leave together
  const int sub = (int)(i & 15);
  const long long w = i >> 4;
  const long long t = w / Hq;
  const int h = (int)(w % Hq);
  float a[8], o[8];
  unpack8(ld_v4(dout + t * ld + h * D + sub * 8), a);
  unpack8(ld_v4(out + t * ld + h * D + sub * 8), o);
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s = fmaf(a[j], o[j], s);
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  s += __shfl_xor_sync(0xffffffffu, s, 8);
  if (sub == 0) {
    const long long bb = t / S, ss = t % S;
    float* dst = stats + (((bb * Hq + h) * (S / 128) + ss / 128) * (MASKED ? 3 : 2)) * 128 + (ss % 128);
    dst[0] = -lse[(bb * Hq + h) * S + ss] * 1.4426950408889634f;
    dst[128] = -s * scale;
    if (MASKED) dst[256] = __int_as_float(lo[t]);
  }
}

}  // namespace attn_bwd128

namespace {
template <bool MASKED>
int launch_attn_bwd_d128(const void* qkv, const void* out, const void* dout, const void* lse, void* stats, void* dq, void* dk,
                         void* dv, const void* cos_t, const void* sin_t, int B, int S, int Hq, int Hkv, long long ld_qkv,
                         long long ld_out, long long ld_dq, long long ld_dkv, float softmax_scale, const int* lo,
                         const uint32_t* vbits, const int* kv_lo, const int* q_hi, const int* lo_hi, cudaStream_t st) {
  using namespace attn_bwd128;
  if (S % BQ || Hq % Hkv || ld_qkv % 8 || ld_out % 8 || ld_dq % 8 || ld_dkv % 8) return -1;
  const long long T = (long long)B * S;
  {
    const long long threads = T * Hq * 16;
    launch_pdl(attn_dsum_d128_kernel<MASKED>, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, st,
               (const __nv_bfloat16*)dout, (const __nv_bfloat16*)out, (const float*)lse, (float*)stats, B, S, Hq, ld_out,
               softmax_scale, lo);
  }
  CUtensorMap tq, tdo;
  int rc;
  if ((rc = make_tmap_2d(&tq, qkv, T, (Hq + 2 * Hkv) * D, ld_qkv * 2, 128, 64, 2))) return rc;
  if ((rc = make_tmap_2d(&tdo, dout, T, Hq * D, ld_out * 2, 128, 64, 2))) return rc;
  Params p{};
  p.B = B; p.S = S; p.Hq = Hq; p.Hkv = Hkv;
  p.scale = softmax_scale;
  p.scale_log2 = softmax_scale * 1.4426950408889634f;
  p.stats = (const float*)stats;
  p.cos_t = (const float*)cos_t; p.sin_t = (const float*)sin_t;
  p.dq = (__nv_bfloat16*)dq; p.dk = (__nv_bfloat16*)dk; p.dv = (__nv_bfloat16*)dv;
  p.ld_dq = ld_dq; p.ld_dkv = ld_dkv;
  p.lo = lo; p.vbits = vbits; p.kv_lo = kv_lo; p.q_hi = q_hi; p.lo_hi = lo_hi;
  constexpr int DKV_SMEM = DkvCfg<MASKED>::SMEM_BYTES;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_bwd_dkv_d128_kernel<MASKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, DKV_SMEM);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_bwd_dq_d128_kernel<MASKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, DQ_SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const dim3 grid_kv((S / BKV + 1) / 2, Hkv, B), grid_q((S / BQ + 1) / 2, Hq, B);
  launch_pdl(attn_bwd_dkv_d128_kernel<MASKED>, grid_kv, dim3(THREADS), DKV_SMEM, st, tq, tdo, p);
  launch_pdl(attn_bwd_dq_d128_kernel<MASKED>, grid_q, dim3(THREADS), DQ_SMEM_BYTES, st, tq, tdo, p);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}
}  // namespace

// Head size 128.  stats: fp32 scratch of 2 * B * Hq * S elements (3 * ... for the masked entry point); no dQ accumulator.
// dq, dk, dv: bf16 outputs with row strides ld_dq / ld_dkv elements, e.g. the three column blocks of one packed
// [T, (Hq+2*Hkv)*128] buffer.  With cos/sin (fp32 [S, 64] tables) dq and dk leave with the RoPE rotation undone.
ODB_EXPORT int odb_attn_bwd_d128(const void* qkv, const void* out, const void* dout, const void* lse, void* stats, void* dq,
                                 void* dk, void* dv, const void* cos_t, const void* sin_t, int B, int S, int Hq, int Hkv,
                                 long long ld_qkv, long long ld_out, long long ld_dq, long long ld_dkv, float softmax_scale,
                                 cudaStream_t st) {
  return launch_attn_bwd_d128<false>(qkv, out, dout, lse, stats, dq, dk, dv, cos_t, sin_t, B, S, Hq, Hkv, ld_qkv, ld_out, ld_dq,
                                     ld_dkv, softmax_scale, nullptr, nullptr, nullptr, nullptr, nullptr, st);
}

// Same with a mask description (lo, vbits, kv_lo, q_hi, lo_hi from odb_attn_mask_prep).
ODB_EXPORT int odb_attn_bwd_d128_masked(const void* qkv, const void* out, const void* dout, const void* lse, void* stats, void* dq,
                                        void* dk, void* dv, const void* cos_t, const void* sin_t, int B, int S, int Hq, int Hkv,
                                        long long ld_qkv, long long ld_out, long long ld_dq, long long ld_dkv,
                                        float softmax_scale, const void* lo, const void* vbits, const void* kv_lo,
                                        const void* q_hi, const void* lo_hi, cudaStream_t st) {
  if (!lo || !vbits || !kv_lo || !q_hi || !lo_hi) return -1;
  return launch_attn_bwd_d128<true>(qkv, out, dout, lse, stats, dq, dk, dv, cos_t, sin_t, B, S, Hq, Hkv, ld_qkv, ld_out, ld_dq,
                                    ld_dkv, softmax_scale, (const int*)lo, (const uint32_t*)vbits, (const int*)kv_lo,
                                    (const int*)q_hi, (const int*)lo_hi, st);
}
