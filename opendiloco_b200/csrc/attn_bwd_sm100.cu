// Causal flash-attention BACKWARD on tcgen05 / TMEM / TMA for sm_100a (SURVEY.md §2.5 K5), head_dim 64, bf16, MHA + GQA.
//
//   P  = exp(S*scale - lse)          S  = Q K^T
//   dV = P^T dO                      dP = dO V^T
//   dS = P * (dP - D) * scale        D  = rowsum(dO * O)        (pre-pass kernel)
//   dK = dS^T Q                      dQ = dS K                  (dQ: fp32 TMA reduce-add across key tiles, post-pass -> bf16)
//
// One CTA per (batch, kv-head, PAIR of 128-key tiles {x, nq-1-x}) - every CTA runs the same number of iterations.  It
// keeps K and V in shared memory and dK/dV accumulators in tensor memory and walks over the query heads of its GQA group
// and the causal range of 128-query tiles.  The score tiles are computed TRANSPOSED (keys on the TMEM lanes) so that the
// probabilities can feed the dV / dK GEMMs straight from tensor memory - shared-memory bandwidth (128 B/clk) is the
// limiter of this kernel: an M128 N64 K16 MMA with both operands in smem needs 6 KB per 32 tensor cycles.
//     S^T  = K  Q^T    A = K  (smem, K-major)   B = Q  (smem, K-major)   N = 128
//     dP^T = V  dO^T   A = V  (smem, K-major)   B = dO (smem, K-major)   N = 128
//     dV  += P^T  dO   A = P^T  (TMEM, bf16)    B = dO (smem, MN-major)  N = 64
//     dK  += dS^T Q    A = dS^T (TMEM, bf16)    B = Q  (smem, MN-major)  N = 64
//     dQ   = dS   K    A = dS^T tile in smem read MN-major               B = K (smem, MN-major)   N = 64
// The same [128 x 64] swizzled tiles serve as K-major and as MN-major operands - only the descriptor changes.
// TMEM: S^T [0,128)  dP^T [128,256) - overwritten in place by P^T / dS^T (bf16, 2 queries per column) once read -
// dV [256,320) dK [320,384) dQ [384,448).   512 threads in four warpgroups with their own register budgets (setmaxnreg):
// warp 0 TMA + warp 1 MMA (96 regs), warps 4-11 element-wise (two threads per KEY row, 64 queries each; 160 regs) +
// dK/dV epilogue, warps 12-15 dQ drain (TMEM -> staging -> TMA reduce-add; 96 regs).
//
// MASKED instantiation (padding / per-document masks, see odb_attn_mask_prep in attn_sm100.cu): key tile kt visits query
// tiles kt .. q_hi[b, kt]; the per-query-tile statistics block carries a third row, lo of the 128 queries, so an
// element-wise thread (one key row) applies allowed(s, t) = t == s || (lo[s] <= t < s && valid[t]) when its warp needs it.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "packed_math.cuh"

using namespace odb;
using namespace sm100;
using namespace packed_math;

namespace attn_bwd {

constexpr int BQ = 128, BKV = 128, D = 64;
constexpr int TILE = 128 * 128;                  // bytes of a [128 x 64] bf16 tile
// Warp roles: warp 0 TMA, 1 MMA, 2-3 idle | 4 .. 4+4*EWS-1 element-wise | last 4 warps dQ drain.  EWS = threads per key row
// (2: 64 queries each, 512 threads, registers 96/160/160/96; 4: 32 queries each, 768 threads, registers 64/88x4/64).
constexpr int DRAIN_THREADS = 128;
constexpr int EW_WARP0 = 4;
template <int EWS> struct Roles {
  static constexpr int EW_WARPS = 4 * EWS, EW_THREADS = 128 * EWS, DRAIN_WARP0 = EW_WARP0 + EW_WARPS;
  static constexpr int THREADS = 32 * (DRAIN_WARP0 + 4);
  static constexpr int NQ = 128 / EWS;             // queries (score columns) per element-wise thread
  static constexpr int DC = 64 / EWS;              // dK / dV columns per thread in the epilogue
  static constexpr int REG_CTRL = EWS == 2 ? 96 : 64, REG_EW = EWS == 2 ? 160 : 88, REG_DRAIN = EWS == 2 ? 96 : 64;   // must sum to the launch allocation (setmaxnreg trades inside the CTA pool)
};
constexpr int QST = 3;                         // Q / dO / stats pipeline stages
constexpr int STAT_BYTES = 2 * 128 * 4;        // per (b, h, query tile): -lse*log2(e) [128] then -D*scale [128]
constexpr int MASKED_STAT_BYTES = 3 * 128 * 4; // ... then lo [128] (int32) of the MASKED instantiation
// K, V, QST x (Q, dO), dS^T (2 query chunks), dQ staging fp32 [128 x 64] = 2 chunks of 128 B rows, stats, barriers
constexpr int SMEM_BYTES = 2 * TILE + 2 * QST * TILE + 2 * TILE + 2 * TILE + QST * STAT_BYTES + 1024 + 256;
constexpr int MASKED_SMEM_BYTES = SMEM_BYTES + QST * (MASKED_STAT_BYTES - STAT_BYTES);
constexpr uint32_t TMEM_COLS = 512;
constexpr int DEFAULT_EWS = 2;

struct Params {
  int B, S, Hq, Hkv;
  float scale, scale_log2;
  const float* stats;    // [B, Hq, S/128, 2, 128] written by the pre-pass
  long long* dbg;        // optional timeline of CTA (0,0,0): [iteration][16] clock64 stamps (nullptr = off)
  // MASKED only (odb_attn_mask_prep outputs)
  const uint32_t* vbits; // [B, S/32] key-valid bits
  const int* q_hi;       // [B, S/128] last query tile a key tile visits
  const int* lo_hi;      // [B, S/128] largest lo of a query tile
};

#define BWD_STAMP(slot) do { if (dbg_on) p.dbg[it * 16 + (slot)] = clock64(); } while (0)

__device__ __forceinline__ void lds_2x64(uint32_t addr, uint64_t& a, uint64_t& b) {
  asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}
__device__ __forceinline__ uint32_t mul_bf16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}

template <int N>
__device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

template <int N>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t (&r)[N]) {
  static_assert(N == 16 || N == 32 || N == 64);
  if constexpr (N == 16) {
    tmem_ld_32x32b_x16(taddr, r);
  } else {
#pragma unroll
    for (int c = 0; c < N; c += 32) tmem_ld_32x32b_x32(taddr + c, *reinterpret_cast<uint32_t(*)[32]>(&r[c]));
  }
}
template <int N>
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&r)[N]) {
  static_assert(N == 16 || N == 32);
  if constexpr (N == 16) tmem_st_32x32b_x16(taddr, r);
  else tmem_st_32x32b_x32(taddr, r);
}

template <int EWS, bool MASKED = false>
__global__ void __launch_bounds__(Roles<EWS>::THREADS, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_do,
                const __grid_constant__ CUtensorMap tmap_dq, const __grid_constant__ CUtensorMap tmap_dk,
                const __grid_constant__ CUtensorMap tmap_dv, Params p) {
  using R = Roles<EWS>;
  constexpr int SB = MASKED ? MASKED_STAT_BYTES : STAT_BYTES, SF = SB / 4;   // statistics block: bytes / floats
  constexpr int EW_THREADS = R::EW_THREADS, DRAIN_WARP0 = R::DRAIN_WARP0, NQ = R::NQ, DC = R::DC;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = sK + TILE;
  uint8_t* sQ = sV + TILE;                 // QST stages
  uint8_t* sdO = sQ + QST * TILE;          // QST stages
  uint8_t* sdS = sdO + QST * TILE;         // dS^T: [2 query-chunks][128 key rows][128 B]  (also the dK/dV store staging)
  uint8_t* sdQ = sdS + 2 * TILE;           // fp32 staging: [2 column-chunks][128 rows][128 B]
  float* sStat = reinterpret_cast<float*>(sdQ + 2 * TILE);   // QST x {-lse2[128], -dsum*scale[128]}
  uint64_t* kv_full = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sStat) + QST * SB);
  uint64_t* kv_empty = kv_full + 1;        // the key tile's last MMAs retired: K / V may be replaced
  uint64_t* q_full = kv_empty + 1;         // [QST]
  uint64_t* q_empty = q_full + QST;        // [QST]
  uint64_t* s_full = q_empty + QST;        // S^T ready
  uint64_t* dp_full = s_full + 1;          // dP^T ready (and every earlier MMA retired)
  uint64_t* s_free = dp_full + 1;          // S^T lives in registers: the next S^T may overwrite the columns (8 warps)
  uint64_t* pds_full = s_free + 1;         // P^T / dS^T in tensor memory, dS^T in shared memory (8 warp arrivals)
  uint64_t* mma_done = pds_full + 1;       // dV/dK/dQ MMAs of this iteration retired (dQ accumulator ready)
  uint64_t* dq_empty = mma_done + 1;       // dQ accumulator drained (4 warp arrivals)
  uint64_t* dkv_empty = dq_empty + 1;      // dK/dV accumulators read by the epilogue (8 warp arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dkv_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = p.S / BQ;
  // Each CTA owns TWO key tiles of one (batch, kv head): tile x (nq-x query tiles to visit) and tile nq-1-x (x+1), so every
  // CTA runs group*(nq+1) iterations - a balanced grid - and pays the fixed costs once.  `it` is the CTA-wide iteration
  // index all per-iteration barrier parities derive from.
  pdl_launch_dependents();
  const int kb_first = (int)blockIdx.x, kb_second = nq - 1 - (int)blockIdx.x;
  const int nitems = kb_first != kb_second ? 2 : 1;
  const int hk = blockIdx.y, b = blockIdx.z;
  const int group = p.Hq / p.Hkv;
  const int col_k = (p.Hq + hk) * D, col_v = (p.Hq + p.Hkv + hk) * D;
  const bool dbg_cta = p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
  // query tiles kb .. qend-1 of key tile kb
  auto q_end = [&](int kb) { return MASKED ? p.q_hi[b * nq + kb] + 1 : nq; };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_do);
    mbar_init(kv_full, 1);
    mbar_init(kv_empty, 1);
    for (int i = 0; i < QST; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
    mbar_init(s_full, 1);
    mbar_init(dp_full, 1);
    mbar_init(s_free, R::EW_WARPS);
    mbar_init(pds_full, R::EW_WARPS);
    mbar_init(mma_done, 1);
    mbar_init(dq_empty, 4);
    mbar_init(dkv_empty, R::EW_WARPS);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tb = *tmem_slot;
  const uint32_t tS = tb, tdP = tb + 128, tdV = tb + 256, tdK = tb + 320, tdQ = tb + 384;
  pdl_wait();

  // register file split per warpgroup (EWS = 2: 128 threads x {96, 160, 160, 96}; EWS = 4: 80 at launch -> {64, 88 x 4, 64})
  // (each setmaxnreg sits inside its role branch and the branches only re-join at the final barrier, so ptxas allocates
  // every role's code against its own budget)
  if (warp < EW_WARP0) {
    reg_dealloc<R::REG_CTRL>();
    if (warp == 0 && lane == 0) {
      int st = 0, ph = 0;                                // Q stage ring position / phase
      for (int w = 0; w < nitems; ++w) {
        const int kb = w ? kb_second : kb_first;         // causal: query tiles kb..nq-1
        mbar_wait(kv_empty, (w & 1) ^ 1);
        mbar_arrive_expect_tx(kv_full, 2 * TILE);
        tma_load_2d(sK, &tmap_qkv, kv_full, col_k, b * p.S + kb * BKV);
        tma_load_2d(sV, &tmap_qkv, kv_full, col_v, b * p.S + kb * BKV);
        for (int hh = 0; hh < group; ++hh) {
          const int h = hk * group + hh;
          for (int qi = kb, qe = q_end(kb); qi < qe; ++qi) {
            mbar_wait(&q_empty[st], ph ^ 1);
            mbar_arrive_expect_tx(&q_full[st], 2 * TILE + SB);
            tma_load_2d(sQ + st * TILE, &tmap_qkv, &q_full[st], h * D, b * p.S + qi * BQ);
            tma_load_2d(sdO + st * TILE, &tmap_do, &q_full[st], h * D, b * p.S + qi * BQ);
            bulk_load_1d(sStat + st * SF, p.stats + (((size_t)b * p.Hq + h) * nq + qi) * SF, SB, &q_full[st]);
            if (++st == QST) { st = 0; ph ^= 1; }
          }
        }
      }
    } else if (warp == 1) {
      constexpr uint32_t id_s = make_idesc_bf16(128, 128, 0, 0);     // S^T, dP^T
      constexpr uint32_t id_ts = make_idesc_bf16(128, 64, 0, 1);     // dV, dK: A from tensor memory, B MN-major
      constexpr uint32_t id_q = make_idesc_bf16(128, 64, 1, 1);      // dQ: both operands MN-major
      const bool leader = elect_one();
      const uint64_t kd = make_smem_desc_sw128(smem_u32(sK), 16, 1024);        // K as K-major A (S^T) / MN-major B (dQ)
      const uint64_t vd = make_smem_desc_sw128(smem_u32(sV), 16, 1024);
      const uint64_t dsd_mn = make_smem_desc_sw128(smem_u32(sdS), TILE, 1024);   // dS: 2 MN chunks (64 queries) TILE bytes apart
      const bool dbg_on = dbg_cta && lane == 0;
      int st = 0, ph = 0;                                // stage / phase of the NEXT S^T to issue
      // Software pipeline (the tensor pipe executes in issue order):
      //   S^T(it+1) is issued as soon as the element-wise warps hold S^T(it) in registers, so it runs under their math;
      //   dV/dK(it) follow once P^T/dS^T(it) are in place, then dP^T(it+1) (it overwrites the columns P^T/dS^T(it) were
      //   read from), and last dQ(it) once the drain warps emptied the previous dQ tile.
      auto issue_s = [&]() {
        const uint64_t qd = make_smem_desc_sw128(smem_u32(sQ + st * TILE), 16, 1024);
        mbar_wait(&q_full[st], ph);
        tc_fence_after_sync();
        if (leader) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tS, kd + 2 * k, qd + 2 * k, id_s, k > 0);
          umma_commit(s_full);
        }
        __syncwarp();
      };
      auto issue_dp = [&](int stg) {
        const uint64_t dod = make_smem_desc_sw128(smem_u32(sdO + stg * TILE), 16, 1024);
        if (leader) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss(tdP, vd + 2 * k, dod + 2 * k, id_s, k > 0);
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
        int cur = st;                                    // stage of iteration `it`
        issue_dp(cur);
        if (++st == QST) { st = 0; ph ^= 1; }
        for (int i = 0; i < iters; ++i) {
          const int it = g + i;
          const uint64_t qd = make_smem_desc_sw128(smem_u32(sQ + cur * TILE), 16, 1024);
          const uint64_t dod = make_smem_desc_sw128(smem_u32(sdO + cur * TILE), 16, 1024);
          const int nxt = st;
          BWD_STAMP(9);
          if (i + 1 < iters) {
            mbar_wait(s_free, it & 1);
            issue_s();
            if (++st == QST) { st = 0; ph ^= 1; }
          }
          BWD_STAMP(10);
          mbar_wait(pds_full, it & 1);                   // P^T, dS^T in tensor memory; dS^T in shared memory
          if (i == 0 && w > 0) mbar_wait(dkv_empty, (w - 1) & 1);   // the epilogue read the previous key tile's dK / dV
          tc_fence_after_sync();
          BWD_STAMP(11);
          const bool first = (i == 0);
          if (leader) {
            // A straight from tensor memory: 16 queries = 8 columns per K step.  Each element-wise thread's NQ dP^T
            // columns now hold P^T (first NQ/2) and dS^T (last NQ/2) of its NQ queries.
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_ts(tdV, tdP + (16 * k / NQ) * NQ + (16 * k % NQ) / 2, dod + 128 * k, id_ts, (first && k == 0) ? 0u : 1u);
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_ts(tdK, tdP + (16 * k / NQ) * NQ + NQ / 2 + (16 * k % NQ) / 2, qd + 128 * k, id_ts, (first && k == 0) ? 0u : 1u);
          }
          __syncwarp();
          // dP^T(it+1) only has to wait for dV / dK(it) (they read P^T / dS^T out of its columns); dQ(it) reads dS from
          // shared memory, so it goes AFTER - the element-wise warps get dP^T(it+1) one GEMM earlier
          if (i + 1 < iters) issue_dp(nxt);
          if (it > 0) mbar_wait(dq_empty, (it - 1) & 1); // previous dQ tile drained
          tc_fence_after_sync();
          BWD_STAMP(12);
          if (leader) {
#pragma unroll
            for (int k = 0; k < 8; ++k) umma_ss(tdQ, dsd_mn + 128 * k, kd + 128 * k, id_q, k > 0);
            umma_commit(&q_empty[cur]);
            umma_commit(mma_done);
            if (i + 1 == iters) umma_commit(kv_empty);
          }
          __syncwarp();
          cur = nxt;
        }
        g += iters;
      }
    }
  } else if (warp >= DRAIN_WARP0) {
    reg_dealloc<R::REG_DRAIN>();
    // ------------------------------------------------------------------ dQ drain warps
    // dQ tile of iteration `it`: TMEM -> fp32 staging -> TMA reduce-add into the fp32 accumulator, off the critical path
    // of the element-wise warps.
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const bool elected = threadIdx.x == DRAIN_WARP0 * 32;
    const bool dbg_on = dbg_cta && elected;
    for (int w = 0, it = 0; w < nitems; ++w) {
      const int kb = w ? kb_second : kb_first;
      for (int hh = 0; hh < group; ++hh) {
        const int h = hk * group + hh;
        for (int qi = kb, qe = q_end(kb); qi < qe; ++qi, ++it) {
          mbar_wait(mma_done, it & 1);
          tc_fence_after_sync();
          if (elected) tma_store_wait_read<0>();         // previous reduce finished reading the staging tile
          named_bar_sync(3, DRAIN_THREADS);
          BWD_STAMP(7);
#pragma unroll
          for (int c = 0; c < 2; ++c) {                  // 32 fp32 columns at a time (register budget of this warpgroup)
            uint32_t dq[32];
            tmem_ld_32x32b_x32(tdQ + lane_off + c * 32, dq);
            tmem_ld_wait();
            if (c == 1) {
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0) mbar_arrive(dq_empty);
              BWD_STAMP(6);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u)
              *reinterpret_cast<uint4*>(sdQ + c * TILE + row * 128 + ((u ^ (row & 7)) * 16)) =
                  make_uint4(dq[u * 4 + 0], dq[u * 4 + 1], dq[u * 4 + 2], dq[u * 4 + 3]);
          }
          fence_proxy_async_smem();
          named_bar_sync(4, DRAIN_THREADS);
          if (elected) {
            tma_reduce_add_2d(&tmap_dq, sdQ, h * D, b * p.S + qi * BQ);
            tma_reduce_add_2d(&tmap_dq, sdQ + TILE, h * D + 32, b * p.S + qi * BQ);
            tma_store_commit();
          }
          BWD_STAMP(8);
        }
      }
    }
    if (elected) tma_store_wait<0>();
  } else {
    // ------------------------------------------------------------------ element-wise warps
    reg_alloc<R::REG_EW>();
    const int q = warp & 3;
    const int row = q * 32 + lane;                       // KEY row inside the tile == TMEM lane
    const int part = (warp - EW_WARP0) >> 2;             // queries [NQ*part, NQ*part + NQ) of the query tile
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const float c = p.scale_log2;
    const uint64_t c2 = pack2(c, c), sc2 = pack2(p.scale, p.scale);
    const bool elected = threadIdx.x == EW_WARP0 * 32;
    const bool dbg_on = dbg_cta && elected;
    const uint32_t tPD = tdP + lane_off + part * NQ;     // this thread's dP^T columns; P^T -> first half, dS^T -> second half
    int st = 0, ph = 0;
    for (int w = 0, it = 0; w < nitems; ++w) {
      const int kb = w ? kb_second : kb_first;
      const int key = kb * BKV + row;                    // MASKED: this thread's key position and its valid bit
      const bool key_valid = MASKED ? (p.vbits[(size_t)b * (p.S / 32) + key / 32] >> (key & 31)) & 1u : true;
      for (int hh = 0; hh < group; ++hh) {
        for (int qi = kb, qe = q_end(kb); qi < qe; ++qi, ++it) {
          const bool diag = (qi == kb);
          const uint32_t stat = smem_u32(sStat + st * SF + part * NQ);
          BWD_STAMP(0);
          mbar_wait(&q_full[st], ph);                    // the statistics of this query tile are in shared memory
          mbar_wait(s_full, it & 1);
          tc_fence_after_sync();
          BWD_STAMP(1);
          uint32_t pp[NQ / 2];
          {
            uint32_t sr[NQ];
            tmem_ld_cols<NQ>(tS + lane_off + part * NQ, sr);
            tmem_ld_wait();
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(s_free);          // S^T(it+1) may now be computed into the same columns
            BWD_STAMP(2);
            if constexpr (MASKED) {
              // queries qi*128 + part*NQ + i; the warp takes the causal code when none of its keys needs a masked element
              const bool need = diag || !key_valid || key < p.lo_hi[b * nq + qi];
              if (__any_sync(0xffffffffu, need)) {
                const int rel = key - (qi * BQ + part * NQ);   // i == rel: the query is this key
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
                if (row > part * NQ + i) sr[i] = 0xff800000u;     // key after query: -inf -> P = 0
            }
            // P = exp2(S*c - lse2[query]): packed fp32x2 math; of every four exponentials two go through the MUFU and two
            // through the FMA-pipe polynomial (see attn_sm100.cu).  The per-query statistics are broadcast reads.
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
          BWD_STAMP(3);
          mbar_wait(dp_full, it & 1);                    // dP^T ready (dV / dK of the previous tile retired)
          tc_fence_after_sync();
          uint32_t ds[NQ / 2];
          {
            uint32_t dr[NQ];
            tmem_ld_cols<NQ>(tPD, dr);
            tmem_ld_wait();
            // dS = P * (dP*scale - D*scale): the bracket in packed fp32, the product in packed bf16 (the P the dV GEMM sees)
#pragma unroll
            for (int i = 0; i < NQ; i += 4) {
              uint64_t nda, ndb;
              lds_2x64(stat + 512 + i * 4, nda, ndb);
              ds[i / 2] = mul_bf16x2(pp[i / 2], cvt_bf16x2(ffma2(pack2u(dr[i], dr[i + 1]), sc2, nda)));
              ds[i / 2 + 1] = mul_bf16x2(pp[i / 2 + 1], cvt_bf16x2(ffma2(pack2u(dr[i + 2], dr[i + 3]), sc2, ndb)));
            }
          }
          if (it > 0) mbar_wait(mma_done, (it - 1) & 1);   // dQ of the previous tile no longer reads the dS buffer
          if (w > 0 && hh == 0 && qi == kb) {
            // the dS buffer doubled as the dK / dV store staging of the previous key tile: its TMA store must have read it
            if (elected) tma_store_wait_read<0>();
            named_bar_sync(1, EW_THREADS);
          }
          BWD_STAMP(4);
          // P^T / dS^T -> tensor memory (A operands of dV / dK), dS^T -> shared memory (A operand of dQ, MN-major)
          tmem_st_cols<NQ / 2>(tPD, pp);
          tmem_st_cols<NQ / 2>(tPD + NQ / 2, ds);
          {
            // query index part*NQ + i sits in 64-query chunk (part*NQ)/64 at 16-byte unit ((part*NQ) % 64) / 8 + u of its key row
            uint8_t* drow = sdS + ((part * NQ) >> 6) * TILE + row * 128;
            const int u0 = ((part * NQ) & 63) >> 3;
#pragma unroll
            for (int u = 0; u < NQ / 8; ++u)
              *reinterpret_cast<uint4*>(drow + (((u0 + u) ^ (row & 7)) * 16)) =
                  make_uint4(ds[u * 4 + 0], ds[u * 4 + 1], ds[u * 4 + 2], ds[u * 4 + 3]);
          }
          tmem_st_wait();
          fence_proxy_async_smem();
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(pds_full);
          BWD_STAMP(5);
          if (++st == QST) { st = 0; ph ^= 1; }
        }
      }
      // ---- dK / dV epilogue of this key tile: this thread's 32 columns -> bf16 -> staging (the dS buffer) -> TMA store
      mbar_wait(mma_done, (it - 1) & 1);
      tc_fence_after_sync();
      uint32_t r[DC];
      tmem_ld_cols<DC>(tdK + lane_off + part * DC, r);
      tmem_ld_wait();
#pragma unroll
      for (int u = 0; u < DC / 8; ++u) {
        float f[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(r[u * 8 + i]);
        *reinterpret_cast<uint4*>(sdS + row * 128 + (((part * (DC / 8) + u) ^ (row & 7)) * 16)) = pack8(f);
      }
      tmem_ld_cols<DC>(tdV + lane_off + part * DC, r);
      tmem_ld_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(dkv_empty);             // the next key tile may start accumulating
#pragma unroll
      for (int u = 0; u < DC / 8; ++u) {
        float f[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(r[u * 8 + i]);
        *reinterpret_cast<uint4*>(sdS + TILE + row * 128 + (((part * (DC / 8) + u) ^ (row & 7)) * 16)) = pack8(f);
      }
      fence_proxy_async_smem();
      named_bar_sync(2, EW_THREADS);
      if (elected) {
        tma_store_2d(&tmap_dk, sdS, hk * D, b * p.S + kb * BKV);
        tma_store_2d(&tmap_dv, sdS + TILE, hk * D, b * p.S + kb * BKV);
        tma_store_commit();
      }
    }
    if (elected) tma_store_wait<0>();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tb, TMEM_COLS);
}

// Pre-pass: per (token, head) D = sum_d dO * O, stored together with the forward's log-sum-exp in the layout the main
// kernel bulk-copies per query tile: stats[b, h, s/128, 0, s%128] = -lse * log2(e), stats[..., 1, ...] = -D * scale.
// Eight lanes per (token, head) (16 bytes of dO and O each); the same threads zero the fp32 dQ accumulator row.
// MASKED: a third row carries lo[s] (int32 bits).
template <bool MASKED = false>
__global__ void __launch_bounds__(256) attn_dsum_kernel(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ out,
                                                        const float* __restrict__ lse, float* __restrict__ stats,
                                                        float* __restrict__ dq_acc, int B, int S, int Hq, long long ld, float scale,
                                                        const int* __restrict__ lo = nullptr) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)B * S * Hq * 8;
  if (i >= total) return;                                // total is a multiple of 8: whole lane groups leave together
  const int sub = (int)(i & 7);
  const long long w = i >> 3;
  const long long t = w / Hq;
  const int h = (int)(w % Hq);
  float a[8], o[8];
  unpack8(ld_v4(dout + t * ld + h * 64 + sub * 8), a);
  unpack8(ld_v4(out + t * ld + h * 64 + sub * 8), o);
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s = fmaf(a[j], o[j], s);
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  float4* z = reinterpret_cast<float4*>(dq_acc + (t * Hq + h) * 64 + sub * 8);
  z[0] = make_float4(0.f, 0.f, 0.f, 0.f);
  z[1] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (sub == 0) {
    const long long bb = t / S, ss = t % S;
    float* dst = stats + (((bb * Hq + h) * (S / 128) + ss / 128) * (MASKED ? 3 : 2)) * 128 + (ss % 128);
    dst[0] = -lse[(bb * Hq + h) * S + ss] * 1.4426950408889634f;
    dst[128] = -s * scale;
    if (MASKED) dst[256] = __int_as_float(lo[t]);
  }
}

// Post-pass: fp32 dQ accumulator -> bf16 into dq_out (row stride ld_out), and - when cos/sin tables are given - the
// transpose RoPE rotation of dQ (on the way) and of dK (in place), so the packed dq|dk|dv buffer leaves ready for the
// projection's dgrad / wgrad GEMMs.  One thread per 8 rotation pairs: x[j..j+8) and x[j+32..j+40) of one (token, head).
__global__ void __launch_bounds__(256) attn_bwd_finish_kernel(const float* __restrict__ dq_acc, __nv_bfloat16* __restrict__ dq_out,
                                                              __nv_bfloat16* __restrict__ dk, const float* __restrict__ cos_t,
                                                              const float* __restrict__ sin_t, long long T, int S, int Hq, int Hkv,
                                                              long long ld_out, long long ld_dk) {
  pdl_launch_dependents();
  pdl_wait();
  const int H = Hq + (cos_t != nullptr ? Hkv : 0);
  const long long total = T * H * 4;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int jv = (int)(i & 3);
  const long long th = i >> 2;
  const int head = (int)(th % H);
  const long long t = th / H;
  float a[8], b[8];
  __nv_bfloat16* dst;
  if (head < Hq) {
    const float* src = dq_acc + (t * Hq + head) * 64 + jv * 8;
    const float4 a0 = ld_f4(src), a1 = ld_f4(src + 4), b0 = ld_f4(src + 32), b1 = ld_f4(src + 36);
    a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
    b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w; b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
    dst = dq_out + t * ld_out + head * 64 + jv * 8;
  } else {
    dst = dk + t * ld_dk + (head - Hq) * 64 + jv * 8;
    unpack8(ld_v4(dst), a);
    unpack8(ld_v4(dst + 32), b);
  }
  if (cos_t != nullptr) {
    const int pos = (int)(t % S);
    const float4 c0 = ld_f4(cos_t + (size_t)pos * 32 + jv * 8), c1 = ld_f4(cos_t + (size_t)pos * 32 + jv * 8 + 4);
    const float4 s0 = ld_f4(sin_t + (size_t)pos * 32 + jv * 8), s1 = ld_f4(sin_t + (size_t)pos * 32 + jv * 8 + 4);
    const float cs[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
    const float sn[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float x = a[j], y = b[j];
      a[j] = x * cs[j] + y * sn[j];                      // rotation by -theta
      b[j] = y * cs[j] - x * sn[j];
    }
  }
  st_v4(dst, pack8(a));
  st_v4(dst + 32, pack8(b));
}

}  // namespace attn_bwd

static long long* g_bwd_dbg = nullptr;
// debugging aid: device buffer [iterations][16] that receives the clock64 timeline of CTA (0,0,0); nullptr switches it off
ODB_EXPORT int odb_attn_bwd_set_dbg(void* buf) {
  g_bwd_dbg = (long long*)buf;
  return 0;
}

namespace {
template <bool MASKED>
int launch_attn_bwd(const void* qkv, const void* out, const void* dout, const void* lse, void* stats, void* dq_acc, void* dq,
                    void* dk, void* dv, const void* cos_t, const void* sin_t, int B, int S, int Hq, int Hkv, long long ld_qkv,
                    long long ld_out, long long ld_dq, long long ld_dkv, float softmax_scale, const int* lo,
                    const uint32_t* vbits, const int* q_hi, const int* lo_hi, cudaStream_t st) {
  using namespace attn_bwd;
  if (S % BQ || Hq % Hkv || ld_qkv % 8 || ld_out % 8 || ld_dq % 8 || ld_dkv % 8) return -1;
  const long long T = (long long)B * S;
  {
    const long long threads = T * Hq * 8;
    launch_pdl(attn_dsum_kernel<MASKED>, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, st, (const __nv_bfloat16*)dout,
               (const __nv_bfloat16*)out, (const float*)lse, (float*)stats, (float*)dq_acc, B, S, Hq, ld_out, softmax_scale, lo);
  }
  CUtensorMap tq, tdo, tdq, tdk, tdv;
  int rc;
  if ((rc = make_tmap_2d(&tq, qkv, T, (Hq + 2 * Hkv) * D, ld_qkv * 2, 128, 64, 2))) return rc;
  if ((rc = make_tmap_2d(&tdo, dout, T, Hq * D, ld_out * 2, 128, 64, 2))) return rc;
  if ((rc = make_tmap_2d(&tdq, dq_acc, T, Hq * D, (long long)Hq * D * 4, 128, 32, 4))) return rc;
  if ((rc = make_tmap_2d(&tdk, dk, T, Hkv * D, ld_dkv * 2, 128, 64, 2))) return rc;
  if ((rc = make_tmap_2d(&tdv, dv, T, Hkv * D, ld_dkv * 2, 128, 64, 2))) return rc;
  Params p{};
  p.B = B; p.S = S; p.Hq = Hq; p.Hkv = Hkv;
  p.scale = softmax_scale;
  p.scale_log2 = softmax_scale * 1.4426950408889634f;
  p.stats = (const float*)stats;
  p.dbg = g_bwd_dbg;
  p.vbits = vbits; p.q_hi = q_hi; p.lo_hi = lo_hi;
  dim3 grid((S / BKV + 1) / 2, Hkv, B);
  if constexpr (MASKED) {
    // two threads per key row (the default split) only
    static bool attr_set = false;
    if (!attr_set) {
      cudaError_t e = cudaFuncSetAttribute(attn_bwd_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MASKED_SMEM_BYTES);
      if (e != cudaSuccess) return (int)e;
      attr_set = true;
    }
    launch_pdl(attn_bwd_kernel<2, true>, grid, dim3(Roles<2>::THREADS), MASKED_SMEM_BYTES, st, tq, tdo, tdq, tdk, tdv, p);
  } else {
    static int ews = 0;
    if (!ews) {
      const char* env = getenv("ODB_ATTN_BWD_SPLIT");      // element-wise threads per key row: 2 or 4
      ews = (env && atoi(env) == 2) ? 2 : (env && atoi(env) == 4) ? 4 : DEFAULT_EWS;
      cudaError_t e = cudaFuncSetAttribute(attn_bwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_bwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e != cudaSuccess) { ews = 0; return (int)e; }
    }
    if (ews == 2) launch_pdl(attn_bwd_kernel<2>, grid, dim3(Roles<2>::THREADS), SMEM_BYTES, st, tq, tdo, tdq, tdk, tdv, p);
    else launch_pdl(attn_bwd_kernel<4>, grid, dim3(Roles<4>::THREADS), SMEM_BYTES, st, tq, tdo, tdq, tdk, tdv, p);
  }
  {
    const long long threads = T * (Hq + (cos_t ? Hkv : 0)) * 4;
    launch_pdl(attn_bwd_finish_kernel, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, st, (const float*)dq_acc,
               (__nv_bfloat16*)dq, (__nv_bfloat16*)dk, (const float*)cos_t, (const float*)sin_t, T, S, Hq, Hkv, ld_dq, ld_dkv);
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}
}  // namespace

// stats: fp32 scratch of 2 * B * Hq * S elements (per-query statistics, written by the pre-pass);
// dq_acc: fp32 [T, Hq*64] scratch (zeroed by the pre-pass, accumulated with TMA reduce-add);
// dq, dk, dv: bf16 outputs with row strides ld_dq / ld_dkv elements - e.g. the three column blocks of one packed
// [T, (Hq+2*Hkv)*64] buffer.  With cos/sin (fp32 [S, 32] tables) dq and dk leave with the RoPE rotation undone.
ODB_EXPORT int odb_attn_bwd(const void* qkv, const void* out, const void* dout, const void* lse, void* stats, void* dq_acc,
                            void* dq, void* dk, void* dv, const void* cos_t, const void* sin_t, int B, int S, int Hq, int Hkv,
                            long long ld_qkv, long long ld_out, long long ld_dq, long long ld_dkv, float softmax_scale,
                            cudaStream_t st) {
  return launch_attn_bwd<false>(qkv, out, dout, lse, stats, dq_acc, dq, dk, dv, cos_t, sin_t, B, S, Hq, Hkv, ld_qkv, ld_out,
                                ld_dq, ld_dkv, softmax_scale, nullptr, nullptr, nullptr, nullptr, st);
}

// Same with a mask description (lo, vbits, q_hi, lo_hi from odb_attn_mask_prep); stats then holds 3 * B * Hq * S elements.
ODB_EXPORT int odb_attn_bwd_masked(const void* qkv, const void* out, const void* dout, const void* lse, void* stats, void* dq_acc,
                                   void* dq, void* dk, void* dv, const void* cos_t, const void* sin_t, int B, int S, int Hq,
                                   int Hkv, long long ld_qkv, long long ld_out, long long ld_dq, long long ld_dkv,
                                   float softmax_scale, const void* lo, const void* vbits, const void* q_hi, const void* lo_hi,
                                   cudaStream_t st) {
  if (!lo || !vbits || !q_hi || !lo_hi) return -1;
  return launch_attn_bwd<true>(qkv, out, dout, lse, stats, dq_acc, dq, dk, dv, cos_t, sin_t, B, S, Hq, Hkv, ld_qkv, ld_out, ld_dq,
                               ld_dkv, softmax_scale, (const int*)lo, (const uint32_t*)vbits, (const int*)q_hi,
                               (const int*)lo_hi, st);
}
