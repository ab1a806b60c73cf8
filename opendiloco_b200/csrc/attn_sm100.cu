// Causal flash-attention forward on tcgen05 / TMEM / TMA for sm_100a (SURVEY.md §2.5 K5), head_dim 64 or 128, bf16, MHA + GQA.
//
// Reads q/k/v straight out of the packed projection buffer qkv[T, (Hq + 2*Hkv) * 64] (token-major rows: no transposes)
// through ONE tensor map, writes out[T, Hq*64] token-major (the o-proj GEMM's A operand) and lse[B, Hq, S].
//
// One CTA per (batch, q-head, 128-query block); two CTAs co-reside per SM (112 KB smem, 256 TMEM columns each) so one
// CTA's softmax overlaps the other's MMAs.  320 threads:
//   warp 0     TMA: Q once, then K_j / V_j 128-key tiles through a 2-stage mbarrier ring
//   warp 1     MMA: S = Q K_j^T  (tcgen05.mma M128 N128 K16 x4, both operands K-major, accumulator S in TMEM)
//                   O += P V_j   (M128 N64 K16 x8; A = P from shared memory K-major, B = V_j tile MN-major)
//   warps 2-9  softmax: TWO threads per query row (TMEM lane == row; warps 2-5 take keys 0-63 of the tile, warps 6-9 keys
//              64-127, row max exchanged through shared memory): tcgen05.ld S, online max/sum with exp2, causal mask
//              on the diagonal tile, rescale O in TMEM (tcgen05.ld/st), write P (bf16) into the swizzled smem operand;
//              epilogue: O / l -> bf16 -> swizzled staging tile -> TMA store
//
// Head size 128 (template parameter D): every [128 x D] operand is two 64-column TMA boxes, QK^T takes eight K16 steps
// across them, PV is N = 128 with V's two boxes as its MN chunks, and the softmax threads rescale / store 64 O columns
// each.  160 KB of shared memory and 320 TMEM columns (allocated 512) leave room for one CTA per SM only.
//
// MASKED instantiation (padding / per-document masks, described by odb_attn_mask_prep below): every role walks key tiles
// kv_lo[b, qt] .. qt instead of 0 .. qt; a warp whose rows see only allowed keys in a tile takes the causal code, the
// others apply allowed(s, t) = t == s || (lo[s] <= t < s && valid[t]) as -inf.  A row may meet fully masked tiles before
// its first allowed key, so the online softmax keeps its reference at -inf without producing NaN there.
#include "common.cuh"
#include "sm100_ptx.cuh"
#include "packed_math.cuh"
#include <climits>

using namespace odb;
using namespace sm100;
using namespace packed_math;

namespace attn {

constexpr int BQ = 128, BKV = 128;
constexpr int TILE_BYTES = 128 * 128;           // a [128 x 64] bf16 box (128-byte rows); a [128 x D] operand is D/64 boxes
constexpr int THREADS = 320;
constexpr int SOFTMAX_THREADS = 256;
// Per head size D (64 or 128):
//   D = 64 : 7 boxes + barriers = 114,816 B: two CTAs per SM need 2 x (smem + 1 KB reserved) <= 227 KB, so there is no slack
//            for a manual 1024-byte round-up - the dynamic window is declared 1024-aligned instead (it starts at the CTA's
//            smem base).  TMEM 256 columns - S: [0,128)  O: [128,192)  P (bf16, 2 keys per column): [192,256)
//   D = 128: 14 boxes (Q 2, K 2 x 2, V 2, out staging 2) = 160 KB: one CTA per SM.  S 128 + O 128 + P 64 = 320 columns, so
//            the allocation is 512 - S: [0,128)  O: [128,256)  P: [256,320)
template <int D> struct FwdCfg {
  static_assert(D == 64 || D == 128, "head size");
  static constexpr int NB = D / 64;             // 64-column boxes per [128 x D] operand
  static constexpr int OP_BYTES = NB * TILE_BYTES;
  static constexpr int SMEM_BYTES = OP_BYTES /*Q*/ + 2 * OP_BYTES /*K x2*/ + OP_BYTES /*V x1*/ + OP_BYTES /*out staging*/ + 128 /*barriers*/;
  static constexpr uint32_t TMEM_COLS = D == 64 ? 256 : 512;
  static constexpr int MIN_BLOCKS = D == 64 ? 2 : 1;
};

struct Params {
  int B, S, Hq, Hkv;
  float scale_log2;        // softmax_scale * log2(e)
  float* lse;              // [B, Hq, S], natural log
  long long* dbg;          // optional timeline of CTA (0,0,0): [tile][16] clock64 stamps (nullptr = off)
  // MASKED only (odb_attn_mask_prep outputs)
  const int* lo;           // [B*S] first allowed key of every query
  const uint32_t* vbits;   // [B, S/32] key-valid bits
  const int* kv_lo;        // [B, S/128] first key tile a query tile visits
};

#define ATT_STAMP(slot) do { if (dbg_on) p.dbg[j * 16 + (slot)] = clock64(); } while (0)

template <bool MASKED, int D = 64>
__global__ void __launch_bounds__(THREADS, FwdCfg<D>::MIN_BLOCKS)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_out, Params p) {
  constexpr int NB = FwdCfg<D>::NB, OP_BYTES = FwdCfg<D>::OP_BYTES;
  constexpr uint32_t TMEM_COLS = FwdCfg<D>::TMEM_COLS;
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ float red[2 * 256];                 // row max / row sum exchange between the two column halves (double-buffered)
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u)) __trap();     // swizzled tiles need 1024-byte alignment
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + OP_BYTES;
  uint8_t* sV = sK + 2 * OP_BYTES;              // single V stage: V_{j+1} is only needed after softmax_{j+1}
  uint8_t* sOut = sV + OP_BYTES;                // output staging tile (P lives in tensor memory)
  uint64_t* q_full = reinterpret_cast<uint64_t*>(sOut + OP_BYTES);
  uint64_t* k_full = q_full + 1;                // [2]
  uint64_t* k_empty = k_full + 2;               // [2]
  uint64_t* v_full = k_empty + 2;
  uint64_t* v_empty = v_full + 1;
  uint64_t* s_full = v_empty + 1;
  uint64_t* p_full = s_full + 1;
  uint64_t* s_free = p_full + 1;                // S_j is in registers: the next QK may overwrite the S columns
  uint64_t* o_done = s_free + 1;
  uint64_t* q_empty = o_done + 1;               // every QK^T of the current query tile retired: Q may be replaced
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_empty + 1);

  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = p.S / BQ;
  // Each CTA owns TWO query tiles of one (batch, head): tile nq-1-x (long) and tile x (short).  Every CTA therefore
  // walks nq+1 key tiles - a perfectly balanced grid - and the fixed cost (barrier init, TMEM allocation, pipeline
  // fill) is paid once per ~nq+1 tiles instead of once per ~nq/2.  `tg` below is the CTA-wide running tile index that
  // all barrier parities are derived from.
  const int qb[2] = {nq - 1 - (int)blockIdx.x, (int)blockIdx.x};
  const int nitems = qb[0] != qb[1] ? 2 : 1;
  const int h = blockIdx.y, b = blockIdx.z;
  const int hk = h / (p.Hq / p.Hkv);
  const int col_q = h * D, col_k = (p.Hq + hk) * D, col_v = (p.Hq + p.Hkv + hk) * D;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_qkv);
    tma_prefetch_desc(&tmap_out);
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&k_full[i], 1); mbar_init(&k_empty[i], 1); }
    mbar_init(v_full, 1);
    mbar_init(v_empty, 1);
    mbar_init(s_full, 1);
    mbar_init(p_full, 8);      // one arrival per softmax warp
    mbar_init(s_free, 8);
    mbar_init(o_done, 1);
    mbar_init(q_empty, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tS = tmem_base, tO = tmem_base + 128, tP = tmem_base + 128 + D;
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      // K runs one tile ahead of V: K_{j+1} is requested as soon as its stage is free (QK_{j-1} retired), V_j after
      // PV_{j-1} retired - V_j is not needed before softmax_j is done, K_{j+1} is needed right after softmax_j's S load.
      auto load_k = [&](int j, int tg) {
        const int st = tg & 1;
        mbar_wait(&k_empty[st], ((tg >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&k_full[st], OP_BYTES);
#pragma unroll
        for (int c = 0; c < NB; ++c)
          tma_load_2d(sK + st * OP_BYTES + c * TILE_BYTES, &tmap_qkv, &k_full[st], col_k + 64 * c, b * p.S + j * BKV);
      };
      for (int w = 0, t0 = 0; w < nitems; ++w) {
        const int j0 = MASKED ? p.kv_lo[b * nq + qb[w]] : 0;
        const int nkv = qb[w] + 1 - j0;          // causal: key tiles j0..qblk
        mbar_wait(q_empty, (w & 1) ^ 1);
        mbar_arrive_expect_tx(q_full, OP_BYTES);
#pragma unroll
        for (int c = 0; c < NB; ++c) tma_load_2d(sQ + c * TILE_BYTES, &tmap_qkv, q_full, col_q + 64 * c, b * p.S + qb[w] * BQ);
        load_k(j0, t0);
        for (int j = 0; j < nkv; ++j) {
          const int tg = t0 + j;
          if (j + 1 < nkv) load_k(j0 + j + 1, tg + 1);
          mbar_wait(v_empty, (tg & 1) ^ 1);
          mbar_arrive_expect_tx(v_full, OP_BYTES);
#pragma unroll
          for (int c = 0; c < NB; ++c)
            tma_load_2d(sV + c * TILE_BYTES, &tmap_qkv, v_full, col_v + 64 * c, b * p.S + (j0 + j) * BKV);
        }
        t0 += nkv;
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc_qk = make_idesc_bf16(BQ, BKV, 0, 0);   // S[128,128] = Q (K-major) x K^T (K-major)
    constexpr uint32_t idesc_pv = make_idesc_bf16(BQ, D, 0, 1);     // O[128,D] = P (TMEM, K-major) x V (smem, MN-major)
    const bool leader = elect_one();             // the same lane issues every MMA / commit of this CTA
    const uint64_t qd = make_smem_desc_sw128(smem_u32(sQ), 16, 1024);
    // V read MN-major: at D = 128 its two 64-column boxes are the two MN chunks, one box (LBO) apart
    const uint64_t vd = make_smem_desc_sw128(smem_u32(sV), NB > 1 ? TILE_BYTES : 16, 1024);
    const uint64_t kd0 = make_smem_desc_sw128(smem_u32(sK), 16, 1024);
    const uint64_t kd1 = make_smem_desc_sw128(smem_u32(sK + OP_BYTES), 16, 1024);
    const bool dbg_cta = p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && lane == 0;
    auto issue_qk = [&](int tg, bool last) {
      const int st = tg & 1;
      mbar_wait(&k_full[st], (tg >> 1) & 1);
      tc_fence_after_sync();
      if (leader) {
        const uint64_t kd = st ? kd1 : kd0;
        umma_ss(tS, qd, kd, idesc_qk, 0u);
        umma_ss(tS, qd + 2, kd + 2, idesc_qk, 1u);
        umma_ss(tS, qd + 4, kd + 4, idesc_qk, 1u);
        umma_ss(tS, qd + 6, kd + 6, idesc_qk, 1u);
        // D = 128: the second 64-column box of Q and K (descriptor addresses count 16-byte units)
#pragma unroll
        for (int k = 4; k < 4 * NB; ++k) {
          const uint32_t o = (k / 4) * (TILE_BYTES >> 4) + 2 * (k % 4);
          umma_ss(tS, qd + o, kd + o, idesc_qk, 1u);
        }
        umma_commit(s_full);
        umma_commit(&k_empty[st]);               // K stage reusable once this QK retired
        if (last) umma_commit(q_empty);          // ... and so is Q after the tile's last QK
      }
      __syncwarp();
    };
    for (int w = 0, t0 = 0; w < nitems; ++w) {
    const int nkv = qb[w] + 1 - (MASKED ? p.kv_lo[b * nq + qb[w]] : 0);
    const bool dbg_on = dbg_cta && w == 0;
    mbar_wait(q_full, w & 1);
    if (w > 0) mbar_wait(s_free, (t0 - 1) & 1);  // the previous query tile's last S has been read
    issue_qk(t0, nkv == 1);                      // S_0 = Q K_0^T
    for (int j = 0; j < nkv; ++j) {
      const int tg = t0 + j;
      ATT_STAMP(8);
      // As soon as the softmax warps hold S_j in registers, the next QK^T goes into the same TMEM columns - it runs while
      // they compute the probabilities, so S_{j+1} is waiting for them when they come back.
      if (j + 1 < nkv) {
        mbar_wait(s_free, tg & 1);
        issue_qk(tg + 1, j + 2 == nkv);
      }
      ATT_STAMP(9);
      mbar_wait(p_full, tg & 1);                 // P_j in tensor memory, O rescaled
      ATT_STAMP(10);
      mbar_wait(v_full, tg & 1);
      tc_fence_after_sync();
      if (leader) {
        // A operand straight from tensor memory: 16 keys of P = 8 columns per K step, no shared-memory read for A
        umma_ts(tO, tP, vd, idesc_pv, j > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 1; k < BKV / 16; ++k) umma_ts(tO, tP + 8 * k, vd + 128 * k, idesc_pv, 1u);
        umma_commit(v_empty);                    // V stage reusable
        umma_commit(o_done);                     // O (and P) stable
      }
      __syncwarp();
      ATT_STAMP(11);
    }
    t0 += nkv;
    }
  } else {
    // ------------------------------------------------------------------ softmax / correction / epilogue
    const int q = warp & 3;
    const int row = q * 32 + lane;               // query row inside the tile == TMEM lane
    const int half = (warp - 2) >> 2;            // 0: keys [0,64) of every tile and O columns [0,D/2) ; 1: the other halves
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const float c = p.scale_log2;
    const bool dbg_cta = p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 64;
    for (int w = 0, t0 = 0; w < nitems; ++w) {
    const int qblk = qb[w];
    const int j0 = MASKED ? p.kv_lo[b * nq + qblk] : 0;
    const int nkv = qblk + 1 - j0;
    const int row0 = b * p.S + qblk * BQ;        // first token row of this query tile
    const bool dbg_on = dbg_cta && w == 0;
    const int qpos = qblk * BQ + row;            // MASKED: this row's query position and its first allowed key
    const int lo_q = MASKED ? p.lo[b * p.S + qpos] : 0;
    float m = -INFINITY, l = 0.f;                // l: this thread's half of the row sum
    for (int j = 0; j < nkv; ++j) {
      const int tg = t0 + j;
      ATT_STAMP(0);
      mbar_wait(s_full, tg & 1);
      tc_fence_after_sync();
      ATT_STAMP(1);
      const bool diag = (j0 + j == qblk);
      uint32_t sr[64];
      tmem_ld_32x32b_x32(tS + lane_off + half * 64, *reinterpret_cast<uint32_t(*)[32]>(&sr[0]));
      tmem_ld_32x32b_x32(tS + lane_off + half * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&sr[32]));
      tmem_ld_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_free);        // S_j now lives in registers
      ATT_STAMP(2);
      if constexpr (MASKED) {
        // keys kbase + i of this thread; the warp takes the causal code when none of its rows needs a masked element
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
      } else if (diag) {
#pragma unroll
        for (int i = 0; i < 64; ++i)
          if (half * 64 + i > row) sr[i] = 0xff800000u;      // -inf
      }
      float mx4[4] = {m, m, m, m};
#pragma unroll
      for (int i = 0; i < 64; i += 4) {
        mx4[0] = fmaxf(mx4[0], __uint_as_float(sr[i]));
        mx4[1] = fmaxf(mx4[1], __uint_as_float(sr[i + 1]));
        mx4[2] = fmaxf(mx4[2], __uint_as_float(sr[i + 2]));
        mx4[3] = fmaxf(mx4[3], __uint_as_float(sr[i + 3]));
      }
      float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      // combine with the thread that owns the other 64 keys of this row
      red[(tg & 1) * 256 + half * 128 + row] = mx;
      named_bar_sync(2, SOFTMAX_THREADS);
      ATT_STAMP(3);
      mx = fmaxf(mx, red[(tg & 1) * 256 + (half ^ 1) * 128 + row]);
      // lazy rescaling: the reference point m only moves when the row maximum grew by more than 8 in the exp2 domain;
      // until then probabilities may exceed 1 (<= 2^8), which fp32 sums and bf16 P represent without trouble, and O / l
      // need no correction.  Both threads of a row see the same mx, so they take the same decision.
      if ((mx - m) * c <= 8.f) mx = m;
      float alpha = fast_exp2((m - mx) * c);         // m = -inf on the first tile -> 0
      float mc = mx * c;
      if constexpr (MASKED) {
        // every key of this row so far is masked: keep m = -inf, l = 0 and O = 0 (P is 0 up to the 2^-126 floor of the
        // polynomial, which the first allowed key's alpha = 0 wipes out) instead of -inf - -inf = NaN
        if (mx == -INFINITY) { alpha = 1.f; mc = 0.f; }
      }
      // p = exp2(s*c - m*c) with packed fp32x2 arithmetic (FFMA2 / FADD2).  Of every four elements two go through the
      // MUFU (ex2.approx) and two through a Cody-Waite + degree-3 polynomial on the FMA pipe, so both pipes work in
      // parallel (16384 exponentials per tile would otherwise keep the 16-lane MUFU busy for 1024 cycles per SM).
      uint32_t pk[32];
      const uint64_t c2 = pack2(c, c), nmc2 = pack2(-mc, -mc);
      uint64_t sum2a = pack2(0.f, 0.f), sum2b = pack2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 64; i += 4) {
        const uint64_t ya = ffma2(pack2u(sr[i], sr[i + 1]), c2, nmc2);
        const uint64_t yb = ffma2(pack2u(sr[i + 2], sr[i + 3]), c2, nmc2);
        float a0, a1;
        unpack2(ya, a0, a1);
        const uint64_t pa = pack2(fast_exp2(a0), fast_exp2(a1));      // MUFU pair (exp2(-inf) = 0 handles the mask)
        const uint64_t pb = poly_exp2x2(yb);                          // FMA-pipe pair (clamped at 2^-126)
        sum2a = fadd2(sum2a, pa);
        sum2b = fadd2(sum2b, pb);
        pk[i / 2] = cvt_bf16x2(pa);
        pk[i / 2 + 1] = cvt_bf16x2(pb);
      }
      {
        float s0, s1, s2, s3;
        unpack2(sum2a, s0, s1);
        unpack2(sum2b, s2, s3);
        l = l * alpha + ((s0 + s1) + (s2 + s3));
      }
      m = mx;
      ATT_STAMP(4);
      if (j > 0) {
        mbar_wait(o_done, (tg - 1) & 1);         // PV_{j-1} retired: O is stable, P may be overwritten
        tc_fence_after_sync();
        // rescale this thread's D/2 columns of the running output - skipped when no row of the warp moved its reference max
        if (!__all_sync(0xffffffffu, alpha == 1.f)) {
#pragma unroll
          for (int c = 0; c < NB; ++c) {
            uint32_t r[32];
            tmem_ld_32x32b_x32(tO + lane_off + half * (D / 2) + 32 * c, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
            tmem_st_32x32b_x32(tO + lane_off + half * (D / 2) + 32 * c, r);
          }
        }
      }
      ATT_STAMP(5);
      // P -> tensor memory: row == lane, this thread's 64 keys = 32 packed columns (the MMA reads A from TMEM)
      tmem_st_32x32b_x32(tP + lane_off + half * 32, pk);
      tmem_st_wait();
      ATT_STAMP(6);
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
      ATT_STAMP(7);
    }
    t0 += nkv;
    // ---- epilogue: total row sum = both halves
    named_bar_sync(2, SOFTMAX_THREADS);          // everyone is done reading the last tile's max exchange
    red[half * 128 + row] = l;
    named_bar_sync(2, SOFTMAX_THREADS);
    l += red[(half ^ 1) * 128 + row];
    mbar_wait(o_done, (t0 - 1) & 1);
    tc_fence_after_sync();
    const float inv_l = 1.f / l;
    uint8_t* stg = sOut;
#pragma unroll
    for (int c = 0; c < NB; ++c) {
      // this thread's columns half*D/2 + 32c .. +32: D = 64 - box 0, 16-byte units half*4 + u; D = 128 - box half, units 4c + u
      uint32_t r[32];
      tmem_ld_32x32b_x32(tO + lane_off + half * (D / 2) + 32 * c, r);
      tmem_ld_wait();
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int box = NB > 1 ? half : 0, unit = NB > 1 ? 4 * c + u : half * 4 + u;
        float f[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(r[u * 8 + i]) * inv_l;
        *reinterpret_cast<uint4*>(stg + box * TILE_BYTES + row * 128 + ((unit ^ (row & 7)) * 16)) = pack8(f);
      }
    }
    if (half == 0) p.lse[((size_t)b * p.Hq + h) * p.S + qblk * BQ + row] = (m * c + log2f(l)) * 0.6931471805599453f;
    fence_proxy_async_smem();
    named_bar_sync(1, SOFTMAX_THREADS);
    if (threadIdx.x == 64) {
#pragma unroll
      for (int c = 0; c < NB; ++c) tma_store_2d(&tmap_out, stg + c * TILE_BYTES, col_q + 64 * c, row0);
      tma_store_commit();
      tma_store_wait<0>();
    }
    }  // query tiles of this CTA
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}


// Mask description for the MASKED kernels (one CTA per row b; see ops/kernels.py::attn_mask_prep for the reference):
//   valid[t]  = mask[b, t] != 0                      docstart[s] = 1 + last p < s with ids[b, p] == eos (0 when eos < 0)
//   lo[s]     = min(s, first t >= docstart[s] with valid[t])
//   vbits[b, t/32] bit t%32 = valid[t]   kv_lo[b, qt] = min lo / 128   lo_hi[b, qt] = max lo   over query tile qt
//   q_hi[b, kt] = max{qt : kv_lo[b, qt] <= kt}
// Chunked scans: thread c owns positions [c*ch, (c+1)*ch); the chunk aggregates are scanned across the block.
constexpr int PREP_THREADS = 256;

template <bool MAX>
__device__ int block_scan_incl(int v, int* sh) {           // inclusive max / min scan in thread order
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v = MAX ? max(v, u) : min(v, u);
  }
  if (lane == 31) sh[warp] = v;
  __syncthreads();
  if (warp == 0) {
    int t = lane < PREP_THREADS / 32 ? sh[lane] : (MAX ? INT_MIN : INT_MAX);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t = MAX ? max(t, u) : min(t, u);
    }
    if (lane < PREP_THREADS / 32) sh[lane] = t;
  }
  __syncthreads();
  if (warp > 0) v = MAX ? max(v, sh[warp - 1]) : min(v, sh[warp - 1]);
  __syncthreads();
  return v;
}

__device__ __forceinline__ bool mask_valid(const uint8_t* mask, int esz, long long i) {
  if (mask == nullptr) return true;
  const uint8_t* e = mask + i * esz;
  uint8_t any = 0;
  for (int k = 0; k < esz; ++k) any |= e[k];
  return any != 0;
}

__global__ void __launch_bounds__(PREP_THREADS) attn_mask_prep_kernel(const long long* __restrict__ ids,
                                                                      const uint8_t* __restrict__ mask, int esz, int S,
                                                                      long long eos, int* __restrict__ lo,
                                                                      uint32_t* __restrict__ vbits, int* __restrict__ kv_lo,
                                                                      int* __restrict__ q_hi, int* __restrict__ lo_hi) {
  extern __shared__ int nv[];                                // [S] first valid position >= p (S when none)
  __shared__ int sh[32], agg[PREP_THREADS];
  int* t_min = nv + S;                                       // [nq] per query tile: min lo, max lo
  int* t_max = t_min + (S + 127) / 128;
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x, tid = threadIdx.x, nq = (S + 127) / 128, nw = (S + 31) / 32;
  const long long row = (long long)b * S;
  const int ch = (S + PREP_THREADS - 1) / PREP_THREADS;
  for (int q = tid; q < nq; q += PREP_THREADS) { t_min[q] = INT_MAX; t_max[q] = INT_MIN; }
  for (int w = tid; w < nw; w += PREP_THREADS) {
    uint32_t bits = 0;
    for (int k = 0; k < 32 && w * 32 + k < S; ++k) bits |= (uint32_t)mask_valid(mask, esz, row + w * 32 + k) << k;
    vbits[(long long)b * nw + w] = bits;
  }
  {  // suffix min of valid positions: thread tid owns chunk PREP_THREADS-1-tid, so a prefix scan over threads is a suffix scan
    const int c = PREP_THREADS - 1 - tid, p0 = min(S, c * ch), p1 = min(S, p0 + ch);
    int first = S;
    for (int p = p1 - 1; p >= p0; --p) if (mask_valid(mask, esz, row + p)) first = p;
    agg[tid] = block_scan_incl<false>(first, sh);
    __syncthreads();
    int cur = tid > 0 ? agg[tid - 1] : S;
    for (int p = p1 - 1; p >= p0; --p) {
      if (mask_valid(mask, esz, row + p)) cur = p;
      nv[p] = cur;
    }
  }
  __syncthreads();
  {  // prefix max of (last EOS + 1), then lo
    const int p0 = min(S, tid * ch), p1 = min(S, p0 + ch);
    int ds = 0;
    if (eos >= 0)
      for (int p = p0; p < p1; ++p) if (ids[row + p] == eos) ds = p + 1;
    agg[tid] = block_scan_incl<true>(ds, sh);
    __syncthreads();
    ds = tid > 0 ? agg[tid - 1] : 0;
    for (int p = p0; p < p1; ++p) {
      const int l = min(p, nv[ds]);
      lo[row + p] = l;
      atomicMin(&t_min[p / 128], l);
      atomicMax(&t_max[p / 128], l);
      if (eos >= 0 && ids[row + p] == eos) ds = p + 1;
    }
  }
  __syncthreads();
  for (int q = tid; q < nq; q += PREP_THREADS) {
    kv_lo[(long long)b * nq + q] = t_min[q] / 128;
    lo_hi[(long long)b * nq + q] = t_max[q];
  }
  for (int kt = tid; kt < nq; kt += PREP_THREADS) {
    int hi = kt;                                             // kv_lo[kt] <= kt always
    for (int q = nq - 1; q > kt; --q)
      if (t_min[q] / 128 <= kt) { hi = q; break; }
    q_hi[(long long)b * nq + kt] = hi;
  }
}
}  // namespace attn

namespace {
template <bool MASKED, int D>
int launch_attn_fwd(const void* qkv, void* out, void* lse, int B, int S, int Hq, int Hkv, long long ld_qkv, long long ld_out,
                    float softmax_scale, void* dbg, const int* lo, const uint32_t* vbits, const int* kv_lo, cudaStream_t st) {
  using namespace attn;
  constexpr int SMEM_BYTES = FwdCfg<D>::SMEM_BYTES;
  if (S % BQ || Hq % Hkv || ld_qkv % 8 || ld_out % 8) return -1;
  CUtensorMap tq, to;
  int rc;
  const long long T = (long long)B * S;
  if ((rc = make_tmap_2d(&tq, qkv, T, (Hq + 2 * Hkv) * D, ld_qkv * 2, 128, 64, 2))) return rc;
  if ((rc = make_tmap_2d(&to, out, T, Hq * D, ld_out * 2, 128, 64, 2))) return rc;
  Params p{};
  p.B = B; p.S = S; p.Hq = Hq; p.Hkv = Hkv;
  p.scale_log2 = softmax_scale * 1.4426950408889634f;
  p.lse = (float*)lse;
  p.dbg = (long long*)dbg;
  p.lo = lo; p.vbits = vbits; p.kv_lo = kv_lo;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_kernel<MASKED, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  dim3 grid((S / BQ + 1) / 2, Hq, B);
  launch_pdl(attn_fwd_kernel<MASKED, D>, grid, dim3(THREADS), SMEM_BYTES, st, tq, to, p);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}
}  // namespace

// qkv: [B*S, (Hq+2*Hkv)*64] bf16 (row stride ld_qkv elements); out: [B*S, Hq*64] bf16; lse: [B, Hq, S] fp32
ODB_EXPORT int odb_attn_fwd(const void* qkv, void* out, void* lse, int B, int S, int Hq, int Hkv, long long ld_qkv,
                            long long ld_out, float softmax_scale, void* dbg, cudaStream_t st) {
  return launch_attn_fwd<false, 64>(qkv, out, lse, B, S, Hq, Hkv, ld_qkv, ld_out, softmax_scale, dbg, nullptr, nullptr, nullptr, st);
}

// Same with a mask description (lo, vbits, kv_lo from odb_attn_mask_prep).
ODB_EXPORT int odb_attn_fwd_masked(const void* qkv, void* out, void* lse, int B, int S, int Hq, int Hkv, long long ld_qkv,
                                   long long ld_out, float softmax_scale, const void* lo, const void* vbits, const void* kv_lo,
                                   cudaStream_t st) {
  if (!lo || !vbits || !kv_lo) return -1;
  return launch_attn_fwd<true, 64>(qkv, out, lse, B, S, Hq, Hkv, ld_qkv, ld_out, softmax_scale, nullptr, (const int*)lo,
                                   (const uint32_t*)vbits, (const int*)kv_lo, st);
}

// Head size 128: qkv [B*S, (Hq+2*Hkv)*128], out [B*S, Hq*128]; otherwise the same arguments as odb_attn_fwd.
ODB_EXPORT int odb_attn_fwd_d128(const void* qkv, void* out, void* lse, int B, int S, int Hq, int Hkv, long long ld_qkv,
                                 long long ld_out, float softmax_scale, void* dbg, cudaStream_t st) {
  return launch_attn_fwd<false, 128>(qkv, out, lse, B, S, Hq, Hkv, ld_qkv, ld_out, softmax_scale, dbg, nullptr, nullptr, nullptr, st);
}

ODB_EXPORT int odb_attn_fwd_d128_masked(const void* qkv, void* out, void* lse, int B, int S, int Hq, int Hkv, long long ld_qkv,
                                        long long ld_out, float softmax_scale, const void* lo, const void* vbits, const void* kv_lo,
                                        cudaStream_t st) {
  if (!lo || !vbits || !kv_lo) return -1;
  return launch_attn_fwd<true, 128>(qkv, out, lse, B, S, Hq, Hkv, ld_qkv, ld_out, softmax_scale, nullptr, (const int*)lo,
                                    (const uint32_t*)vbits, (const int*)kv_lo, st);
}

// ids: int64 [B, S]; mask: optional [B, S] of any integer / bool type (mask_elem_bytes per element); eos < 0: no document
// masking.  Outputs (int32): lo [B*S], vbits [B, ceil(S/32)], kv_lo / q_hi / lo_hi [B, ceil(S/128)].
ODB_EXPORT int odb_attn_mask_prep(const void* ids, const void* mask, int mask_elem_bytes, int B, int S, long long eos, void* lo,
                                  void* vbits, void* kv_lo, void* q_hi, void* lo_hi, cudaStream_t st) {
  using namespace attn;
  if (B <= 0 || S <= 0 || (mask && mask_elem_bytes <= 0)) return -1;
  const size_t smem = ((size_t)S + 2 * ((S + 127) / 128)) * sizeof(int);
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_mask_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    smem_set = smem;
  }
  launch_pdl(attn_mask_prep_kernel, dim3(B), dim3(PREP_THREADS), smem, st, (const long long*)ids, (const uint8_t*)mask,
             mask_elem_bytes, S, eos, (int*)lo, (uint32_t*)vbits, (int*)kv_lo, (int*)q_hi, (int*)lo_hi);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}
