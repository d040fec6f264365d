// Flash attention forward + backward on tcgen05 / TMEM / TMA (sm_100a), head dimension 64.
//
// Layouts are chosen so that attention plugs between the QKV GEMM and the output projection with no
// transposes or copies:   qkv  : [B, S, 3, H, 64] bf16  (exactly the output of the fused QKV linear)
//                         out  : [B, S, H, 64]    bf16  (exactly the input of the projection linear)
//                         dqkv : [B, S, 3, H, 64] bf16  (exactly the upstream gradient of the QKV linear)
//
// Forward: one CTA per (128-query tile, head, batch).  Warp 0 = TMA producer (Q once, then a 2-stage K/V ring),
// warp 1 = single-thread tcgen05.mma issuer, warps 2-5 = softmax (one query row per thread).  Per 128-key tile:
//   S = Q K^T (TMEM, 128 cols) -> online softmax in registers (two tcgen05.ld passes: max, then exp2) -> P (bf16) into
//   swizzled shared memory -> O_t = P V (TMEM, 64 cols) -> O = O * alpha + O_t in registers.
// 113 KB of shared memory and 256 TMEM columns per CTA, so two CTAs share an SM and one CTA's softmax overlaps the
// other's MMAs.
//
// Backward: one CTA per (128-key tile, head, batch) looping over the query tiles that see it.  Five GEMMs per tile pair
// (S = Q K^T, dP = dO V^T, dV += P^T dO, dK += dS^T Q, dQ_t = dS K), all on tcgen05 with K-major or MN-major shared-
// memory descriptors over the *same* TMA-loaded tiles; dV/dK accumulate in TMEM across the loop, dQ tiles are reduced
// into fp32 buffers and summed once at the end.  Key tiles 2m and 2m+1 reduce into slot m of the buffer: a zeroed
// accumulator that receives exactly two fp32 adds ends with the same bits in either arrival order, and the final sum runs
// over the slots in a fixed order, so dQ is bitwise reproducible from run to run.  At most kDqGroupTiles key tiles run per
// launch; longer sequences take several launches, each folding its slots into a running fp32 total in slot order, so the
// scratch stays at most kDqGroupTiles / 2 + 1 dQ-sized fp32 buffers whatever the sequence length.
//
// The reference computes attention as unfused softmax(QK^T)V framework ops (examples/bert/modeling.py attention_layer).
#include "epl_common.cuh"
#include <algorithm>
#include <cstdio>

namespace epl {

constexpr int kD = 64;                  // head dimension
constexpr int kTile = 128;              // queries / keys per tile
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kNegBig = -1.0e30f;

EPL_DEVICE void tma_load_3d(void* smem_dst, const void* desc, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      :: "r"(smem_u32(smem_dst)), "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// 16 consecutive fp32 columns of this thread's TMEM lane
EPL_DEVICE void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}

// write 8 bf16 (one 16-byte chunk) of row `r`, logical chunk `c` (0..15) of a [128 x 128] bf16 tile stored as two
// 128B-swizzled atoms of [128 rows x 128 B]
EPL_DEVICE void st_swizzled_chunk(unsigned char* base, int r, int c, const uint32_t (&w)[4]) {
  unsigned char* p = base + (c >> 3) * (kTile * 128) + r * 128 + (((c & 7) ^ (r & 7)) << 4);
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

EPL_DEVICE float ex2_approx(float x) {            // bare MUFU.EX2 (exp2f() adds a denormal-range rescale: 3 extra instructions)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
EPL_DEVICE void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
         "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
EPL_DEVICE void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- softmax passes over this thread's 64 columns (one half) of one S tile row.  kMask: only tiles that touch the causal
// diagonal or the sequence end pay for the compare + select. -----------------------------------------------------------
template <bool kMask>
EPL_DEVICE float attn_half_max(const uint32_t (&v0)[32], const uint32_t (&v1)[32], int lim) {
  float m0 = kNegBig, m1 = kNegBig, m2 = kNegBig, m3 = kNegBig;
#pragma unroll
  for (int t = 0; t < 32; t += 4) {
    m0 = fmaxf(m0, (!kMask || t + 0 < lim) ? __uint_as_float(v0[t + 0]) : kNegBig);
    m1 = fmaxf(m1, (!kMask || t + 1 < lim) ? __uint_as_float(v0[t + 1]) : kNegBig);
    m2 = fmaxf(m2, (!kMask || t + 2 < lim) ? __uint_as_float(v0[t + 2]) : kNegBig);
    m3 = fmaxf(m3, (!kMask || t + 3 < lim) ? __uint_as_float(v0[t + 3]) : kNegBig);
  }
#pragma unroll
  for (int t = 0; t < 32; t += 4) {
    m0 = fmaxf(m0, (!kMask || t + 32 < lim) ? __uint_as_float(v1[t + 0]) : kNegBig);
    m1 = fmaxf(m1, (!kMask || t + 33 < lim) ? __uint_as_float(v1[t + 1]) : kNegBig);
    m2 = fmaxf(m2, (!kMask || t + 34 < lim) ? __uint_as_float(v1[t + 2]) : kNegBig);
    m3 = fmaxf(m3, (!kMask || t + 35 < lim) ? __uint_as_float(v1[t + 3]) : kNegBig);
  }
  return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
}

// 32 columns -> probabilities -> bf16 -> four 16-byte chunks of the swizzled P tile; returns their sum
template <bool kMask>
EPL_DEVICE float attn_exp_32(const uint32_t (&v)[32], int lim, float c, float mc, unsigned char* p_smem, int r, int chunk0) {
  float rs0 = 0.f, rs1 = 0.f, rs2 = 0.f, rs3 = 0.f;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float e[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const float x = ex2_approx(fmaf(__uint_as_float(v[g * 8 + t]), c, -mc));
      e[t] = (!kMask || g * 8 + t < lim) ? x : 0.f;
    }
    rs0 += e[0] + e[4]; rs1 += e[1] + e[5]; rs2 += e[2] + e[6]; rs3 += e[3] + e[7];
    uint32_t w[4];
#pragma unroll
    for (int q2 = 0; q2 < 4; ++q2) w[q2] = pack_bf16x2(e[2 * q2], e[2 * q2 + 1]);
    st_swizzled_chunk(p_smem, r, chunk0 + g, w);
  }
  return (rs0 + rs1) + (rs2 + rs3);
}

struct AttnParams {
  int B, S, H;
  float scale;            // 1/sqrt(D)
  int causal;
  __nv_bfloat16* out;     // fwd: [B,S,H,64]
  float* lse;             // [B,H,S]  (natural-log units)
  // backward only
  const float* delta;     // [B,H,S]  rowsum(dO * O)
  float* dq_acc;          // [slots,B,S,H,64] fp32, slot (kt-kt0)/2 zero on entry where key tile kt adds to it
  int kt0;                // first key tile of this launch (blockIdx.x = kt - kt0)
  __nv_bfloat16* dqkv;    // [B,S,3,H,64]
  long long* dbg;         // optional phase timestamps of CTA (0,0,0): [step][8] softmax warp 2, [64 + step][8] MMA thread
};

// ================================================================================================================
// forward
// ================================================================================================================
constexpr int kFwdThreads = 320;      // warp 0: TMA, warp 1: MMA, warps 2-9: softmax (two warps per TMEM lane quarter)

struct FwdSmem {
  static constexpr int kQ = 0;
  static constexpr int kK = kQ + kTile * 128;            // 2 stages
  static constexpr int kV = kK + 2 * kTile * 128;        // 2 stages
  static constexpr int kP = kV + 2 * kTile * 128;        // 32 KB
  static constexpr int kBar = kP + 2 * kTile * 128;
  static constexpr int kXm = kBar + 96;                  // bf16 [2 halves][128 rows]: row-max exchange between the two halves
  static constexpr int kTotal = kXm + 2 * kTile * 2;     // 115296 B: two CTAs per SM
};

// Softmax thread layout: query row r = quarter*32 + lane is shared by TWO threads (warps w and w+4 address the same TMEM
// lanes); thread `half` owns S columns [64*half, 64*half+64) and O columns [32*half, 32*half+32).  O accumulates in TMEM
// across the whole key loop (tcgen05 accumulate) and is only touched by the softmax threads when the running maximum
// moves by more than 2^8 (lazy rescale) — the common tile costs 2 TMEM loads, 64 max, 64 FFMA + 64 MUFU, 8 smem stores.
__global__ void __launch_bounds__(kFwdThreads, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const AttnParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bar_q = reinterpret_cast<uint64_t*>(smem + FwdSmem::kBar);
  uint64_t* kv_full = bar_q + 1;        // [2]
  uint64_t* kv_empty = kv_full + 2;     // [2]
  uint64_t* s_full = kv_empty + 2;
  uint64_t* p_ready = s_full + 1;
  uint64_t* o_full = p_ready + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q_tiles = (p.S + kTile - 1) / kTile;
  const int qt = q_tiles - 1 - (int)blockIdx.x;          // heaviest (causal) tiles first
  const int h = blockIdx.y, b = blockIdx.z;
  const int q0 = qt * kTile;
  const int n_kv = p.causal ? qt + 1 : q_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_qkv);
    mbar_init(bar_q, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
    mbar_init(s_full, 1); mbar_init(p_ready, 8); mbar_init(o_full, 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<256>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_s = tmem, tmem_o = tmem + 128;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(bar_q, kTile * 128);
      tma_load_3d(smem + FwdSmem::kQ, &map_qkv, bar_q, h * kD, q0, b);
      for (int j = 0; j < n_kv; ++j) {
        const int s = j & 1;
        mbar_wait(&kv_empty[s], ((j >> 1) & 1) ^ 1);
        mbar_expect_tx(&kv_full[s], 2 * kTile * 128);
        tma_load_3d(smem + FwdSmem::kK + s * kTile * 128, &map_qkv, &kv_full[s], (p.H + h) * kD, j * kTile, b);
        tma_load_3d(smem + FwdSmem::kV + s * kTile * 128, &map_qkv, &kv_full[s], (2 * p.H + h) * kD, j * kTile, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc_s = make_idesc_f16(kTile, kTile, 1, 0, 0);      // S = Q K^T : both K-major
      const uint32_t idesc_o = make_idesc_f16(kTile, kD, 1, 0, 1);         // O += P V  : A K-major, B (V) MN-major
      const uint32_t sq = smem_u32(smem + FwdSmem::kQ), sp = smem_u32(smem + FwdSmem::kP);
      mbar_wait(bar_q, 0);
      const bool stamp = p.dbg != nullptr && (blockIdx.x | blockIdx.y | blockIdx.z) == 0;
      for (int j = 0; j < n_kv; ++j) {
        const int s = j & 1;
        const uint32_t sk = smem_u32(smem + FwdSmem::kK + s * kTile * 128), sv = smem_u32(smem + FwdSmem::kV + s * kTile * 128);
        if (stamp) p.dbg[(64 + j) * 8 + 0] = clock64();
        mbar_wait(&kv_full[s], (j >> 1) & 1);
        tc_fence_after();
        if (stamp) p.dbg[(64 + j) * 8 + 1] = clock64();
        // S(j) = Q K(j)^T.  (S(j-1) has been consumed: p_ready(j-1) was awaited before P V(j-1) was issued.)
#pragma unroll
        for (int k = 0; k < kD / 16; ++k)
          umma_f16(tmem_s, make_smem_desc_sw128(sq + k * 32, 16, 1024), make_smem_desc_sw128(sk + k * 32, 16, 1024), idesc_s, k != 0);
        umma_commit(s_full);
        if (stamp) p.dbg[(64 + j) * 8 + 2] = clock64();
        // O += P(j) V(j) once the softmax warps have written P(j) (and rescaled O if the maximum moved)
        mbar_wait(p_ready, j & 1);
        tc_fence_after();
        if (stamp) p.dbg[(64 + j) * 8 + 3] = clock64();
#pragma unroll
        for (int kk = 0; kk < kTile / 16; ++kk) {
          const uint64_t da = make_smem_desc_sw128(sp + (kk >> 2) * (kTile * 128) + (kk & 3) * 32, 16, 1024);
          const uint64_t db = make_smem_desc_sw128(sv + kk * 2048, kTile * 128, 1024);
          umma_f16(tmem_o, da, db, idesc_o, (j | kk) != 0);
        }
        umma_commit(o_full);
        umma_commit(&kv_empty[s]);
        if (stamp) p.dbg[(64 + j) * 8 + 4] = clock64();
      }
    }
  } else {
    const int quarter = warp & 3, half = (warp - 2) >> 2;
    const int r = quarter * 32 + lane;                     // query row inside the tile
    const int qidx = q0 + r;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const uint32_t my_s = tmem_s + lane_addr + half * 64, my_o = tmem_o + lane_addr + half * 32;
    __nv_bfloat16* xm = reinterpret_cast<__nv_bfloat16*>(smem + FwdSmem::kXm);
    const float c = p.scale * kLog2e;
    float m = kNegBig, l = 0.f;
    const bool stamp = p.dbg != nullptr && warp == 2 && lane == 0 && (blockIdx.x | blockIdx.y | blockIdx.z) == 0;
    for (int j = 0; j < n_kv; ++j) {
      if (stamp) p.dbg[j * 8 + 0] = clock64();
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      if (stamp) p.dbg[j * 8 + 1] = clock64();
      uint32_t v0[32], v1[32];
      tmem_ld_32x32(my_s, v0);
      tmem_ld_32x32(my_s + 32, v1);
      const int k0 = j * kTile;
      const bool need_mask = (k0 + kTile > p.S) || (p.causal && j == qt);
      // columns [0, lim) of this thread's half are visible to this query row (branch-free: one compare + select each)
      const int lim = (need_mask ? min(p.S - k0, p.causal ? qidx - k0 + 1 : kTile) : kTile) - half * 64;
      tmem_ld_wait();
      if (stamp) p.dbg[j * 8 + 2] = clock64();
      float mx = need_mask ? attn_half_max<true>(v0, v1, lim) : attn_half_max<false>(v0, v1, lim);
      // both halves must agree on the maximum bit for bit: exchange it rounded to bf16 (any value near the true maximum
      // is a valid softmax offset)
      const __nv_bfloat16 mxb = __float2bfloat16_rn(mx);
      xm[half * kTile + r] = mxb;
      asm volatile("bar.sync %0, 64;" :: "r"(1 + quarter) : "memory");
      mx = fmaxf(__bfloat162float(mxb), __bfloat162float(xm[(half ^ 1) * kTile + r]));
      // lazy rescale: keep the old offset unless the maximum grew by more than 2^8 (P stays <= 256, exact enough in
      // bf16 / fp32 accumulation); the decision is made per warp because the TMEM accesses are warp-collective
      if (stamp) p.dbg[j * 8 + 3] = clock64();
      const bool grow = (mx - m) * c > 8.f;
      if (__any_sync(0xffffffffu, grow)) {
        const float m_new = grow ? mx : m;
        const float alpha = ex2_approx((m - m_new) * c);
        m = m_new;
        l *= alpha;
        if (j > 0) {
          mbar_wait(o_full, (j - 1) & 1);                  // P V(j-1) has landed in TMEM
          tc_fence_after();
#pragma unroll 1
          for (int ch = 0; ch < 2; ++ch) {                 // 16 columns at a time: the S registers stay live across this
            uint32_t o[16];
            tmem_ld_32x16(my_o + ch * 16, o);
            tmem_ld_wait();
#pragma unroll
            for (int t = 0; t < 16; ++t) o[t] = __float_as_uint(__uint_as_float(o[t]) * alpha);
            tmem_st_32x16(my_o + ch * 16, o);
          }
          tmem_st_wait();
        }
      }
      const float mc = m * c;
      if (stamp) p.dbg[j * 8 + 4] = clock64();
      float rowsum;
      if (need_mask) {
        rowsum = attn_exp_32<true>(v0, lim, c, mc, smem + FwdSmem::kP, r, half * 8);
        rowsum += attn_exp_32<true>(v1, lim - 32, c, mc, smem + FwdSmem::kP, r, half * 8 + 4);
      } else {
        rowsum = attn_exp_32<false>(v0, lim, c, mc, smem + FwdSmem::kP, r, half * 8);
        rowsum += attn_exp_32<false>(v1, lim - 32, c, mc, smem + FwdSmem::kP, r, half * 8 + 4);
      }
      l += rowsum;
      if (stamp) p.dbg[j * 8 + 5] = clock64();
      tc_fence_before();
      fence_proxy_async();                                 // generic-proxy smem writes -> visible to the UMMA (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(p_ready);
      if (stamp) p.dbg[j * 8 + 6] = clock64();
    }
    // epilogue: O / l -> bf16.  P is dead once the last P V has completed, so its storage carries the row-sum exchange.
    mbar_wait(o_full, (n_kv - 1) & 1);
    tc_fence_after();
    float* xl = reinterpret_cast<float*>(smem + FwdSmem::kP);
    xl[half * kTile + r] = l;
    uint32_t o[32];
    tmem_ld_32x32(my_o, o);
    asm volatile("bar.sync %0, 64;" :: "r"(1 + quarter) : "memory");
    l += xl[(half ^ 1) * kTile + r];
    tmem_ld_wait();
    if (qidx < p.S) {
      const float inv = 1.f / l;
      __nv_bfloat16* dst = p.out + (((size_t)b * p.S + qidx) * p.H + h) * kD + half * 32;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 w;
        w.x = pack_bf16x2(__uint_as_float(o[g * 8 + 0]) * inv, __uint_as_float(o[g * 8 + 1]) * inv);
        w.y = pack_bf16x2(__uint_as_float(o[g * 8 + 2]) * inv, __uint_as_float(o[g * 8 + 3]) * inv);
        w.z = pack_bf16x2(__uint_as_float(o[g * 8 + 4]) * inv, __uint_as_float(o[g * 8 + 5]) * inv);
        w.w = pack_bf16x2(__uint_as_float(o[g * 8 + 6]) * inv, __uint_as_float(o[g * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(dst + g * 8) = w;
      }
      if (half == 0) p.lse[((size_t)b * p.H + h) * p.S + qidx] = m * p.scale + logf(l);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<256>(tmem);
  }
}

// ================================================================================================================
// backward
// ================================================================================================================
// delta[b,h,s] = sum_d dO[b,s,h,d] * O[b,s,h,d].  Eight lanes per (b,s,h) row (16-byte loads), four rows per lane group in
// flight: 128 rows per 256-thread block.  (The one-warp-per-row version with 4-byte loads ran at a quarter of HBM speed.)
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o,
                                                          float* __restrict__ delta, int B, int S, int H) {
  const int64_t rows = (int64_t)B * S * H;
  const int sub = threadIdx.x & 7;                                   // 16-byte chunk of the 128-byte row
  const int64_t base = (int64_t)blockIdx.x * 128 + (threadIdx.x >> 3);
  uint4 a[4], g[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t row = base + u * 32;
    if (row < rows) {
      a[u] = *reinterpret_cast<const uint4*>(o + row * kD + sub * 8);
      g[u] = *reinterpret_cast<const uint4*>(d_o + row * kD + sub * 8);
    } else {
      a[u] = make_uint4(0, 0, 0, 0); g[u] = make_uint4(0, 0, 0, 0);
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const uint32_t aw[4] = {a[u].x, a[u].y, a[u].z, a[u].w}, gw[4] = {g[u].x, g[u].y, g[u].z, g[u].w};
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 af = unpack_bf16x2(aw[e]), gf = unpack_bf16x2(gw[e]);
      s = fmaf(af.x, gf.x, fmaf(af.y, gf.y, s));
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    const int64_t row = base + u * 32;
    if (sub == 0 && row < rows) {
      const int64_t bs = row / H;
      const int hh = (int)(row % H);
      const int64_t bb = bs / S, ss = bs % S;
      delta[(bb * H + hh) * S + ss] = s;
    }
  }
}

// dQ of one launch (key tiles kt0 ..): v = (first launch ? 0 : total) + slots 0, 1, ... in slot order; written as bf16 into
// dqkv after the last launch, else to the fp32 total.  8 elements per thread.  Causal: query tile i only received adds from
// key tiles kt0 .. i, i.e. from slots <= (i - kt0) / 2.
__global__ void __launch_bounds__(256) attn_dq_convert_kernel(const float* __restrict__ acc, float* __restrict__ dq_total,
                                                               __nv_bfloat16* __restrict__ dqkv, int64_t rows, int H, int S,
                                                               int causal, int slots, int kt0, int first, int last_launch) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // over rows * H * 8 chunks
  const int64_t total = rows * H * (kD / 8);
  if (i >= total) return;
  const int64_t row = i / (H * (kD / 8));
  const int rem = (int)(i % (H * (kD / 8)));
  const int hh = rem / (kD / 8), ch = rem % (kD / 8);
  const int qt = (int)(row % S) / kTile;
  const int last = !causal ? slots - 1 : (qt < kt0 ? -1 : min((qt - kt0) / 2, slots - 1));
  const int64_t off = (row * H + hh) * kD + ch * 8;
  const float* src = acc + off;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b2 = a;
  int m = 0;
  if (!first) {
    a = reinterpret_cast<const float4*>(dq_total + off)[0];
    b2 = reinterpret_cast<const float4*>(dq_total + off)[1];
  } else if (last >= 0) {
    a = reinterpret_cast<const float4*>(src)[0];
    b2 = reinterpret_cast<const float4*>(src)[1];
    m = 1;
  }
  for (; m <= last; ++m) {
    const float4 x = reinterpret_cast<const float4*>(src + (int64_t)m * rows * H * kD)[0];
    const float4 y = reinterpret_cast<const float4*>(src + (int64_t)m * rows * H * kD)[1];
    a.x += x.x; a.y += x.y; a.z += x.z; a.w += x.w;
    b2.x += y.x; b2.y += y.y; b2.z += y.z; b2.w += y.w;
  }
  if (!last_launch) {
    reinterpret_cast<float4*>(dq_total + off)[0] = a;
    reinterpret_cast<float4*>(dq_total + off)[1] = b2;
    return;
  }
  uint4 w;
  w.x = pack_bf16x2(a.x, a.y); w.y = pack_bf16x2(a.z, a.w); w.z = pack_bf16x2(b2.x, b2.y); w.w = pack_bf16x2(b2.z, b2.w);
  *reinterpret_cast<uint4*>(dqkv + (row * 3 * H + hh) * kD + ch * 8) = w;
}

struct BwdSmem {
  static constexpr int kK = 0;
  static constexpr int kV = kK + kTile * 128;
  static constexpr int kQ = kV + kTile * 128;            // 2 stages
  static constexpr int kDO = kQ + 2 * kTile * 128;       // 2 stages
  static constexpr int kP = kDO + 2 * kTile * 128;       // 32 KB
  static constexpr int kDS = kP + 2 * kTile * 128;       // 32 KB
  static constexpr int kDQ = kDS + 2 * kTile * 128;      // 32 KB fp32 [128 rows][64] staging for the TMA reduce-add of dQ
  static constexpr int kBar = kDQ + kTile * kD * 4;
  static constexpr int kTotal = kBar + 128;
};

// dQ tile (fp32, [128 x 64] plain row-major in shared memory) += into dq_acc[b, q0.., h*64..] with ONE TMA reduction
EPL_DEVICE void tma_reduce_add_3d(const void* desc, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
               :: "l"(desc), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// one dQ tile: TMEM -> (x scale) -> shared staging -> TMA reduce-add.  Replaces 8192 scalar fp32 atomics per tile pair.
// Called by all 256 compute threads; thread (row r, half) stages columns [32*half, 32*half+32).
EPL_DEVICE void flush_dq_tile(unsigned char* stage, uint32_t t_dq_lane, int r, int half, bool issuer, float scale,
                              const void* map_dq, int col0, int row0, int b) {
  if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // previous reduce has read the staging tile
  asm volatile("bar.sync 1, 256;" ::: "memory");
  // staging = two 128B-swizzled atoms of [128 rows x 32 fp32]; chunk g of row r lives at (g ^ (r & 7)) -> conflict-free stores
  {
    uint32_t v[32];
    tmem_ld_32x32(t_dq_lane + half * 32, v);
    tmem_ld_wait();
    unsigned char* rowp = stage + half * (kTile * 128) + r * 128;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      float4 w = make_float4(__uint_as_float(v[g * 4 + 0]) * scale, __uint_as_float(v[g * 4 + 1]) * scale,
                             __uint_as_float(v[g * 4 + 2]) * scale, __uint_as_float(v[g * 4 + 3]) * scale);
      *reinterpret_cast<float4*>(rowp + ((g ^ (r & 7)) << 4)) = w;
    }
  }
  fence_proxy_async();
  asm volatile("bar.sync 1, 256;" ::: "memory");
  if (issuer) {
    tma_reduce_add_3d(map_dq, stage, col0, row0, b);
    tma_reduce_add_3d(map_dq, stage + kTile * 128, col0 + 32, row0, b);
    tma_store_commit();
  }
}

constexpr int kBwdThreads = 320;      // warp 0: TMA, warp 1: MMA, warps 2-9: compute (two warps per TMEM lane quarter)

__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do,
                const __grid_constant__ CUtensorMap map_dq, const AttnParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bar_kv = reinterpret_cast<uint64_t*>(smem + BwdSmem::kBar);
  uint64_t* q_full = bar_kv + 1;       // [2]
  uint64_t* q_empty = q_full + 2;      // [2]
  uint64_t* sdp_full = q_empty + 2;
  uint64_t* pds_ready = sdp_full + 1;
  uint64_t* dq_full = pds_ready + 1;
  uint64_t* acc_full = dq_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles = (p.S + kTile - 1) / kTile;
  const int kt = p.kt0 + blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int k0 = kt * kTile;
  const int i_begin = p.causal ? kt : 0;
  const int n_q = tiles - i_begin;
  const int dq_slot_b = (blockIdx.x >> 1) * p.B + b;  // dQ goes to slot (kt-kt0)/2 (outer coordinate of the map: slot * B + b)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_qkv); tma_prefetch_desc(&map_do);
    mbar_init(bar_kv, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 1); }
    mbar_init(sdp_full, 1); mbar_init(pds_ready, 8); mbar_init(dq_full, 1); mbar_init(acc_full, 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t t_s = tmem, t_dp = tmem + 128, t_dv = tmem + 256, t_dk = tmem + 320, t_dq = tmem + 384;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(bar_kv, 2 * kTile * 128);
      tma_load_3d(smem + BwdSmem::kK, &map_qkv, bar_kv, (p.H + h) * kD, k0, b);
      tma_load_3d(smem + BwdSmem::kV, &map_qkv, bar_kv, (2 * p.H + h) * kD, k0, b);
      for (int n = 0; n < n_q; ++n) {
        const int s = n & 1, i = i_begin + n;
        mbar_wait(&q_empty[s], ((n >> 1) & 1) ^ 1);
        mbar_expect_tx(&q_full[s], 2 * kTile * 128);
        tma_load_3d(smem + BwdSmem::kQ + s * kTile * 128, &map_qkv, &q_full[s], h * kD, i * kTile, b);
        tma_load_3d(smem + BwdSmem::kDO + s * kTile * 128, &map_do, &q_full[s], h * kD, i * kTile, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t id_s = make_idesc_f16(kTile, kTile, 1, 0, 0);     // S, dP: K-major x K-major
      const uint32_t id_acc = make_idesc_f16(kTile, kD, 1, 1, 1);      // dV, dK: A^T (MN-major) x B (MN-major)
      const uint32_t id_dq = make_idesc_f16(kTile, kD, 1, 0, 1);       // dQ: dS (K-major) x K (MN-major)
      const uint32_t sk = smem_u32(smem + BwdSmem::kK), sv = smem_u32(smem + BwdSmem::kV);
      const uint32_t sp = smem_u32(smem + BwdSmem::kP), sds = smem_u32(smem + BwdSmem::kDS);
      mbar_wait(bar_kv, 0);
      for (int n = 0; n < n_q; ++n) {
        const int s = n & 1;
        const uint32_t sq = smem_u32(smem + BwdSmem::kQ + s * kTile * 128), sdo = smem_u32(smem + BwdSmem::kDO + s * kTile * 128);
        mbar_wait(&q_full[s], (n >> 1) & 1);       // (S / dP of the previous tile were consumed before pds_ready(n-1))
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < kD / 16; ++k) {
          umma_f16(t_s, make_smem_desc_sw128(sq + k * 32, 16, 1024), make_smem_desc_sw128(sk + k * 32, 16, 1024), id_s, k != 0);
          umma_f16(t_dp, make_smem_desc_sw128(sdo + k * 32, 16, 1024), make_smem_desc_sw128(sv + k * 32, 16, 1024), id_s, k != 0);
        }
        umma_commit(sdp_full);
        mbar_wait(pds_ready, n & 1);                        // P and dS are in shared memory
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < kTile / 16; ++kk) {
          // dV += P^T dO ; dK += dS^T Q   (contraction over the 128 queries: 16 rows per MMA)
          const uint64_t a_p = make_smem_desc_sw128(sp + kk * 2048, kTile * 128, 1024);
          const uint64_t a_ds = make_smem_desc_sw128(sds + kk * 2048, kTile * 128, 1024);
          const uint64_t b_do = make_smem_desc_sw128(sdo + kk * 2048, kTile * 128, 1024);
          const uint64_t b_q = make_smem_desc_sw128(sq + kk * 2048, kTile * 128, 1024);
          umma_f16(t_dv, a_p, b_do, id_acc, (n | kk) != 0);
          umma_f16(t_dk, a_ds, b_q, id_acc, (n | kk) != 0);
          // dQ_t = dS K   (contraction over the 128 keys)
          const uint64_t a_dsk = make_smem_desc_sw128(sds + (kk >> 2) * (kTile * 128) + (kk & 3) * 32, 16, 1024);
          const uint64_t b_k = make_smem_desc_sw128(sk + kk * 2048, kTile * 128, 1024);
          umma_f16(t_dq, a_dsk, b_k, id_dq, kk != 0);
        }
        umma_commit(dq_full);
        umma_commit(&q_empty[s]);
      }
      umma_commit(acc_full);
    }
  } else {
    const int quarter = warp & 3, half = (warp - 2) >> 2;
    const int r = quarter * 32 + lane;
    const bool issuer = warp == 2 && lane == 0;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const float c = p.scale * kLog2e;
    for (int n = 0; n < n_q; ++n) {
      const int i = i_begin + n;
      const int qidx = i * kTile + r;
      const bool q_ok = qidx < p.S;
      const float lse2 = q_ok ? p.lse[((size_t)b * p.H + h) * p.S + qidx] * kLog2e : 0.f;
      const float dlt = q_ok ? p.delta[((size_t)b * p.H + h) * p.S + qidx] : 0.f;
      const bool need_mask = (k0 + kTile > p.S) || (p.causal && i == kt) || !q_ok;
      // columns [0, lim) of this thread's 64-column half are visible to this query row
      const int lim0 = (!q_ok ? 0 : (need_mask ? min(p.S - k0, p.causal ? qidx - k0 + 1 : kTile) : kTile)) - half * 64;
      mbar_wait(sdp_full, n & 1);
      tc_fence_after();
      if (n > 0) {
        // dQ tile of the previous iteration -> fp32 accumulation buffer (also frees P / dS for rewriting)
        mbar_wait(dq_full, (n - 1) & 1);
        tc_fence_after();
        flush_dq_tile(smem + BwdSmem::kDQ, t_dq + lane_addr, r, half, issuer, p.scale, &map_dq, h * kD, (i - 1) * kTile, dq_slot_b);
      }
#pragma unroll 1
      for (int ch = 0; ch < 2; ++ch) {
        uint32_t sv_[32], dpv[32];
        tmem_ld_32x32(t_s + lane_addr + half * 64 + ch * 32, sv_);
        tmem_ld_32x32(t_dp + lane_addr + half * 64 + ch * 32, dpv);
        tmem_ld_wait();
        const int lim = lim0 - ch * 32;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t w[4], w2[4];
#pragma unroll
          for (int q2 = 0; q2 < 4; ++q2) {
            const int t = g * 8 + 2 * q2;
            float e0 = ex2_approx(fmaf(__uint_as_float(sv_[t]), c, -lse2)), e1 = ex2_approx(fmaf(__uint_as_float(sv_[t + 1]), c, -lse2));
            if (need_mask) {
              e0 = (t < lim) ? e0 : 0.f;
              e1 = (t + 1 < lim) ? e1 : 0.f;
            }
            w[q2] = pack_bf16x2(e0, e1);
            w2[q2] = pack_bf16x2(e0 * (__uint_as_float(dpv[t]) - dlt), e1 * (__uint_as_float(dpv[t + 1]) - dlt));
          }
          st_swizzled_chunk(smem + BwdSmem::kP, r, half * 8 + ch * 4 + g, w);
          st_swizzled_chunk(smem + BwdSmem::kDS, r, half * 8 + ch * 4 + g, w2);
        }
      }
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(pds_ready);
    }
    // last dQ tile
    {
      mbar_wait(dq_full, (n_q - 1) & 1);
      tc_fence_after();
      flush_dq_tile(smem + BwdSmem::kDQ, t_dq + lane_addr, r, half, issuer, p.scale, &map_dq, h * kD, (i_begin + n_q - 1) * kTile,
                    dq_slot_b);
    }
    if (issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all dQ reductions have landed
    // dK, dV of this key tile -> dqkv (row = key index): half 0 writes dV (slot 2), half 1 writes dK (slot 1)
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const int kidx = k0 + r;
    {
      const uint32_t src = half == 0 ? t_dv : t_dk;
      const float mul = half == 0 ? 1.f : p.scale;
      __nv_bfloat16* dst = p.dqkv + ((((size_t)b * p.S + kidx) * 3 + (half == 0 ? 2 : 1)) * p.H + h) * kD;
#pragma unroll 1
      for (int ch = 0; ch < 2; ++ch) {
        uint32_t v[32];
        tmem_ld_32x32(src + lane_addr + ch * 32, v);
        tmem_ld_wait();
        if (kidx < p.S) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint4 w;
            w.x = pack_bf16x2(__uint_as_float(v[g * 8 + 0]) * mul, __uint_as_float(v[g * 8 + 1]) * mul);
            w.y = pack_bf16x2(__uint_as_float(v[g * 8 + 2]) * mul, __uint_as_float(v[g * 8 + 3]) * mul);
            w.z = pack_bf16x2(__uint_as_float(v[g * 8 + 4]) * mul, __uint_as_float(v[g * 8 + 5]) * mul);
            w.w = pack_bf16x2(__uint_as_float(v[g * 8 + 6]) * mul, __uint_as_float(v[g * 8 + 7]) * mul);
            *reinterpret_cast<uint4*>(dst + ch * 32 + g * 8) = w;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
}

// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn attn_get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) != cudaSuccess || !sym) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}
// fp32 [B, S, cols], box {32, 128, 1}, 128B swizzle (TMA reduce-add target for dQ)
static int make_map_3d_f32(CUtensorMap* map, const void* ptr, uint64_t B, uint64_t S, uint64_t cols) {
  EncodeTiledFn enc = attn_get_encode();
  if (!enc) return -10;
  cuuint64_t dims[3] = {cols, S, B};
  cuuint64_t strides[2] = {cols * 4, S * cols * 4};
  cuuint32_t box[3] = {32, kTile, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r;
  EPL_ENCODE_RETRY(r, ptr, enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE));
  return r == CUDA_SUCCESS ? 0 : -11;
}

// [B, S, cols] bf16, box {64, 128, 1}
static int make_map_3d(CUtensorMap* map, const void* ptr, uint64_t B, uint64_t S, uint64_t cols) {
  EncodeTiledFn enc = attn_get_encode();
  if (!enc) return -10;
  cuuint64_t dims[3] = {cols, S, B};
  cuuint64_t strides[2] = {cols * 2, S * cols * 2};
  cuuint32_t box[3] = {kD, kTile, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r;
  EPL_ENCODE_RETRY(r, ptr, enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE));
  return r == CUDA_SUCCESS ? 0 : -11;
}

}  // namespace epl
using namespace epl;

static long long* g_attn_dbg = nullptr;
extern "C" void epl_attn_set_debug(void* ptr) { g_attn_dbg = (long long*)ptr; }

extern "C" int epl_attn_fwd(const void* qkv, void* out, void* lse, int B, int S, int H, float scale, int causal, void* stream) {
  CUtensorMap map;
  int rc = make_map_3d(&map, qkv, B, S, (uint64_t)3 * H * kD);
  if (rc) return rc;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdSmem::kTotal);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  AttnParams p{};
  p.B = B; p.S = S; p.H = H; p.scale = scale; p.causal = causal; p.out = (__nv_bfloat16*)out; p.lse = (float*)lse; p.dbg = g_attn_dbg;
  dim3 grid((S + kTile - 1) / kTile, H, B);
  attn_fwd_kernel<<<grid, kFwdThreads, FwdSmem::kTotal, (cudaStream_t)stream>>>(map, p);
  return EPL_CHECK_LAUNCH();
}

// dq_acc: fp32 [epl_attn_dq_slots(S),B,S,H,64] scratch (zeroed here where it is added to); delta: fp32 [B,H,S] scratch.
// One launch: ceil(tiles / 2) slots; several launches: kDqGroupTiles / 2 slots + the running total.
constexpr int kDqGroupTiles = 16;
extern "C" int epl_attn_dq_slots(int S) {
  const int tiles = (S + kTile - 1) / kTile;
  return tiles <= kDqGroupTiles ? (tiles + 1) / 2 : kDqGroupTiles / 2 + 1;
}

extern "C" int epl_attn_bwd(const void* qkv, const void* out, const void* d_out, const void* lse, void* delta, void* dq_acc,
                            void* dqkv, int B, int S, int H, float scale, int causal, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap map_qkv, map_do, map_dq;
  int rc = make_map_3d(&map_qkv, qkv, B, S, (uint64_t)3 * H * kD);
  if (rc) return rc;
  rc = make_map_3d(&map_do, d_out, B, S, (uint64_t)H * kD);
  if (rc) return rc;
  const int tiles = (S + kTile - 1) / kTile;
  const int slots = std::min((tiles + 1) / 2, kDqGroupTiles / 2);       // per launch; slot index `slots` holds the total
  rc = make_map_3d_f32(&map_dq, dq_acc, (uint64_t)slots * B, S, (uint64_t)H * kD);
  if (rc) return rc;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdSmem::kTotal);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  const int64_t rows = (int64_t)B * S * H;
  attn_delta_kernel<<<(int)((rows + 127) / 128), 256, 0, st>>>((const __nv_bfloat16*)out, (const __nv_bfloat16*)d_out, (float*)delta, B, S, H);
  const size_t row_bytes = (size_t)H * kD * sizeof(float);
  float* dq_total = (float*)dq_acc + (size_t)slots * B * S * H * kD;
  const int64_t chunks = (int64_t)B * S * H * (kD / 8);
  AttnParams p{};
  p.B = B; p.S = S; p.H = H; p.scale = scale; p.causal = causal; p.lse = (float*)const_cast<void*>(lse);
  p.delta = (const float*)delta; p.dq_acc = (float*)dq_acc; p.dqkv = (__nv_bfloat16*)dqkv;
  for (int kt0 = 0; kt0 < tiles; kt0 += kDqGroupTiles) {
    const int n_kt = std::min(kDqGroupTiles, tiles - kt0);
    for (int m = 0; m < (n_kt + 1) / 2; ++m) {         // causal: slot m is added to from query tile kt0 + 2m on
      const int r0 = causal ? std::min((kt0 + 2 * m) * kTile, S) : 0;
      char* base = (char*)dq_acc + ((size_t)m * B * S + r0) * row_bytes;
      if (r0 < S) cudaMemset2DAsync(base, (size_t)S * row_bytes, 0, (size_t)(S - r0) * row_bytes, B, st);
    }
    p.kt0 = kt0;
    attn_bwd_kernel<<<dim3(n_kt, H, B), kBwdThreads, BwdSmem::kTotal, st>>>(map_qkv, map_do, map_dq, p);
    attn_dq_convert_kernel<<<(int)((chunks + 255) / 256), 256, 0, st>>>((const float*)dq_acc, dq_total, (__nv_bfloat16*)dqkv,
                                                                         (int64_t)B * S, H, S, causal, (n_kt + 1) / 2, kt0,
                                                                         kt0 == 0, kt0 + kDqGroupTiles >= tiles);
  }
  return EPL_CHECK_LAUNCH();
}
