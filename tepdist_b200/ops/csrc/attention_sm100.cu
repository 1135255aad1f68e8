// Fused (flash) causal attention forward for sm_100a, head_dim 64, bf16.
//   S = Q K^T            tcgen05.mma  (A = Q  K-major, B = K  K-major)   -> TMEM (double buffered)
//   P = online softmax   8 softmax warps read S with tcgen05.ld (two threads per query row, 64 cols each)
//   O += P V             tcgen05.mma  (A = P  K-major from smem, B = V MN-major) -> TMEM -> registers
// Q/K/V are read straight out of the fused qkv projection buffer [B, S, H, 3, D] (heads-major) with 4-D TMA maps
// (no head-split transposes), O is written as [B, S, H, D] so it feeds the output projection GEMM.
// The reference gets attention from XLA-fused batched dots + softmax fusions (SURVEY Appendix C);
// this kernel is the B200-native replacement.
#include "sm100_ptx.cuh"
#include "launch.cuh"
#include <stdio.h>

using namespace sm100;

namespace {

inline bool exp_poly_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("TEPDIST_ATTN_EXP_POLY");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

inline bool fwd2_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("TEPDIST_ATTN_FWD2");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

constexpr int HD = 64;        // head dim
constexpr int BQ = 128;       // query rows per CTA
constexpr int BKV = 128;      // kv rows per iteration
constexpr int KV_STAGES = 3;
constexpr int SEG_MAX_BLOCKS = 2048;   // S <= 262144: the visited-block list lives in shared memory
constexpr int FWD_THREADS = 64 + 256;

constexpr int TILE_BYTES = 128 * HD * 2;  // 16 KB: a [128 x 64] bf16 tile (one SW128 chunk)
constexpr int SM_Q = 0;
constexpr int SM_K = SM_Q + TILE_BYTES;
constexpr int SM_V = SM_K + KV_STAGES * TILE_BYTES;
constexpr int SM_P = SM_V + KV_STAGES * TILE_BYTES;   // [128 x 128] bf16 = 2 chunks
constexpr int SM_BAR = SM_P + 2 * TILE_BYTES;
constexpr int SM_MAX = SM_BAR + 256;                  // float [2 iter parity][2 halves][128]
constexpr int FWD_SMEM = SM_MAX + 2 * 2 * 128 * 4 + 1024;
constexpr int SM_SEG_IDS = SM_MAX + 2 * 2 * 128 * 4;              // SEG: int [KV_STAGES][128] key ids
constexpr int SM_SEG_LIST = SM_SEG_IDS + KV_STAGES * 128 * 4;     // SEG: int visited count, then the list
constexpr int FWD_SEG_SMEM = SM_SEG_LIST + 16 + SEG_MAX_BLOCKS * 4 + 1024;

// Document masking (SEG = 1 instantiations).  Query i may attend to key j only if seg_q[i] == seg_k[j] (on top of the causal
// rule).  attn_seg_range_kernel first writes the [min, max] id of every 128-row block; a (query block, key block) pair whose
// intervals do not overlap is skipped, and inside a visited block the 128 key ids staged in shared memory next to K / V mask
// element-wise (skipped for rows whose document covers the whole key block).  Skipping is an optimisation only: any int32 ids
// give exact results.  Rows that see no key at all produce o = 0, lse = -inf.
struct AttnSeg {
  const int* seg_q;     // int32, row b at seg_q + b * stride
  const int* seg_k;
  const int2* rng_q;    // [B, S / 128] (min, max) of the query ids of each block
  const int2* rng_k;
  long long stride;
};

__device__ __forceinline__ bool seg_overlap(int2 a, int2 b) { return a.x <= b.y && b.x <= a.y; }

// 1-D bulk copy global -> shared, completing on an mbarrier (16-byte aligned, size a multiple of 16)
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// One warp per (batch row, 128-id block): out[b * nblk + blk] = (min, max).  blockIdx.y selects the query (0) or key (1) ids.
__global__ void __launch_bounds__(256) attn_seg_range_kernel(const AttnSeg sg, int2* rng_q, int2* rng_k, int B, int nblk) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  if (w >= B * nblk) return;
  const int b = w / nblk, blk = w % nblk;
  const int* src = (blockIdx.y ? sg.seg_k : sg.seg_q) + b * sg.stride + blk * 128;
  const int4 x = reinterpret_cast<const int4*>(src)[lane];
  int mn = min(min(x.x, x.y), min(x.z, x.w)), mx = max(max(x.x, x.y), max(x.z, x.w));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if (lane == 0) (blockIdx.y ? rng_k : rng_q)[w] = make_int2(mn, mx);
}

// Visited-block list of one CTA, built by one warp: list[k] = the k-th block c in [c0, c1) with seg_overlap(mine, rng[c]).
__device__ __forceinline__ int seg_visit_list(const int2* rng, int c0, int c1, int2 mine, int* list, int lane) {
  int n = 0;
  for (int base = c0; base < c1; base += 32) {
    const int c = base + lane;
    const bool vis = c < c1 && seg_overlap(mine, rng[c]);
    const unsigned m = __ballot_sync(0xffffffffu, vis);
    if (vis) list[n + __popc(m & ((1u << lane) - 1u))] = c;
    n += __popc(m);
  }
  return n;
}

struct AttnFwdParams {
  void* O;      // bf16 [B, S, H, D]
  float* lse;   // fp32 [B, H, S]   (natural-log domain, scaled scores)
  int B, H, S, causal;
  float scale_log2;  // softmax scale * log2(e)
  float scale;
};

// 2^x on the FMA / ALU pipes (no MUFU): round-to-nearest split x = n + f with the 1.5 * 2^23 magic constant, degree-4
// polynomial for 2^f on [-0.5, 0.5] (rel. error 4e-5, below bf16 resolution), exponent spliced in with integer adds.
// The softmax of D = 64 attention is MUFU-bound (16 ex2 / clk / SM vs 128 FMA lanes): evaluating every second exponential
// this way (POLY = 1 instantiations, TEPDIST_ATTN_EXP_POLY=1) trades 1 MUFU op for ~8 FMA / ALU ops on idle pipes.
__device__ __forceinline__ float exp2_poly(float x) {
  x = fmaxf(x, -125.f);
  const float magic = 12582912.f;
  const float t = x + magic;
  const float f = x - (t - magic);
  float p = fmaf(0.0096181291f, f, 0.0555041087f);
  p = fmaf(p, f, 0.2402265070f);
  p = fmaf(p, f, 0.6931471806f);
  p = fmaf(p, f, 1.0f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int POLY, int SEG>
__global__ void __launch_bounds__(FWD_THREADS, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                const __grid_constant__ CUtensorMap tmap_v, const AttnFwdParams p, const AttnSeg sg) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* kv_full = bars + 1;               // [3]
  uint64_t* kv_empty = bars + 4;              // [3]
  uint64_t* s_full = bars + 7;                // [2]
  uint64_t* s_empty = bars + 9;               // [2]
  uint64_t* p_full = bars + 11;
  uint64_t* pv_full = bars + 12;
  uint64_t* pv_empty = bars + 13;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);
  float* smax = reinterpret_cast<float*>(smem + SM_MAX);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = p.S / BQ;
  const int BH = p.B * p.H;
  const int qb = nq - 1 - (int)(blockIdx.x / BH);  // heavy (long) rows first
  const int bh = blockIdx.x % BH;
  const int b = bh / p.H, h = bh % p.H;
  int n_kv = p.causal ? (qb + 1) : (p.S / BKV);
  int* seg_ids = reinterpret_cast<int*>(smem + SM_SEG_IDS);
  int* seg_list = reinterpret_cast<int*>(smem + SM_SEG_LIST) + 4;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
    mbar_init(q_full, 1);
    for (int i = 0; i < KV_STAGES; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], 8); }
    mbar_init(p_full, 8);
    mbar_init(pv_full, 1);
    mbar_init(pv_empty, 8);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();      // (launch.cuh) the prologue above ran under the previous kernel's tail
  pdl_trigger();
  if (SEG) {         // every role walks the same list of key blocks whose id interval meets the query block's
    if (warp == 2) {
      const int nv = seg_visit_list(sg.rng_k + (size_t)b * nq, 0, n_kv, sg.rng_q[(size_t)b * nq + qb], seg_list, lane);
      if (lane == 0) seg_list[-1] = nv;
    }
    __syncthreads();
    n_kv = seg_list[-1];
  }
  const uint32_t TM_S = tmem_base;          // 2 x 128 columns
  const uint32_t TM_PV = tmem_base + 256;   // 64 columns

  if (warp == 0) {
    if (elect_one()) {
      if (!SEG || n_kv > 0) {
        mbar_expect_tx(q_full, TILE_BYTES);
        tma_load_4d(smem + SM_Q, &tmap_q, q_full, 0, qb * BQ, h, b);
      }
      for (int j = 0; j < n_kv; ++j) {
        const int st = j % KV_STAGES;
        const uint32_t ph = (j / KV_STAGES) & 1;
        const int jb = SEG ? seg_list[j] : j;
        mbar_wait(&kv_empty[st], ph ^ 1);
        mbar_expect_tx(&kv_full[st], 2 * TILE_BYTES + (SEG ? BKV * 4 : 0));
        tma_load_4d(smem + SM_K + st * TILE_BYTES, &tmap_k, &kv_full[st], 0, jb * BKV, h, b);
        tma_load_4d(smem + SM_V + st * TILE_BYTES, &tmap_v, &kv_full[st], 0, jb * BKV, h, b);
        if (SEG) bulk_load(seg_ids + st * BKV, sg.seg_k + b * sg.stride + jb * BKV, BKV * 4, &kv_full[st]);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc(UMMA_BF16, UMMA_BF16, 128, 128, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc(UMMA_BF16, UMMA_BF16, 128, 64, 0, 1);
      const uint32_t sq = smem_u32(smem + SM_Q);
      const uint32_t sp = smem_u32(smem + SM_P);
      auto issue_s = [&](int j) {
        const int st = j % KV_STAGES;
        mbar_wait(&kv_full[st], (j / KV_STAGES) & 1);
        if (j >= 2) mbar_wait(&s_empty[j & 1], ((j - 2) >> 1) & 1);
        tc_fence_after();
        const uint32_t sk = smem_u32(smem + SM_K + st * TILE_BYTES);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k) {
          umma_f16_ss(TM_S + (j & 1) * 128, make_smem_desc_sw128(sq + k * 32, 0, 1024),
                      make_smem_desc_sw128(sk + k * 32, 0, 1024), idesc_s, k > 0 ? 1u : 0u);
        }
        umma_commit(&s_full[j & 1]);
      };
      if (!SEG || n_kv > 0) {
        mbar_wait(q_full, 0);
        issue_s(0);
      }
      for (int j = 0; j < n_kv; ++j) {
        if (j + 1 < n_kv) issue_s(j + 1);
        mbar_wait(p_full, j & 1);
        if (j > 0) mbar_wait(pv_empty, (j - 1) & 1);
        tc_fence_after();
        const uint32_t sv = smem_u32(smem + SM_V + (j % KV_STAGES) * TILE_BYTES);
#pragma unroll
        for (int k = 0; k < BKV / 16; ++k) {
          umma_f16_ss(TM_PV, make_smem_desc_sw128(sp + (k >> 2) * TILE_BYTES + (k & 3) * 32, 0, 1024),
                      make_smem_desc_sw128(sv + k * 2048, TILE_BYTES, 1024), idesc_pv, k > 0 ? 1u : 0u);
        }
        umma_commit(pv_full);
        umma_commit(&kv_empty[j % KV_STAGES]);
      }
    }
  } else {
    // ===================== softmax / correction / epilogue: 8 warps =====================
    const int sw = warp - 2;             // 0..7
    const int quarter = warp & 3;        // TMEM lane quarter this warp may access
    const int half = (sw >= 4) ? 1 : 0;  // hmm: warps 2..5 -> half 0 ; 6..9 -> half 1
    const int row = quarter * 32 + lane; // query row within the tile (== TMEM lane)
    const int q_global = qb * BQ + row;
    const uint32_t lane_addr = uint32_t(quarter * 32) << 16;
    float m_run = -INFINITY, l_run = 0.f, alpha_prev = 1.f;
    float o[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) o[i] = 0.f;
    const int my_seg = SEG ? sg.seg_q[b * sg.stride + q_global] : 0;

    for (int j = 0; j < n_kv; ++j) {
      mbar_wait(&s_full[j & 1], (j >> 1) & 1);
      tc_fence_after();
      uint32_t r0[32], r1[32];
      tmem_ld_32x32(TM_S + lane_addr + (j & 1) * 128 + half * 64, r0);
      tmem_ld_32x32(TM_S + lane_addr + (j & 1) * 128 + half * 64 + 32, r1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_empty[j & 1]);

      float s[64];
#pragma unroll
      for (int i = 0; i < 32; ++i) { s[i] = __uint_as_float(r0[i]); s[32 + i] = __uint_as_float(r1[i]); }
      const int jb = SEG ? seg_list[j] : j;
      const int col0 = jb * BKV + half * 64;
      if (p.causal && jb == qb) {
#pragma unroll
        for (int i = 0; i < 64; ++i) if (col0 + i > q_global) s[i] = -INFINITY;
      }
      if (SEG) {
        const int2 kr = sg.rng_k[(size_t)b * nq + jb];
        if (!(kr.x == my_seg && kr.y == my_seg)) {   // the key block is not all of this row's document: compare ids
          mbar_wait(&kv_full[j % KV_STAGES], (j / KV_STAGES) & 1);   // (complete already: S(j) was computed from this stage)
          const int4* ids = reinterpret_cast<const int4*>(seg_ids + (j % KV_STAGES) * BKV + half * 64);
#pragma unroll
          for (int g = 0; g < 16; ++g) {
            const int4 id = ids[g];
            if (id.x != my_seg) s[4 * g + 0] = -INFINITY;
            if (id.y != my_seg) s[4 * g + 1] = -INFINITY;
            if (id.z != my_seg) s[4 * g + 2] = -INFINITY;
            if (id.w != my_seg) s[4 * g + 3] = -INFINITY;
          }
        }
      }
      float mx = -INFINITY;
#pragma unroll
      for (int i = 0; i < 64; ++i) mx = fmaxf(mx, s[i]);
      float* mbuf = smax + (j & 1) * 256;
      mbuf[half * 128 + row] = mx;
      named_bar_sync(1, 256);
      mx = fmaxf(mx, mbuf[(1 - half) * 128 + row]);
      const float m_new = fmaxf(m_run, mx);
      // SEG: a row that has seen no key yet keeps m = -inf; a finite stand-in keeps alpha and P at exact zeros instead of NaN
      const float m_ref = (SEG && m_new == -INFINITY) ? 0.f : m_new;
      const float alpha = exp2f((m_run - m_ref) * p.scale_log2);  // m_run = -inf -> 0
      const float mb = m_ref * p.scale_log2;
      float lsum = 0.f;
      uint32_t pk[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float p0 = exp2f(fmaf(s[2 * i], p.scale_log2, -mb));
        const float x1 = fmaf(s[2 * i + 1], p.scale_log2, -mb);
        const float p1 = POLY ? exp2_poly(x1) : exp2f(x1);
        lsum += p0 + p1;
        pk[i] = pack_bf16x2(p0, p1);
      }
      l_run = l_run * alpha + lsum;
      m_run = m_new;

      if (j > 0) {  // fold in the previous P V product (also guarantees P smem is free again)
        mbar_wait(pv_full, (j - 1) & 1);
        tc_fence_after();
        uint32_t pv[32];
        tmem_ld_32x32(TM_PV + lane_addr + half * 32, pv);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pv_empty);
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = fmaf(o[i], alpha_prev, __uint_as_float(pv[i]));
      }
      alpha_prev = alpha;

      // P (bf16) -> smem, SW128 K-major: chunk = half, row-major 128 B rows, 16 B granules XOR (row & 7)
      uint8_t* prow = smem + SM_P + half * TILE_BYTES + row * 128;
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        uint4 u = make_uint4(pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
        *reinterpret_cast<uint4*>(prow + ((g ^ (row & 7)) << 4)) = u;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
    }
    // last P V product
    if (!SEG || n_kv > 0) {
      mbar_wait(pv_full, (n_kv - 1) & 1);
      tc_fence_after();
      uint32_t pv[32];
      tmem_ld_32x32(TM_PV + lane_addr + half * 32, pv);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; ++i) o[i] = fmaf(o[i], alpha_prev, __uint_as_float(pv[i]));
    }
    // combine the two halves' row sums
    float* lbuf = smax;  // reuse (all max exchanges are complete after this barrier)
    named_bar_sync(1, 256);
    lbuf[half * 128 + row] = l_run;
    named_bar_sync(1, 256);
    const float l_tot = l_run + lbuf[(1 - half) * 128 + row];
    const float inv = (SEG && l_tot == 0.f) ? 0.f : 1.f / l_tot;
    __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(p.O) +
                          (((size_t)b * p.S + q_global) * p.H + h) * HD + half * 32;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      uint4 u;
      u.x = pack_bf16x2(o[8 * g + 0] * inv, o[8 * g + 1] * inv);
      u.y = pack_bf16x2(o[8 * g + 2] * inv, o[8 * g + 3] * inv);
      u.z = pack_bf16x2(o[8 * g + 4] * inv, o[8 * g + 5] * inv);
      u.w = pack_bf16x2(o[8 * g + 6] * inv, o[8 * g + 7] * inv);
      reinterpret_cast<uint4*>(orow)[g] = u;
    }
    if (half == 0)
      p.lse[((size_t)b * p.H + h) * p.S + q_global] = (SEG && l_tot == 0.f) ? -INFINITY : m_run * p.scale + __logf(l_tot);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}


// =====================================================================================================
// Forward, two query tiles per CTA (EXPERIMENTAL, TEPDIST_ATTN_FWD2=1; not yet run on hardware).
//
// The kernel above is bound by the softmax, not by the tensor pipe: 128 x 128 exponentials per KV block at 16 MUFU / clk /
// SM are 1024 clk, and its 8 softmax warps all walk the same phases (TMEM load, row max, exchange, exp, fold, store) in
// lock-step, so the MUFU pipe idles about half of the time.  Here one CTA owns TWO 128-row query tiles (A, B) that share
// every K / V stage; each tile has its own 4 softmax warps (one thread per query row: no cross-warp max exchange), its own
// S accumulator (single-buffered) and its own O accumulator in TMEM.  The MMA warp serves the tiles alternately
// (PV_A(j), S_A(j+1), PV_B(j), S_B(j+1), ...), so while tile A waits for its next S the MUFU pipe works on tile B.
// O stays in TMEM across KV blocks (PV accumulates); the running maximum is only a REFERENCE that is raised -- and O / l
// rescaled in place with tcgen05.ld / st -- when the block maximum exceeds it by more than 2^8 (exact: every P of a row is
// relative to the same reference at the end, nothing overflows below 2^8).
// TMEM: S_A [0,128) S_B [128,256) O_A [256,320) O_B [320,384).  smem: Q_A Q_B | K x3 | V x3 | P_A P_B = 192 KB.
// =====================================================================================================
constexpr int F2_THREADS = 64 + 256;
constexpr int F2_Q = 0;                                   // 2 tiles
constexpr int F2_K = F2_Q + 2 * TILE_BYTES;
constexpr int F2_V = F2_K + KV_STAGES * TILE_BYTES;
constexpr int F2_P = F2_V + KV_STAGES * TILE_BYTES;       // 2 tiles x 2 chunks
constexpr int F2_BAR = F2_P + 4 * TILE_BYTES;
constexpr int F2_SMEM = F2_BAR + 256 + 1024;

__global__ void __launch_bounds__(F2_THREADS, 1)
attn_fwd2_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                 const __grid_constant__ CUtensorMap tmap_v, const AttnFwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + F2_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* kv_full = bars + 1;     // [3]
  uint64_t* kv_empty = bars + 4;    // [3]
  uint64_t* s_full = bars + 7;      // [2] per tile
  uint64_t* s_empty = bars + 9;     // [2]
  uint64_t* p_full = bars + 11;     // [2]
  uint64_t* pv_full = bars + 13;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 15);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq2 = p.S / 256;
  const int BH = p.B * p.H;
  const int qb2 = nq2 - 1 - (int)(blockIdx.x / BH);   // heavy rows first
  const int bh = blockIdx.x % BH;
  const int b = bh / p.H, h = bh % p.H;
  const int nkv_t[2] = {p.causal ? 2 * qb2 + 1 : p.S / BKV, p.causal ? 2 * qb2 + 2 : p.S / BKV};
  const int nkv = nkv_t[1];

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
    mbar_init(q_full, 1);
    for (int i = 0; i < KV_STAGES; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_full[t], 1);
      mbar_init(&s_empty[t], 4);
      mbar_init(&p_full[t], 4);
      mbar_init(&pv_full[t], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(q_full, 2 * TILE_BYTES);
      tma_load_4d(smem + F2_Q, &tmap_q, q_full, 0, qb2 * 256, h, b);
      tma_load_4d(smem + F2_Q + TILE_BYTES, &tmap_q, q_full, 0, qb2 * 256 + 128, h, b);
      for (int j = 0; j < nkv; ++j) {
        const int st = j % KV_STAGES;
        mbar_wait(&kv_empty[st], ((j / KV_STAGES) & 1) ^ 1);
        mbar_expect_tx(&kv_full[st], 2 * TILE_BYTES);
        tma_load_4d(smem + F2_K + st * TILE_BYTES, &tmap_k, &kv_full[st], 0, j * BKV, h, b);
        tma_load_4d(smem + F2_V + st * TILE_BYTES, &tmap_v, &kv_full[st], 0, j * BKV, h, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc(UMMA_BF16, UMMA_BF16, 128, 128, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc(UMMA_BF16, UMMA_BF16, 128, 64, 0, 1);
      auto issue_s = [&](int t, int j) {     // S_t(j) = Q_t K(j)^T ; needs K stage j and the tile's S buffer drained
        const int st = j % KV_STAGES;
        mbar_wait(&kv_full[st], (j / KV_STAGES) & 1);
        if (j > 0) mbar_wait(&s_empty[t], (j - 1) & 1);
        tc_fence_after();
        const uint32_t sq = smem_u32(smem + F2_Q + t * TILE_BYTES);
        const uint32_t sk = smem_u32(smem + F2_K + st * TILE_BYTES);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
          umma_f16_ss(tmem_base + t * 128, make_smem_desc_sw128(sq + k * 32, 0, 1024), make_smem_desc_sw128(sk + k * 32, 0, 1024),
                      idesc_s, k > 0 ? 1u : 0u);
        umma_commit(&s_full[t]);
      };
      auto issue_pv = [&](int t, int j) {    // O_t += P_t(j) V(j)
        mbar_wait(&p_full[t], j & 1);
        tc_fence_after();
        const uint32_t sp = smem_u32(smem + F2_P + t * 2 * TILE_BYTES);
        const uint32_t sv = smem_u32(smem + F2_V + (j % KV_STAGES) * TILE_BYTES);
#pragma unroll
        for (int k = 0; k < BKV / 16; ++k)
          umma_f16_ss(tmem_base + 256 + t * 64, make_smem_desc_sw128(sp + (k >> 2) * TILE_BYTES + (k & 3) * 32, 0, 1024),
                      make_smem_desc_sw128(sv + k * 2048, TILE_BYTES, 1024), idesc_pv, (j > 0 || k > 0) ? 1u : 0u);
        umma_commit(&pv_full[t]);
      };
      mbar_wait(q_full, 0);
      issue_s(0, 0);
      issue_s(1, 0);
      for (int j = 0; j < nkv; ++j) {
        for (int t = 0; t < 2; ++t) {
          if (j < nkv_t[t]) {
            issue_pv(t, j);
            if (j + 1 < nkv_t[t]) issue_s(t, j + 1);
          }
        }
        umma_commit(&kv_empty[j % KV_STAGES]);   // every MMA that reads stage j has been issued
      }
    }
  } else {
    // ===================== softmax: warps 2-5 tile A, warps 6-9 tile B; one thread per query row =====================
    const int t = (warp - 2) >> 2;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int q_global = qb2 * 256 + t * 128 + row;
    const uint32_t lane_addr = uint32_t(quarter * 32) << 16;
    const uint32_t TM_S = tmem_base + lane_addr + t * 128;
    const uint32_t TM_O = tmem_base + lane_addr + 256 + t * 64;
    const int n_mine = nkv_t[t];
    float m_ref = -INFINITY, l_run = 0.f;
    for (int j = 0; j < n_mine; ++j) {
      mbar_wait(&s_full[t], j & 1);
      tc_fence_after();
      const bool diag = p.causal && j == n_mine - 1;
      // ---- pass 1: row maximum
      float mx = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(TM_S + c * 32, r);
        tmem_ld_wait();
        const int col0 = j * BKV + c * 32;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float v = __uint_as_float(r[i]);
          if (diag && col0 + i > q_global) v = -INFINITY;
          mx = fmaxf(mx, v);
        }
      }
      // ---- reference maximum: raise it (and rescale O, l) only when the block exceeds it by more than 2^8
      float alpha = 1.f;
      bool raise = false;
      if (j == 0) {
        m_ref = mx;
      } else if ((mx - m_ref) * p.scale_log2 > 8.f) {
        alpha = exp2f((m_ref - mx) * p.scale_log2);
        raise = true;
      }
      if (j > 0) {   // PV(j-1) done: the P buffer may be overwritten and O is stable
        mbar_wait(&pv_full[t], (j - 1) & 1);
        tc_fence_after();
      }
      if (__any_sync(0xffffffffu, raise)) {   // tcgen05.ld / st are warp-collective: lanes that keep their reference use alpha = 1
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          uint32_t r[32];
          tmem_ld_32x32(TM_O + c * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
          tmem_st_32x32(TM_O + c * 32, r);
        }
        tmem_st_wait();
        if (raise) { l_run *= alpha; m_ref = mx; }
      }
      const float mb = m_ref * p.scale_log2;
      // ---- pass 2: P = 2^(s*c - mb) -> bf16 -> smem (SW128 K-major, chunk = 64 columns), row sum
      float lsum = 0.f;
      uint8_t* prow = smem + F2_P + t * 2 * TILE_BYTES + row * 128;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t r[32];
        tmem_ld_32x32(TM_S + c * 32, r);
        tmem_ld_wait();
        if (c == 3) {   // S fully consumed: the MMA warp may overwrite it with S(j+1)
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&s_empty[t]);
        }
        const int col0 = j * BKV + c * 32;
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float v0 = __uint_as_float(r[2 * i]), v1 = __uint_as_float(r[2 * i + 1]);
          if (diag && col0 + 2 * i > q_global) v0 = -INFINITY;
          if (diag && col0 + 2 * i + 1 > q_global) v1 = -INFINITY;
          const float p0 = exp2f(fmaf(v0, p.scale_log2, -mb));
          const float p1 = exp2f(fmaf(v1, p.scale_log2, -mb));
          lsum += p0 + p1;
          pk[i] = pack_bf16x2(p0, p1);
        }
        uint8_t* pc = prow + (c >> 1) * TILE_BYTES;     // columns 0-63 -> chunk 0, 64-127 -> chunk 1
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int gran = (c & 1) * 4 + g;              // 16-byte granule inside the 128-byte row
          *reinterpret_cast<uint4*>(pc + ((gran ^ (row & 7)) << 4)) = make_uint4(pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
        }
      }
      l_run += lsum;
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[t]);
    }
    // ---- epilogue: O / l
    mbar_wait(&pv_full[t], (n_mine - 1) & 1);
    tc_fence_after();
    const float inv = 1.f / l_run;
    __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(p.O) + (((size_t)b * p.S + q_global) * p.H + h) * HD;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      uint32_t r[32];
      tmem_ld_32x32(TM_O + c * 32, r);
      tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 u;
        u.x = pack_bf16x2(__uint_as_float(r[8 * g + 0]) * inv, __uint_as_float(r[8 * g + 1]) * inv);
        u.y = pack_bf16x2(__uint_as_float(r[8 * g + 2]) * inv, __uint_as_float(r[8 * g + 3]) * inv);
        u.z = pack_bf16x2(__uint_as_float(r[8 * g + 4]) * inv, __uint_as_float(r[8 * g + 5]) * inv);
        u.w = pack_bf16x2(__uint_as_float(r[8 * g + 6]) * inv, __uint_as_float(r[8 * g + 7]) * inv);
        reinterpret_cast<uint4*>(orow + c * 32)[g] = u;
      }
    }
    p.lse[((size_t)b * p.H + h) * p.S + q_global] = m_ref * p.scale + __logf(l_run);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// =====================================================================================================
// Backward.  One CTA per (kv block j, batch, head); loops over query blocks i (>= j when causal).
//   S  = Q K^T, dP = dO V^T                (tcgen05, TMEM)
//   P  = exp2(S*c - lse), dS = P * (dP - delta)      (8 compute warps, two threads per query row)
//   dV += P^T dO, dK += dS^T Q             (A operands are MN-major views of the P / dS smem tiles)
//   dQ  = dS K  -> fp32 red.add into dq_acc (summed over kv blocks by different CTAs)
// =====================================================================================================
constexpr int BWD_THREADS = 64 + 256;
constexpr int SB_K = 0;
constexpr int SB_V = SB_K + TILE_BYTES;
constexpr int SB_Q = SB_V + TILE_BYTES;          // 2 stages
constexpr int SB_DO = SB_Q + 2 * TILE_BYTES;     // 2 stages
constexpr int SB_P = SB_DO + 2 * TILE_BYTES;     // 2 chunks
constexpr int SB_DS = SB_P + 2 * TILE_BYTES;     // 2 chunks
constexpr int SB_BAR = SB_DS + 2 * TILE_BYTES;
constexpr int BWD_SMEM = SB_BAR + 256 + 1024;
constexpr int SB_SEG_IDS = SB_BAR + 256;               // SEG: int [128] key ids of the CTA's kv block
constexpr int SB_SEG_LIST = SB_SEG_IDS + BKV * 4;      // SEG: int visited count, then the list of query blocks
constexpr int BWD_SEG_SMEM = SB_SEG_LIST + 16 + SEG_MAX_BLOCKS * 4 + 1024;

struct AttnBwdParams {
  const float* lse;    // [B,H,S]
  const float* delta;  // [B,H,S]
  float* dq_acc;       // fp32 [B,S,H,D] (zero-initialised)
  void* dk;            // bf16, strided [B,S,H,D] view
  void* dv;
  long long dstride_b, dstride_s, dstride_h;
  int B, H, S, causal;
  float scale_log2, scale;
};

template <int POLY, int SEG>
__global__ void __launch_bounds__(BWD_THREADS, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_do,
                const AttnBwdParams p, const AttnSeg sg) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SB_BAR);
  uint64_t* kv_full = bars + 0;
  uint64_t* q_full = bars + 1;     // [2]
  uint64_t* q_empty = bars + 3;    // [2]
  uint64_t* s_full = bars + 5;
  uint64_t* s_empty = bars + 6;
  uint64_t* pds_full = bars + 7;
  uint64_t* mma2_done = bars + 8;
  uint64_t* dq_empty = bars + 9;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nq = p.S / BQ;
  const int BH = p.B * p.H;
  const int j = (int)(blockIdx.x / BH);  // kv block; small j = most work, scheduled first
  const int bh = blockIdx.x % BH;
  const int b = bh / p.H, h = bh % p.H;
  const int i0 = p.causal ? j : 0;
  int n_it = nq - i0;
  int* seg_ids = reinterpret_cast<int*>(smem + SB_SEG_IDS);
  int* seg_list = reinterpret_cast<int*>(smem + SB_SEG_LIST) + 4;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
    tma_prefetch_desc(&tmap_do);
    mbar_init(kv_full, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
    mbar_init(s_full, 1);
    mbar_init(s_empty, 8);
    mbar_init(pds_full, 8);
    mbar_init(mma2_done, 1);
    mbar_init(dq_empty, 8);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_trigger();
  if (SEG) {         // every role walks the same list of query blocks whose id interval meets this key block's
    if (warp == 2) {
      const int nv = seg_visit_list(sg.rng_q + (size_t)b * nq, i0, nq, sg.rng_k[(size_t)b * nq + j], seg_list, lane);
      if (lane == 0) seg_list[-1] = nv;
    }
    __syncthreads();
    n_it = seg_list[-1];
  }
  const uint32_t TM_S = tmem_base, TM_DP = tmem_base + 128, TM_DV = tmem_base + 256, TM_DK = tmem_base + 320,
                 TM_DQ = tmem_base + 384;

  if (warp == 0) {
    if (elect_one()) {
      if (!SEG || n_it > 0) {
        mbar_expect_tx(kv_full, 2 * TILE_BYTES + (SEG ? BKV * 4 : 0));
        tma_load_4d(smem + SB_K, &tmap_k, kv_full, 0, j * BKV, h, b);
        tma_load_4d(smem + SB_V, &tmap_v, kv_full, 0, j * BKV, h, b);
        if (SEG) bulk_load(seg_ids, sg.seg_k + b * sg.stride + j * BKV, BKV * 4, kv_full);
      }
      for (int it = 0; it < n_it; ++it) {
        const int st = it & 1;
        const int i = SEG ? seg_list[it] : i0 + it;
        mbar_wait(&q_empty[st], ((it >> 1) & 1) ^ 1);
        mbar_expect_tx(&q_full[st], 2 * TILE_BYTES);
        tma_load_4d(smem + SB_Q + st * TILE_BYTES, &tmap_q, &q_full[st], 0, i * BQ, h, b);
        tma_load_4d(smem + SB_DO + st * TILE_BYTES, &tmap_do, &q_full[st], 0, i * BQ, h, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc(UMMA_BF16, UMMA_BF16, 128, 128, 0, 0);
      constexpr uint32_t idesc_t = make_idesc(UMMA_BF16, UMMA_BF16, 128, 64, 1, 1);   // dV, dK
      constexpr uint32_t idesc_dq = make_idesc(UMMA_BF16, UMMA_BF16, 128, 64, 0, 1);  // dQ
      const uint32_t sk = smem_u32(smem + SB_K), sv = smem_u32(smem + SB_V);
      const uint32_t sp = smem_u32(smem + SB_P), sds = smem_u32(smem + SB_DS);
      auto issue_sdp = [&](int it) {
        const int st = it & 1;
        mbar_wait(&q_full[st], (it >> 1) & 1);
        if (it > 0) mbar_wait(s_empty, (it - 1) & 1);
        tc_fence_after();
        const uint32_t sq = smem_u32(smem + SB_Q + st * TILE_BYTES);
        const uint32_t sdo = smem_u32(smem + SB_DO + st * TILE_BYTES);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
          umma_f16_ss(TM_S, make_smem_desc_sw128(sq + k * 32, 0, 1024), make_smem_desc_sw128(sk + k * 32, 0, 1024),
                      idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
          umma_f16_ss(TM_DP, make_smem_desc_sw128(sdo + k * 32, 0, 1024), make_smem_desc_sw128(sv + k * 32, 0, 1024),
                      idesc_s, k > 0 ? 1u : 0u);
        umma_commit(s_full);
      };
      if (!SEG || n_it > 0) {
        mbar_wait(kv_full, 0);
        issue_sdp(0);
      }
      for (int it = 0; it < n_it; ++it) {
        const int st = it & 1;
        mbar_wait(pds_full, it & 1);
        if (it > 0) mbar_wait(dq_empty, (it - 1) & 1);
        tc_fence_after();
        const uint32_t sq = smem_u32(smem + SB_Q + st * TILE_BYTES);
        const uint32_t sdo = smem_u32(smem + SB_DO + st * TILE_BYTES);
#pragma unroll
        for (int k = 0; k < BQ / 16; ++k)  // dV[kv, d] += sum_q P[q, kv] dO[q, d]
          umma_f16_ss(TM_DV, make_smem_desc_sw128(sp + k * 2048, TILE_BYTES, 1024),
                      make_smem_desc_sw128(sdo + k * 2048, TILE_BYTES, 1024), idesc_t, (it > 0 || k > 0) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < BQ / 16; ++k)  // dK[kv, d] += sum_q dS[q, kv] Q[q, d]
          umma_f16_ss(TM_DK, make_smem_desc_sw128(sds + k * 2048, TILE_BYTES, 1024),
                      make_smem_desc_sw128(sq + k * 2048, TILE_BYTES, 1024), idesc_t, (it > 0 || k > 0) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < BKV / 16; ++k)  // dQ[q, d] = sum_kv dS[q, kv] K[kv, d]
          umma_f16_ss(TM_DQ, make_smem_desc_sw128(sds + (k >> 2) * TILE_BYTES + (k & 3) * 32, 0, 1024),
                      make_smem_desc_sw128(sk + k * 2048, TILE_BYTES, 1024), idesc_dq, k > 0 ? 1u : 0u);
        umma_commit(mma2_done);
        umma_commit(&q_empty[st]);
        if (it + 1 < n_it) issue_sdp(it + 1);
      }
    }
  } else {
    const int sw = warp - 2;
    const int quarter = warp & 3;
    const int half = (sw >= 4) ? 1 : 0;
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = uint32_t(quarter * 32) << 16;
    const float LOG2E = 1.4426950408889634f;
    for (int it = 0; it < n_it; ++it) {
      const int i = SEG ? seg_list[it] : i0 + it;
      const int q_global = i * BQ + row;
      const size_t stat_idx = ((size_t)b * p.H + h) * p.S + q_global;
      const float lse2 = p.lse[stat_idx] * LOG2E;
      const float delta = p.delta[stat_idx];
      mbar_wait(s_full, it & 1);
      tc_fence_after();
      uint32_t rs0[32], rs1[32], rd0[32], rd1[32];
      tmem_ld_32x32(TM_S + lane_addr + half * 64, rs0);
      tmem_ld_32x32(TM_S + lane_addr + half * 64 + 32, rs1);
      tmem_ld_32x32(TM_DP + lane_addr + half * 64, rd0);
      tmem_ld_32x32(TM_DP + lane_addr + half * 64 + 32, rd1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_empty);

      uint8_t* prow = smem + SB_P + half * TILE_BYTES + row * 128;
      uint8_t* dsrow = smem + SB_DS + half * TILE_BYTES + row * 128;
      const bool diag = p.causal && (i == j);
      const int kv0 = j * BKV + half * 64;
      uint32_t vis[2] = {~0u, ~0u};      // SEG: bit e of vis[c] = key kv0 + 32 c + e belongs to this row's document
      if (SEG) {
        const int my_seg = sg.seg_q[b * sg.stride + q_global];
        const int2 kr = sg.rng_k[(size_t)b * nq + j];
        if (!(kr.x == my_seg && kr.y == my_seg)) {
          mbar_wait(kv_full, 0);           // (complete already: S was computed from this stage)
          const int4* ids = reinterpret_cast<const int4*>(seg_ids + half * 64);
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            vis[c] = 0u;
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              const int4 id = ids[c * 8 + g];
              vis[c] |= (uint32_t)((id.x == my_seg) | ((id.y == my_seg) << 1) | ((id.z == my_seg) << 2) | ((id.w == my_seg) << 3)) << (4 * g);
            }
          }
        }
      }
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t pk[16], dk_[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          float pv[2], dsv[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int idx = 2 * e + u;
            const float sv_ = __uint_as_float(c == 0 ? rs0[idx] : rs1[idx]);
            const float dpv = __uint_as_float(c == 0 ? rd0[idx] : rd1[idx]);
            const float xe = fmaf(sv_, p.scale_log2, -lse2);
            float pe = (POLY && u == 1) ? exp2_poly(xe) : exp2f(xe);
            if (diag && (kv0 + c * 32 + idx > q_global)) pe = 0.f;
            if (SEG && !((vis[c] >> idx) & 1u)) pe = 0.f;
            pv[u] = pe;
            dsv[u] = pe * (dpv - delta);
          }
          pk[e] = pack_bf16x2(pv[0], pv[1]);
          dk_[e] = pack_bf16x2(dsv[0], dsv[1]);
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int gran = c * 4 + g;
          const int off = (gran ^ (row & 7)) << 4;
          *reinterpret_cast<uint4*>(prow + off) = make_uint4(pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
          *reinterpret_cast<uint4*>(dsrow + off) = make_uint4(dk_[4 * g], dk_[4 * g + 1], dk_[4 * g + 2], dk_[4 * g + 3]);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(pds_full);

      // dQ tile for this (i, j) pair
      mbar_wait(mma2_done, it & 1);
      tc_fence_after();
      uint32_t rq[32];
      tmem_ld_32x32(TM_DQ + lane_addr + half * 32, rq);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(dq_empty);
      float* dqp = p.dq_acc + (((size_t)b * p.S + q_global) * p.H + h) * HD + half * 32;
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dqp + 4 * g),
                     "f"(__uint_as_float(rq[4 * g]) * p.scale), "f"(__uint_as_float(rq[4 * g + 1]) * p.scale),
                     "f"(__uint_as_float(rq[4 * g + 2]) * p.scale), "f"(__uint_as_float(rq[4 * g + 3]) * p.scale)
                     : "memory");
      }
    }
    // dV, dK for this kv block (complete after the last mma2_done, already waited)
    tc_fence_after();
    {
      uint32_t rv[32], rk[32];
      if (!SEG || n_it > 0) {
        tmem_ld_32x32(TM_DV + lane_addr + half * 32, rv);
        tmem_ld_32x32(TM_DK + lane_addr + half * 32, rk);
        tmem_ld_wait();
      } else {         // no query sees this key block: dK = dV = 0
#pragma unroll
        for (int i = 0; i < 32; ++i) rv[i] = rk[i] = 0u;
      }
      const size_t off = (size_t)b * p.dstride_b + (size_t)(j * BKV + row) * p.dstride_s + (size_t)h * p.dstride_h + half * 32;
      uint4* dvp = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.dv) + off);
      uint4* dkp = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.dk) + off);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 u, w;
        u.x = pack_bf16x2(__uint_as_float(rv[8 * g + 0]), __uint_as_float(rv[8 * g + 1]));
        u.y = pack_bf16x2(__uint_as_float(rv[8 * g + 2]), __uint_as_float(rv[8 * g + 3]));
        u.z = pack_bf16x2(__uint_as_float(rv[8 * g + 4]), __uint_as_float(rv[8 * g + 5]));
        u.w = pack_bf16x2(__uint_as_float(rv[8 * g + 6]), __uint_as_float(rv[8 * g + 7]));
        w.x = pack_bf16x2(__uint_as_float(rk[8 * g + 0]) * p.scale, __uint_as_float(rk[8 * g + 1]) * p.scale);
        w.y = pack_bf16x2(__uint_as_float(rk[8 * g + 2]) * p.scale, __uint_as_float(rk[8 * g + 3]) * p.scale);
        w.z = pack_bf16x2(__uint_as_float(rk[8 * g + 4]) * p.scale, __uint_as_float(rk[8 * g + 5]) * p.scale);
        w.w = pack_bf16x2(__uint_as_float(rk[8 * g + 6]) * p.scale, __uint_as_float(rk[8 * g + 7]) * p.scale);
        dvp[g] = u;
        dkp[g] = w;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// delta[b,h,s] = sum_d dO * O ; 8 lanes per (b, s, h) row of 64 elements (one 16-byte load per lane and tensor).
__global__ void attn_delta_kernel(const __nv_bfloat16* __restrict__ dO, const __nv_bfloat16* __restrict__ O,
                                  float* __restrict__ delta, int B, int S, int H) {
  const long long gid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long row = gid >> 3;
  const int sub = (int)(gid & 7);
  pdl_wait();
  if (row >= (long long)B * S * H) return;
  const int hh = row % H, s = (row / H) % S, bb = row / ((long long)H * S);
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(dO + row * HD) + sub);
  const uint4 c = __ldg(reinterpret_cast<const uint4*>(O + row * HD) + sub);
  const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&a);
  const __nv_bfloat162* hc = reinterpret_cast<const __nv_bfloat162*>(&c);
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 fa = __bfloat1622float2(ha[i]), fc = __bfloat1622float2(hc[i]);
    v += fa.x * fc.x + fa.y * fc.y;
  }
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  if (sub == 0) delta[((size_t)bb * H + hh) * S + s] = v;
}

// dq (bf16, strided) = dq_acc (fp32 contiguous [B,S,H,D])
// (the accumulator is zeroed again on the way out, so the persistent workspace never needs a separate memset)
__global__ void attn_dq_cast_kernel(float* __restrict__ acc, __nv_bfloat16* __restrict__ dq, int B, int S, int H,
                                    long long sb, long long ss, long long sh) {
  const size_t n8 = (size_t)B * S * H * (HD / 8);
  pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const int v = i % (HD / 8);
    size_t r = i / (HD / 8);
    const int hh = r % H; r /= H;
    const int s = r % S;
    const int bb = r / S;
    const float4 x = reinterpret_cast<const float4*>(acc)[i * 2], y = reinterpret_cast<const float4*>(acc)[i * 2 + 1];
    uint4 u;
    u.x = pack_bf16x2(x.x, x.y); u.y = pack_bf16x2(x.z, x.w); u.z = pack_bf16x2(y.x, y.y); u.w = pack_bf16x2(y.z, y.w);
    *reinterpret_cast<uint4*>(dq + (size_t)bb * sb + (size_t)s * ss + (size_t)hh * sh + v * 8) = u;
    reinterpret_cast<float4*>(acc)[i * 2] = make_float4(0.f, 0.f, 0.f, 0.f);
    reinterpret_cast<float4*>(acc)[i * 2 + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// Builds the AttnSeg of a masked call: checks the id layout and runs the [min, max] pre-pass into a persistent workspace.
// Returns 0, or an error code.
int seg_prepare(AttnSeg* sg, const void* seg_q, const void* seg_k, long long stride, int B, int S, cudaStream_t st) {
  const int nblk = S / 128;
  if (nblk > SEG_MAX_BLOCKS || stride < S || stride % 4 || ((uintptr_t)seg_q | (uintptr_t)seg_k) % 16) return -3;
  static int2* ws = nullptr;
  static size_t cap = 0;
  const size_t need = (size_t)2 * B * nblk;
  if (need > cap) {
    if (ws) cudaFree(ws);
    if (cudaMalloc(&ws, need * sizeof(int2)) != cudaSuccess) return -7;
    cap = need;
  }
  sg->seg_q = (const int*)seg_q; sg->seg_k = (const int*)seg_k; sg->stride = stride;
  sg->rng_q = ws; sg->rng_k = ws + (size_t)B * nblk;
  const int warps = B * nblk;
  return (int)tepd::launch(attn_seg_range_kernel, dim3((warps + 7) / 8, 2), dim3(256), 0, st, *sg, ws, ws + (size_t)B * nblk, B, nblk);
}

}  // namespace

// 4-D map over a [B, S, H, D]-addressable bf16 tensor given element strides; box = {64, box_rows, 1, 1}.
extern "C" int tepd_make_tmap_bshd(CUtensorMap* out, const void* ptr, int B, int S, int H, int D, long long stride_b,
                                   long long stride_s, long long stride_h, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return -1;
  cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)S, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)stride_s * 2, (cuuint64_t)stride_h * 2, (cuuint64_t)stride_b * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}

// q, k, v: bf16 pointers addressed as [B, S, H, D] with the given element strides (shared by q/k/v).
// seg_q / seg_k: int32 document ids (row b at seg + b * seg_stride, 16-byte aligned), or null for the plain causal / full mask.
extern "C" int tepd_attn_fwd(const void* q, const void* k, const void* v, void* o, void* lse, int B, int H, int S, int D,
                             float scale, int causal, long long stride_b, long long stride_s, long long stride_h,
                             const void* seg_q, const void* seg_k, long long seg_stride, void* stream) {
  if (D != HD || S % 128 != 0) return -2;
  CUtensorMap tq, tk, tv;
  int rc = tepd_make_tmap_bshd(&tq, q, B, S, H, D, stride_b, stride_s, stride_h, BQ);
  if (rc) return 100 + rc;
  rc = tepd_make_tmap_bshd(&tk, k, B, S, H, D, stride_b, stride_s, stride_h, BKV);
  if (rc) return 200 + rc;
  rc = tepd_make_tmap_bshd(&tv, v, B, S, H, D, stride_b, stride_s, stride_h, BKV);
  if (rc) return 300 + rc;
  static bool cfg = false;
  if (!cfg) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_fwd_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_fwd_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SEG_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_fwd_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SEG_SMEM);
    if (e != cudaSuccess) return (int)e;
    cfg = true;
  }
  AttnFwdParams p;
  p.O = o; p.lse = (float*)lse; p.B = B; p.H = H; p.S = S; p.causal = causal;
  p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
  cudaStream_t cs = reinterpret_cast<cudaStream_t>(stream);
  const int grid = (S / BQ) * B * H;
  AttnSeg sg = {};
  if (seg_q != nullptr || seg_k != nullptr) {   // document mask: always the default kernel (the two-tile variant has no mask)
    if (seg_q == nullptr || seg_k == nullptr) return -3;
    rc = seg_prepare(&sg, seg_q, seg_k, seg_stride, B, S, cs);
    if (rc) return rc;
    if (exp_poly_enabled())
      return (int)tepd::launch(attn_fwd_kernel<1, 1>, dim3(grid), dim3(FWD_THREADS), FWD_SEG_SMEM, cs, tq, tk, tv, p, sg);
    return (int)tepd::launch(attn_fwd_kernel<0, 1>, dim3(grid), dim3(FWD_THREADS), FWD_SEG_SMEM, cs, tq, tk, tv, p, sg);
  }
  if (fwd2_enabled() && S % 256 == 0) {   // experimental two-tile kernel
    static bool cfg2 = false;
    if (!cfg2) {
      cudaError_t e = cudaFuncSetAttribute(attn_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, F2_SMEM);
      if (e != cudaSuccess) return (int)e;
      cfg2 = true;
    }
    return (int)tepd::launch(attn_fwd2_kernel, dim3((S / 256) * B * H), dim3(F2_THREADS), F2_SMEM, reinterpret_cast<cudaStream_t>(stream),
                             tq, tk, tv, p);
  }
  if (exp_poly_enabled())
    return (int)tepd::launch(attn_fwd_kernel<1, 0>, dim3(grid), dim3(FWD_THREADS), FWD_SMEM, cs, tq, tk, tv, p, sg);
  return (int)tepd::launch(attn_fwd_kernel<0, 0>, dim3(grid), dim3(FWD_THREADS), FWD_SMEM, cs, tq, tk, tv, p, sg);
}

// (host) TEPDIST_ATTN_EXP_POLY=1 selects the POLY = 1 instantiations
// do, o: contiguous [B,S,H,D]; q/k/v strided views; dq/dk/dv strided views (shared strides).
extern "C" int tepd_attn_bwd(const void* dO, const void* q, const void* k, const void* v, const void* o, const void* lse,
                             void* dq_acc, void* dq, void* dk, void* dv, int B, int H, int S, int D, float scale,
                             int causal, long long stride_b, long long stride_s, long long stride_h, long long dstride_b,
                             long long dstride_s, long long dstride_h, const void* seg_q, const void* seg_k,
                             long long seg_stride, void* stream) {
  if (D != HD || S % 128 != 0) return -2;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUtensorMap tq, tk, tv, tdo;
  int rc = tepd_make_tmap_bshd(&tq, q, B, S, H, D, stride_b, stride_s, stride_h, BQ);
  if (rc) return 100 + rc;
  rc = tepd_make_tmap_bshd(&tk, k, B, S, H, D, stride_b, stride_s, stride_h, BKV);
  if (rc) return 200 + rc;
  rc = tepd_make_tmap_bshd(&tv, v, B, S, H, D, stride_b, stride_s, stride_h, BKV);
  if (rc) return 300 + rc;
  rc = tepd_make_tmap_bshd(&tdo, dO, B, S, H, D, (long long)S * H * D, (long long)H * D, D, BQ);
  if (rc) return 400 + rc;
  static float* delta_buf = nullptr;
  static size_t delta_cap = 0;
  const size_t need = (size_t)B * H * S;
  if (need > delta_cap) {
    if (delta_buf) cudaFree(delta_buf);
    if (cudaMalloc(&delta_buf, need * sizeof(float)) != cudaSuccess) return -5;
    delta_cap = need;
  }
  {
    const long long rows = (long long)B * S * H;
    cudaError_t le = tepd::launch(attn_delta_kernel, dim3((unsigned)((rows * 8 + 255) / 256)), dim3(256), 0, st,
                                  (const __nv_bfloat16*)dO, (const __nv_bfloat16*)o, delta_buf, B, S, H);
    if (le != cudaSuccess) return (int)le;
  }
  // persistent, self-clearing fp32 dQ accumulator (used when the caller passes no buffer)
  static float* dq_ws = nullptr;
  static size_t dq_cap = 0;
  if (dq_acc == nullptr) {
    const size_t needq = (size_t)B * S * H * HD;
    if (needq > dq_cap) {
      if (dq_ws) cudaFree(dq_ws);
      if (cudaMalloc(&dq_ws, needq * sizeof(float)) != cudaSuccess) return -6;
      cudaMemsetAsync(dq_ws, 0, needq * sizeof(float), st);
      dq_cap = needq;
    }
    dq_acc = dq_ws;
  }
  static bool cfg = false;
  if (!cfg) {
    cudaError_t e = cudaFuncSetAttribute(attn_bwd_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_bwd_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_bwd_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SEG_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attn_bwd_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SEG_SMEM);
    if (e != cudaSuccess) return (int)e;
    cfg = true;
  }
  AttnBwdParams p;
  p.lse = (const float*)lse; p.delta = delta_buf; p.dq_acc = (float*)dq_acc; p.dk = dk; p.dv = dv;
  p.dstride_b = dstride_b; p.dstride_s = dstride_s; p.dstride_h = dstride_h;
  p.B = B; p.H = H; p.S = S; p.causal = causal; p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
  const dim3 grid((S / BKV) * B * H);
  AttnSeg sg = {};
  cudaError_t le;
  if (seg_q != nullptr || seg_k != nullptr) {
    if (seg_q == nullptr || seg_k == nullptr) return -3;
    rc = seg_prepare(&sg, seg_q, seg_k, seg_stride, B, S, st);
    if (rc) return rc;
    le = exp_poly_enabled() ? tepd::launch(attn_bwd_kernel<1, 1>, grid, dim3(BWD_THREADS), BWD_SEG_SMEM, st, tq, tk, tv, tdo, p, sg)
                            : tepd::launch(attn_bwd_kernel<0, 1>, grid, dim3(BWD_THREADS), BWD_SEG_SMEM, st, tq, tk, tv, tdo, p, sg);
  } else {
    le = exp_poly_enabled() ? tepd::launch(attn_bwd_kernel<1, 0>, grid, dim3(BWD_THREADS), BWD_SMEM, st, tq, tk, tv, tdo, p, sg)
                            : tepd::launch(attn_bwd_kernel<0, 0>, grid, dim3(BWD_THREADS), BWD_SMEM, st, tq, tk, tv, tdo, p, sg);
  }
  if (le != cudaSuccess) return (int)le;
  return (int)tepd::launch(attn_dq_cast_kernel, dim3(148 * 4), dim3(256), 0, st, (float*)dq_acc, (__nv_bfloat16*)dq, B, S, H,
                           dstride_b, dstride_s, dstride_h);
}
