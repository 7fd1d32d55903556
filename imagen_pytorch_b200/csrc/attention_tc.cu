// tcgen05 flash attention for cosine-sim attention with a KNOWN logit bound (head dim 64).
//
// Cosine-sim attention makes the logits bounded: q and k are unit vectors times learned per-dim scales, so
// |s| <= 8 * max_d|q_scale_d * k_scale_d| (Cauchy-Schwarz).  With that bound C (in log2 units; Q arrives
// pre-multiplied by 8*log2e) the softmax needs NO running maximum and the output accumulator O in TMEM is never rescaled:
// a key tile costs exactly two MMAs + one exp2 per score.  The host only takes this path when C is small enough that the
// row sums stay inside fp32; otherwise the online-softmax kernel in attention.cu is used.
//
// Kernels in this file (history and measurements: DESIGN.md section 3, profiles/r0*_attention_*):
//   flash_attn_pp_kernel   ping-pong over two 128-row query tiles, P through shared memory (round-1 default, kept as variant 12)
//   flash_attn_pt_kernel   + P in tensor memory (tcgen05.st, TS-form MMA), scores preloaded so that S is released before the first
//                          exponential, three elect.sync issuer threads: the default for long key sequences (variant 118)
//   flash_attn_ptp_kernel  the same pipeline as persistent CTAs: the default for <= FA_PERSISTENT_MAX_TILES key tiles
//   cross_attn_tc_kernel   <= 64 keys (cross-attention over the text tokens), persistent, K/V of all heads resident
// Every kernel: warp 0 TMA producer (Q tiles, K/V ring, 128-byte swizzle), one MMA-issuer thread per query tile, softmax warps
// that own (query row, key slice) and read S / write P / read O with tcgen05.ld / tcgen05.st.
//
// Replaces the same reference arithmetic as attention.cu (Attention.forward / CrossAttention.forward einsum ->
// softmax -> einsum, imagen_pytorch.py:565-588, :818-833).
#include <cstdio>
#include "ptx.cuh"
#include <stdlib.h>

namespace {

constexpr int FA_BM = 128;
constexpr int FA_BN = 128;
constexpr int FA_D = 64;
constexpr int FA_PERSISTENT_MAX_TILES = 13;  // persistent kernel up to 1664 keys: 3.4 us + 1.20 us per key tile per item against 5.1 + 1.07 one-shot (profiles/r02_attention_elect_split_sweep.txt)
constexpr int FA_DEFAULT_WAIT_NS = 100;  // barrier waits park instead of spinning (1.58 -> 1.41 ms, profiles/r02_attention_wait_hint_sweep.txt)
constexpr int FA_Q_BYTES = FA_BM * FA_D * 2;        // 16 KB
constexpr int FA_K_BYTES = FA_BN * FA_D * 2;        // 16 KB
constexpr int FA_KV_BYTES = 2 * FA_K_BYTES;         // K + V per stage
constexpr int FA_TMEM_COLS = 512;                   // S0 [0,128) S1 [128,256) O [256,320)

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// exp2 on the FMA/ALU pipes (Cody-Waite split + cubic): the MUFU pipe delivers only 16 exp2/clk/SM, which is THE bound of
// head-dim-64 attention; moving a fraction of the exponentials here frees MUFU issue slots.  |rel err| < 7e-4 (P is bf16).
__device__ __forceinline__ float ex2_poly(float x) {
  x = fmaxf(x, -120.f);
  const float magic = 12582912.f;                 // 1.5 * 2^23: the add rounds x to the nearest integer in the low mantissa bits
  const float xm = x + magic;
  const float f = x - (xm - magic);               // fractional part in [-0.5, 0.5]
  float p = fmaf(f, 0.05550410866f, 0.2402265070f);
  p = fmaf(p, f, 0.6931471806f);
  p = fmaf(p, f, 1.0f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(xm) << 23));   // * 2^n through the exponent field
}

struct FaParams {
  __nv_bfloat16* o;
  long long q_bs, q_hs;
  int q_rs, rows, n_keys;
  int q_heads_first, kv_heads_first;   // coordinate order of the (rows, heads) dims in the tensor maps
  float max_logit;
  uint32_t wait_ns;                    // suspend-time hint of the barrier waits (0 = plain spin); B200_IMAGEN_FA_WAIT_NS
  long long* trace;                    // development only (MODE bit 9, B200_IMAGEN_FA_TRACE): clock64 stamps of one CTA, [warp][key tile][8]
  int trace_cta;
};

// ------------------------------------------------------------------------------------------------------------------
// Ping-pong variant: TWO 128-row query tiles (groups A and B) per CTA share one K/V stream.  Each group has its own
// MMA issuer thread, S accumulator, double-buffered P, O accumulator and four softmax warps, so the groups are fully
// decoupled: while one waits on its TMEM read / proxy fence / barrier round trip the other one exponentiates, and the S
// of the next key tile is issued as soon as a group has pulled its current scores into registers.
// (Measured on B200: in the round-1 one-tile kernel the softmax warps issue only ~27% of the time regardless of their
// number -- the per-tile dependency chain, not MUFU, was the limit; a first ping-pong with ONE issuer thread and a
// single P buffer per group still had the softmax warps waiting on p_empty / the in-order issuer: 1.91 ms.)
// TMEM: S_A [0,128) S_B [128,256) O_A [256,320) O_B [320,384).
// warps: 0 TMA, 1 issuer A (+TMEM alloc), 2 issuer B, 3 idle, 4-7 softmax A, 8-11 softmax B.
// ------------------------------------------------------------------------------------------------------------------
constexpr int PP_STAGES = 4;                       // deep K/V ring: the two groups may drift apart by more than a tile
constexpr int PP_PH_BYTES = FA_BM * 64 * 2;        // one 64-key half of a P tile (16 KB), its own full/empty barriers
constexpr int PP_SMEM = 2 * FA_Q_BYTES + PP_STAGES * FA_KV_BYTES + 4 * PP_PH_BYTES + 1024 + 256;   // 230656 B of the 232448 B limit

template <int POLY, int SUB>   // POLY: every POLY-th exponential goes to the FMA pipe (0 = all on MUFU); SUB: softmax warps per lane quarter per group
__global__ void __launch_bounds__(128 + 256 * SUB, 1)
flash_attn_pp_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                     const __grid_constant__ CUtensorMap mapV, const __grid_constant__ FaParams p) {
  pdl_trigger();
  extern __shared__ uint8_t fa_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(fa_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                                   // [2] query tiles
  uint8_t* sKV = sQ + 2 * FA_Q_BYTES;                   // [PP_STAGES] {K, V}
  uint8_t* sP = sKV + PP_STAGES * FA_KV_BYTES;          // [group][half] 64-key halves of the P tile
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 4 * PP_PH_BYTES);
  uint64_t* q_full = bars;                       // [1]
  uint64_t* kv_full = bars + 1;                  // [4]
  uint64_t* kv_empty = bars + 5;                 // [4]   (count 2: both groups' P V MMAs)
  uint64_t* s_full = bars + 9;                   // [group]
  uint64_t* s_empty = bars + 11;                 // [group]
  uint64_t* p_full = bars + 13;                  // [group][half]
  uint64_t* p_empty = bars + 17;                 // [group][half]
  uint64_t* o_full = bars + 21;                  // [group]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 23);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * (2 * FA_BM);
  const int h = blockIdx.y, b = blockIdx.z;
  const int ntiles = (p.n_keys + FA_BN - 1) / FA_BN;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapQ);
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
    mbar_init(q_full, 1);
    for (int s = 0; s < PP_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 2); }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&s_full[g], 1);
      mbar_init(&s_empty[g], 128 * SUB);
      mbar_init(&o_full[g], 1);
      for (int i = 0; i < 2; ++i) { mbar_init(&p_full[2 * g + i], 128); mbar_init(&p_empty[2 * g + i], 1); }   // per 64-key half (its 128 writer threads)
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, FA_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // provably warp-uniform (see elect_one in ptx.cuh)
  pdl_wait();

  if (warp == 0) {
    if (elect_one()) {
      // ---------------- TMA producer: both query tiles, then the K/V ring
      mbar_expect_tx(q_full, 2 * FA_Q_BYTES);
      for (int g = 0; g < 2; ++g) {
        if (p.q_heads_first) tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, h, row0 + g * FA_BM, b);
        else tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, row0 + g * FA_BM, h, b);
      }
      for (int j = 0; j < ntiles; ++j) {
        const int st = j % PP_STAGES;
        const uint32_t n = (uint32_t)(j / PP_STAGES);
        mbar_wait(&kv_empty[st], (n & 1u) ^ 1u);
        mbar_expect_tx(&kv_full[st], FA_KV_BYTES);
        uint8_t* dst = sKV + st * FA_KV_BYTES;
        if (p.kv_heads_first) {
          tma_load_4d(dst, &mapK, &kv_full[st], 0, h, j * FA_BN, b);
          tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, h, j * FA_BN, b);
        } else {
          tma_load_4d(dst, &mapK, &kv_full[st], 0, j * FA_BN, h, b);
          tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, j * FA_BN, h, b);
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    if (elect_one()) {
      // ---------------- MMA issuer of group g
      const int g = warp - 1;
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FA_BN >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint32_t idesc_pv = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(FA_D >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint64_t qdesc = make_sw128_kmajor_desc(smem_u32(sQ + g * FA_Q_BYTES));
      auto issue_s = [&](int j) {               // S_g(j) = Q_g K_j^T once group g has pulled S_g(j-1) into registers
        const int st = j % PP_STAGES;
        mbar_wait(&kv_full[st], (uint32_t)((j / PP_STAGES) & 1));
        mbar_wait(&s_empty[g], (uint32_t)((j & 1) ^ 1));
        tc_fence_after();
        const uint64_t bdesc = make_sw128_kmajor_desc(smem_u32(sKV + st * FA_KV_BYTES));
#pragma unroll
        for (int k = 0; k < FA_D / 16; ++k)
          umma_bf16(tmem_base + (uint32_t)(g * FA_BN), qdesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_s, k != 0 ? 1u : 0u);
        umma_commit(&s_full[g]);
      };
      mbar_wait(q_full, 0);
      issue_s(0);
      for (int j = 0; j < ntiles; ++j) {
        if (j + 1 < ntiles) issue_s(j + 1);
        const int st = j % PP_STAGES;
        const uint32_t v_addr = smem_u32(sKV + st * FA_KV_BYTES + FA_K_BYTES);
        for (int hf = 0; hf < 2; ++hf) {        // the first 64 keys are multiplied while the second 64 are exponentiated
          const int pb = 2 * g + hf;
          mbar_wait(&p_full[pb], (uint32_t)(j & 1));
          tc_fence_after();
          const uint32_t p_addr = smem_u32(sP + pb * PP_PH_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t adesc = make_sw128_kmajor_desc(p_addr + (uint32_t)(k * 32));
            const uint64_t bdesc = make_sw128_mnmajor_desc(v_addr + (uint32_t)((hf * 4 + k) * 16 * 128), 1024, 1024);
            umma_bf16(tmem_base + (uint32_t)(256 + g * FA_D), adesc, bdesc, idesc_pv, (j | hf | k) != 0 ? 1u : 0u);
          }
          umma_commit(&p_empty[pb]);
        }
        umma_commit(&kv_empty[st]);             // one of the two arrivals that free K_j / V_j
      }
      umma_commit(&o_full[g]);
    }
  } else if (warp >= 4) {
    // ---------------- softmax / epilogue: group g, thread = (query row of that group, column half if SUB == 2).
    // With SUB == 2 each scheduler sub-partition holds four softmax warps in four different phases (2 groups x 2 halves):
    // the MUFU pipe of a sub-partition idles whenever all of its warps are in a TMEM-read / store / fence / barrier phase,
    // which with only two warps per sub-partition happened ~45% of the time (XU pipe 55-59% in ncu).
    const int idx = warp - 4;
    const int g = idx / (4 * SUB);
    const int sub = (idx >> 2) % SUB;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    float l = 0.f;
    const float C = p.max_logit;
    for (int j = 0; j < ntiles; ++j) {
      mbar_wait(&s_full[g], (uint32_t)(j & 1));
      tc_fence_after();
      const int key0 = j * FA_BN;
      const bool ragged = key0 + FA_BN > p.n_keys;
      // 64-key halves of the tile; a thread owns both (SUB == 1) or only half `sub` (SUB == 2).  Scores are pulled from TMEM
      // in chunks of CH columns, load -> wait -> exponentiate (several tcgen05.ld in flight per warp are SLOWER:
      // profiles/r01_tmem_ld_microbench.txt).
      constexpr int CH = SUB == 2 ? 32 : 64;
#pragma unroll 1
      for (int hh = 0; hh < 2 / SUB; ++hh) {
        const int hf = SUB == 2 ? sub : hh;
        const int pb = 2 * g + hf;
        uint8_t* prow = sP + pb * PP_PH_BYTES + r * 128;
#pragma unroll 1
        for (int c0 = 0; c0 < 64; c0 += CH) {
          uint32_t sr[CH];
#pragma unroll
          for (int c = 0; c < CH; c += 32) tmem_ld32_nowait(tmem_base + lane_off + (uint32_t)(g * FA_BN + hf * 64 + c0 + c), sr + c);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < CH; ++i) asm volatile("" : "+r"(sr[i]));   // pin the destination registers behind the wait
          if (c0 + CH == 64 && (SUB == 2 || hh == 1)) {
            tc_fence_before();
            mbar_arrive(&s_empty[g]);           // this thread's share of S_g is in registers
          }
          if (c0 == 0) mbar_wait(&p_empty[pb], (uint32_t)((j & 1) ^ 1));   // the P V MMAs of tile j-1 have finished reading this half
#pragma unroll
          for (int t = 0; t < CH / 8; ++t) {
            uint32_t pk[4];
#pragma unroll
            for (int i = 0; i < 8; i += 2) {
              float p0 = ex2_approx(__uint_as_float(sr[8 * t + i]) - C);
              float p1 = (POLY > 0 && ((8 * t + i + 1) % (POLY > 0 ? POLY : 1)) == POLY - 1) ? ex2_poly(__uint_as_float(sr[8 * t + i + 1]) - C)
                                                                           : ex2_approx(__uint_as_float(sr[8 * t + i + 1]) - C);
              if (ragged) {
                if (key0 + hf * 64 + c0 + 8 * t + i >= p.n_keys) p0 = 0.f;
                if (key0 + hf * 64 + c0 + 8 * t + i + 1 >= p.n_keys) p1 = 0.f;
              }
              l += p0 + p1;
              pk[i >> 1] = pack_bf16x2(p0, p1);
            }
            *reinterpret_cast<uint4*>(prow + (((c0 / 8 + t) ^ (r & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
        }
        fence_proxy_async_smem();
        mbar_arrive(&p_full[pb]);
      }
    }
    // ---- O / l -> global (with SUB == 2 the two column-half threads of a row add their sums and each stores 32 channels)
    mbar_wait(&o_full[g], 0);                // every MMA of group g has completed: its P buffers are free
    tc_fence_after();
    if (SUB == 2) {
      float* sL = reinterpret_cast<float*>(sP + 2 * g * PP_PH_BYTES);   // [sub][128] partial row sums, in the group's own P buffer
      sL[sub * FA_BM + r] = l;
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");         // the 8 softmax warps of this group
      l = sL[r] + sL[FA_BM + r];
    }
    const float inv = 1.f / l;
    const int row = row0 + g * FA_BM + r;
    constexpr int OC = FA_D / SUB;
    __nv_bfloat16* orow = p.o + (long long)b * p.q_bs + (long long)h * p.q_hs + (long long)row * p.q_rs + sub * OC;
    uint32_t orr[OC];
#pragma unroll
    for (int c = 0; c < OC; c += 32) tmem_ld32_nowait(tmem_base + lane_off + (uint32_t)(256 + g * FA_D + sub * OC + c), orr + c);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < OC; ++i) asm volatile("" : "+r"(orr[i]));
    if (row < p.rows) {
#pragma unroll
      for (int t = 0; t < OC / 8; ++t) {
        uint4 u;
        u.x = pack_bf16x2(__uint_as_float(orr[8 * t + 0]) * inv, __uint_as_float(orr[8 * t + 1]) * inv);
        u.y = pack_bf16x2(__uint_as_float(orr[8 * t + 2]) * inv, __uint_as_float(orr[8 * t + 3]) * inv);
        u.z = pack_bf16x2(__uint_as_float(orr[8 * t + 4]) * inv, __uint_as_float(orr[8 * t + 5]) * inv);
        u.w = pack_bf16x2(__uint_as_float(orr[8 * t + 6]) * inv, __uint_as_float(orr[8 * t + 7]) * inv);
        *reinterpret_cast<uint4*>(orow + 8 * t) = u;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, FA_TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// "P in tensor memory" variant of the ping-pong kernel.  The softmax warps write the bf16 probabilities back to TMEM with
// tcgen05.st (two keys per 32-bit column, row = lane) and the O += P V MMA takes its A operand from TMEM (tcgen05.mma with
// [a_tmem]): no shared-memory P tile, no generic->async proxy fence per chunk, no bank conflicts, and the P V MMAs read
// only V (2 KB per K=16 step) from shared memory.  The 64 KB of shared memory the P tiles used become a deeper K/V ring.
// The last key tile's second half is skipped when it holds no valid key (4135 keys = 32 tiles + 39 keys).
// TMEM: S_A [0,128) S_B [128,256) O_A [256,320) O_B [320,384) P_A [384,448) P_B [448,512)  (P: 64 keys per 32 columns).
// ------------------------------------------------------------------------------------------------------------------
constexpr int PT_STAGES = 5;
constexpr int PT_SMEM = 2 * FA_Q_BYTES + PT_STAGES * FA_KV_BYTES + 1024 + 512 + 2048;   // + barriers + row-sum exchange

// 32 scores -> 16 packed bf16x2 probabilities + row-sum contribution.  MODE bit 0: no "- C" (P = exp2(S) directly: the bound only
// has to keep 2^C * n_keys inside fp32, and O / l is invariant to the common factor 2^C -- one FADD less per score); bits 1-2 are
// bottleneck experiments of tools/sweep_attention.py (WRONG results): 2 = no MUFU (the score is copied), 4 = no TMEM read.
// RAGGED is a separate instantiation: the key-bound compare + select per score (ISETP + FSEL) used to run for EVERY tile.
template <int POLY, int MODE, bool RAGGED>
__device__ __forceinline__ void pt_chunk32(const uint32_t* sr, float C, int key_base, int n_keys, uint32_t* pk, float& l) {
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    float x0 = __uint_as_float(sr[i]), x1 = __uint_as_float(sr[i + 1]);
    if (!(MODE & 1)) { x0 -= C; x1 -= C; }
    float p0, p1;
    if (MODE & 2) { p0 = x0; p1 = x1; }
    else {
      p0 = (POLY > 0 && (i % (POLY > 0 ? POLY : 1)) == (POLY > 0 ? POLY : 1) - 1) ? ex2_poly(x0) : ex2_approx(x0);
      p1 = (POLY > 0 && ((i + 1) % (POLY > 0 ? POLY : 1)) == (POLY > 0 ? POLY : 1) - 1) ? ex2_poly(x1) : ex2_approx(x1);
    }
    if (RAGGED) {
      if (key_base + i >= n_keys) p0 = 0.f;
      if (key_base + i + 1 >= n_keys) p1 = 0.f;
    }
    l0 += p0; l1 += p1;
    pk[i >> 1] = pack_bf16x2(p0, p1);
  }
  l += l0 + l1;
}

template <int POLY>
__device__ __forceinline__ bool pt_use_poly(int idx) { return POLY > 0 && (idx % (POLY > 0 ? POLY : 1)) == (POLY > 0 ? POLY : 1) - 1; }

// ORDER: the two groups take turns on the MUFU pipe (token passed through order_bar).  Without it the two identical periodic
// softmax pipelines lock IN phase: both exponentiate at the same time at half speed each, then both wait for their next S tile with
// the MUFU pipe idle (measured: XU pipe 62% busy at 16/clk/SM peak).  With the token, group B's TMEM reads / barrier round trips /
// S MMA latency run under group A's exponentials and vice versa.
template <int POLY, int SUB, bool ORDER, int MODE>   // POLY: every POLY-th exponential on the FMA pipe (0 = all MUFU); SUB: softmax warps per lane quarter per group; MODE: pt_chunk32
__global__ void __launch_bounds__(128 + 256 * SUB, 1)
flash_attn_pt_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                     const __grid_constant__ CUtensorMap mapV, const __grid_constant__ FaParams p) {
  pdl_trigger();
  extern __shared__ uint8_t fa_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(fa_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                                   // [2] query tiles
  uint8_t* sKV = sQ + 2 * FA_Q_BYTES;                   // [PT_STAGES] {K, V}
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + PT_STAGES * FA_KV_BYTES);
  uint64_t* q_full = bars;                              // [1]
  uint64_t* kv_full = bars + 1;                         // [PT_STAGES]
  uint64_t* kv_empty = kv_full + PT_STAGES;             // [PT_STAGES] (count 2: both groups' P V MMAs)
  uint64_t* s_full = kv_empty + PT_STAGES;              // [group]
  uint64_t* s_empty = s_full + 2;                       // [group]
  uint64_t* p_full = s_empty + 2;                       // [group][half][32-key chunk]
  uint64_t* p_empty = p_full + 8;                       // [group][half][32-key chunk]
  uint64_t* o_full = p_empty + 8;                       // [group]
  uint64_t* order_bar = o_full + 2;                     // [group]: group g may start exponentiating its next tile
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(order_bar + 2);
  float* sL = reinterpret_cast<float*>(bars + 64);      // [group][sub][128] partial row sums
  static_assert(1 + 2 * PT_STAGES + 2 + 2 + 8 + 8 + 2 + 2 + 1 <= 64, "barrier block is 512 bytes");

  // MODE bit 3: one mbarrier arrival per softmax WARP (elected lane after __syncwarp) instead of one per thread: 128-256 arrivals
  // on one shared-memory word serialise in the barrier unit, and every one of them sits on the S -> P -> O dependency chain
  constexpr bool WARP_ARRIVE = (MODE & 8) != 0;
  // MODE bit 5: P handed to the MMA issuer in 32-key chunks (own full / empty barrier each) instead of 64-key halves: the chunk a warp
  // writes first was multiplied while it exponentiated its second chunk of the previous tile, so it never waits for the P V MMA
  constexpr bool PCH = (MODE & 32) != 0;
  constexpr bool LATE = (MODE & 64) != 0;
  constexpr bool TRACE = (MODE & 512) != 0;
  // MODE bit 10: the S = Q K^T MMAs of BOTH groups are issued by a third thread (warp 3).  One issuer thread per group was the
  // bottleneck of the kernel: ~20 dependent operations per key tile (4 barrier waits, 12 MMAs with their descriptors, 4 commits) at
  // ~100 cycles each = the 2100-2250 cycles per tile that remained with the exponentials removed.
  constexpr bool SPLIT = (MODE & 1024) != 0;
  const bool traced = TRACE && p.trace != nullptr && (int)(blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z)) == p.trace_cta && ((threadIdx.x >> 5) < 4 || (threadIdx.x & 31) == 0);
#define FA_TR(j_, slot_)                                                                                   \
  do {                                                                                                     \
    if (TRACE && traced && (j_) < 64) p.trace[(((threadIdx.x >> 5) * 64 + (j_)) << 3) + (slot_)] = clock64(); \
  } while (0)   // MODE bit 6: wait for the free P buffer only before the first tcgen05.st, not before the first exponential
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * (2 * FA_BM);
  const int h = blockIdx.y, b = blockIdx.z;
  const int ntiles = (p.n_keys + FA_BN - 1) / FA_BN;
  const bool dead1 = (ntiles - 1) * FA_BN + 64 >= p.n_keys;   // the last tile's second 64-key half holds no valid key
  constexpr uint32_t TM_O = 256, TM_P = 384;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapQ);
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
    mbar_init(q_full, 1);
    for (int s = 0; s < PT_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 2); }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&s_full[g], 1);
      mbar_init(&s_empty[g], WARP_ARRIVE ? 4 * SUB : 128 * SUB);
      mbar_init(&o_full[g], 1);
      mbar_init(&order_bar[g], 4 * SUB);                // one arrival per softmax warp of the OTHER group
      for (int i = 0; i < 4; ++i) { mbar_init(&p_full[4 * g + i], WARP_ARRIVE ? 4 : 128); mbar_init(&p_empty[4 * g + i], 1); }
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, FA_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // provably warp-uniform (see elect_one in ptx.cuh)
  pdl_wait();

  if (warp == 0) {
    if (elect_one()) {
      // ---------------- TMA producer: both query tiles, then the K/V ring
      mbar_expect_tx(q_full, 2 * FA_Q_BYTES);
      for (int g = 0; g < 2; ++g) {
        if (p.q_heads_first) tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, h, row0 + g * FA_BM, b);
        else tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, row0 + g * FA_BM, h, b);
      }
      for (int j = 0; j < ntiles; ++j) {
        const int st = j % PT_STAGES;
        const uint32_t n = (uint32_t)(j / PT_STAGES);
        FA_TR(j, 0);
        mbar_wait_sleep(&kv_empty[st], (n & 1u) ^ 1u, p.wait_ns);
        FA_TR(j, 1);
        mbar_expect_tx(&kv_full[st], FA_KV_BYTES);
        uint8_t* dst = sKV + st * FA_KV_BYTES;
        if (p.kv_heads_first) {
          tma_load_4d(dst, &mapK, &kv_full[st], 0, h, j * FA_BN, b);
          tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, h, j * FA_BN, b);
        } else {
          tma_load_4d(dst, &mapK, &kv_full[st], 0, j * FA_BN, h, b);
          tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, j * FA_BN, h, b);
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    if (elect_one()) {
      // ---------------- MMA issuer of group g
      const int g = warp - 1;
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FA_BN >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint32_t idesc_pv = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(FA_D >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint64_t qdesc = make_sw128_kmajor_desc(smem_u32(sQ + g * FA_Q_BYTES));
      const uint64_t kdesc0 = make_sw128_kmajor_desc(smem_u32(sKV));                           // + stage * (FA_KV_BYTES >> 4)
      const uint64_t vdesc0 = make_sw128_mnmajor_desc(smem_u32(sKV + FA_K_BYTES), 1024, 1024);
      auto issue_s = [&](int j) {               // S_g(j) = Q_g K_j^T once group g has pulled S_g(j-1) into registers
        const int st = j % PT_STAGES;
        FA_TR(j, 0);
        mbar_wait_sleep(&kv_full[st], (uint32_t)((j / PT_STAGES) & 1), p.wait_ns);
        FA_TR(j, 1);
        mbar_wait_sleep(&s_empty[g], (uint32_t)((j & 1) ^ 1), p.wait_ns);
        FA_TR(j, 2);
        tc_fence_after();
        const uint64_t bdesc = kdesc0 + (uint64_t)(st * (FA_KV_BYTES >> 4));
#pragma unroll
        for (int k = 0; k < FA_D / 16; ++k)
          umma_bf16(tmem_base + (uint32_t)(g * FA_BN), qdesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_s, k != 0 ? 1u : 0u);
        umma_commit(&s_full[g]);
      };
      if (!SPLIT) {
        mbar_wait_sleep(q_full, 0, p.wait_ns);
        issue_s(0);
      }
      for (int j = 0; j < ntiles; ++j) {
        if (!SPLIT && j + 1 < ntiles) issue_s(j + 1);
        const int st = j % PT_STAGES;
        if (SPLIT) mbar_wait_sleep(&kv_full[st], (uint32_t)((j / PT_STAGES) & 1), p.wait_ns);   // V_j has landed (this thread did not issue S_j)
        const uint64_t vdesc = vdesc0 + (uint64_t)(st * (FA_KV_BYTES >> 4));
        // the first keys are multiplied while the later ones are exponentiated: halves in order, or (PCH) chunk 0 of both halves first
        for (int u = 0; u < (PCH ? 4 : 2); ++u) {
          const int hf = !PCH ? u : (SUB == 2 ? (u & 1) : (u >> 1)), ci = !PCH ? 0 : (SUB == 2 ? (u >> 1) : (u & 1));   // production order
          if (hf == 1 && dead1 && j == ntiles - 1) continue;
          const int pb = 4 * g + 2 * hf + ci;
          mbar_wait_sleep(&p_full[pb], (uint32_t)(j & 1), p.wait_ns);
          FA_TR(j, 3 + u);
          tc_fence_after();
#pragma unroll
          for (int k = (PCH ? 2 * ci : 0); k < (PCH ? 2 * ci + 2 : 4); ++k) {
            // A: 16 keys = 8 packed columns of this half's P block; B: 16 key rows of V (MN-major, 2 KB)
            const uint32_t a_tmem = tmem_base + TM_P + (uint32_t)(g * 64 + hf * 32 + k * 8);
            const uint64_t bdesc = vdesc + (uint64_t)((hf * 4 + k) * (16 * 128 >> 4));
            umma_bf16_ts(tmem_base + TM_O + (uint32_t)(g * FA_D), a_tmem, bdesc, idesc_pv, (j | u | (k & 1) | (PCH ? 0 : k)) != 0 ? 1u : 0u);
          }
          umma_commit(&p_empty[pb]);
        }
        umma_commit(&kv_empty[st]);             // one of the two arrivals that free K_j / V_j
        FA_TR(j, 7);
      }
      umma_commit(&o_full[g]);
    }
  } else if (SPLIT && warp == 3) {
    if (elect_one()) {
      // ---------------- S issuer of both groups
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FA_BN >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint64_t qdesc0 = make_sw128_kmajor_desc(smem_u32(sQ));
      const uint64_t kdesc0 = make_sw128_kmajor_desc(smem_u32(sKV));
      mbar_wait_sleep(q_full, 0, p.wait_ns);
      for (int j = 0; j < ntiles; ++j) {
        const int st = j % PT_STAGES;
        FA_TR(j, 0);
        mbar_wait_sleep(&kv_full[st], (uint32_t)((j / PT_STAGES) & 1), p.wait_ns);
        const uint64_t bdesc = kdesc0 + (uint64_t)(st * (FA_KV_BYTES >> 4));
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          FA_TR(j, 1 + 3 * g);
          mbar_wait_sleep(&s_empty[g], (uint32_t)((j & 1) ^ 1), p.wait_ns);   // group g has pulled S_g(j-1) into registers
          FA_TR(j, 2 + 3 * g);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < FA_D / 16; ++k)
            umma_bf16(tmem_base + (uint32_t)(g * FA_BN), qdesc0 + (uint64_t)(g * (FA_Q_BYTES >> 4) + 2 * k), bdesc + (uint64_t)(2 * k), idesc_s, k != 0 ? 1u : 0u);
          umma_commit(&s_full[g]);
          FA_TR(j, 3 + 3 * g);
        }
      }
    }
  } else if (warp >= 4) {
    // ---------------- softmax / epilogue: group g, thread = (query row of that group, 64-key half if SUB == 2)
    const int idx = warp - 4;
    const int g = idx / (4 * SUB);
    const int sub = (idx >> 2) % SUB;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    float l = 0.f;
    const float C = p.max_logit;
    for (int j = 0; j < ntiles; ++j) {
      const int key0 = j * FA_BN;
      const bool ragged = key0 + FA_BN > p.n_keys;
      const bool last_dead = dead1 && j == ntiles - 1;
      // token: A(j) follows B(j-1), B(j) follows A(j); a fresh barrier passes A's first wait (parity trick of the empty barriers)
      const uint32_t tok_par = g == 0 ? (uint32_t)((j & 1) ^ 1) : (uint32_t)(j & 1);
      if (SUB == 2 && sub == 1 && last_dead) {          // nothing valid in this warp's half of the last tile: only pass the token on
        if (ORDER) {
          mbar_wait_sleep(&order_bar[g], tok_par, p.wait_ns);
          __syncwarp();
          if (lane == 0) mbar_arrive(&order_bar[g ^ 1]);
        }
        break;
      }
      FA_TR(j, 0);
      mbar_wait_sleep(&s_full[g], (uint32_t)(j & 1), p.wait_ns);
      FA_TR(j, 1);
      tc_fence_after();
      bool have_token = !ORDER;
      constexpr int CH = (SUB == 2 && !(MODE & 16)) ? 32 : 64;   // MODE bit 4: all 64 scores of the thread in registers before the first exponential (S freed earlier)
#pragma unroll 1
      for (int hh = 0; hh < 2 / SUB; ++hh) {
        const int hf = SUB == 2 ? sub : hh;
        if (hf == 1 && last_dead) break;
        const int pb = 4 * g + 2 * hf;
        const uint32_t p_col = tmem_base + lane_off + TM_P + (uint32_t)(g * 64 + hf * 32);
#pragma unroll 1
        for (int c0 = 0; c0 < 64; c0 += CH) {
          uint32_t sr[CH];
          if (MODE & 4) {
#pragma unroll
            for (int i = 0; i < CH; ++i) sr[i] = __float_as_uint(-1.f - (float)(lane + i));
          } else {
            // (one x64 load, or the two x32 loads one after the other, measured the same: profiles/r02_attention_preload_sweep.txt)
#pragma unroll
            for (int c = 0; c < CH; c += 32) tmem_ld32_nowait(tmem_base + lane_off + (uint32_t)(g * FA_BN + hf * 64 + c0 + c), sr + c);
            tmem_ld_wait();
          }
#pragma unroll
          for (int i = 0; i < CH; ++i) asm volatile("" : "+r"(sr[i]));   // pin the destination registers behind the wait
          FA_TR(j, 2);
          if (c0 + CH == 64 && (SUB == 2 || hh == 1 || last_dead)) {
            tc_fence_before();                  // this thread's share of S_g is in registers
            if (WARP_ARRIVE) { __syncwarp(); if (lane == 0) mbar_arrive(&s_empty[g]); }
            else mbar_arrive(&s_empty[g]);
          }
          if (!PCH && !LATE && c0 == 0) {
            FA_TR(j, 3);
            mbar_wait_sleep(&p_empty[pb], (uint32_t)((j & 1) ^ 1), p.wait_ns);   // the P V MMAs of tile j-1 have finished reading this half of P
            tc_fence_after();
            FA_TR(j, 4);
          }
          if (!have_token) {                    // scores are in registers: now wait for this group's turn on the MUFU pipe
            mbar_wait_sleep(&order_bar[g], tok_par, p.wait_ns);
            have_token = true;
          }
#pragma unroll
          for (int t = 0; t < CH / 32; ++t) {
            uint32_t pk[16];
            const int kb = key0 + hf * 64 + c0 + 32 * t;
            if (ragged) pt_chunk32<POLY, MODE, true>(sr + 32 * t, C, kb, p.n_keys, pk, l);
            else pt_chunk32<POLY, MODE, false>(sr + 32 * t, C, kb, p.n_keys, pk, l);
            if (PCH) {
              mbar_wait_sleep(&p_empty[pb + ((c0 + 32 * t) >> 5)], (uint32_t)((j & 1) ^ 1), p.wait_ns);
              tc_fence_after();
            } else if (LATE && c0 == 0 && t == 0) {   // the first 32 exponentials ran while the P V MMAs of tile j-1 were still reading P
              mbar_wait_sleep(&p_empty[pb], (uint32_t)((j & 1) ^ 1), p.wait_ns);
              tc_fence_after();
            }
            tmem_st16(p_col + (uint32_t)((c0 + 32 * t) >> 1), pk);
            if (PCH) {
              tmem_st_wait();
              tc_fence_before();
              if (WARP_ARRIVE) { __syncwarp(); if (lane == 0) mbar_arrive(&p_full[pb + ((c0 + 32 * t) >> 5)]); }
              else mbar_arrive(&p_full[pb + ((c0 + 32 * t) >> 5)]);
            }
          }
        }
        if (ORDER && (SUB == 2 || hh == 1 || last_dead)) {   // exponentials of this tile issued: the other group's turn
          __syncwarp();
          if (lane == 0) mbar_arrive(&order_bar[g ^ 1]);
        }
        FA_TR(j, 5);
        if (!PCH) {
          tmem_st_wait();                        // the stores have landed in tensor memory ...
          tc_fence_before();                     // ... and are ordered before the issuer's MMAs through the barrier
          if (WARP_ARRIVE) { __syncwarp(); if (lane == 0) mbar_arrive(&p_full[pb]); }
          else mbar_arrive(&p_full[pb]);
        }
        FA_TR(j, 6);
      }
    }
    // ---- O / l -> global (with SUB == 2 the two column-half threads of a row add their sums and each stores 32 channels)
    mbar_wait_sleep(&o_full[g], 0, p.wait_ns);
    tc_fence_after();
    if (SUB == 2) {
      float* sLg = sL + g * 2 * FA_BM;
      sLg[sub * FA_BM + r] = l;
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");         // the 8 softmax warps of this group
      l = sLg[r] + sLg[FA_BM + r];
    }
    const float inv = 1.f / l;
    const int row = row0 + g * FA_BM + r;
    constexpr int OC = FA_D / SUB;
    __nv_bfloat16* orow = p.o + (long long)b * p.q_bs + (long long)h * p.q_hs + (long long)row * p.q_rs + sub * OC;
    uint32_t orr[OC];
#pragma unroll
    for (int c = 0; c < OC; c += 32) tmem_ld32_nowait(tmem_base + lane_off + TM_O + (uint32_t)(g * FA_D + sub * OC + c), orr + c);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < OC; ++i) asm volatile("" : "+r"(orr[i]));
    if (row < p.rows) {
#pragma unroll
      for (int t = 0; t < OC / 8; ++t) {
        uint4 u;
        u.x = pack_bf16x2(__uint_as_float(orr[8 * t + 0]) * inv, __uint_as_float(orr[8 * t + 1]) * inv);
        u.y = pack_bf16x2(__uint_as_float(orr[8 * t + 2]) * inv, __uint_as_float(orr[8 * t + 3]) * inv);
        u.z = pack_bf16x2(__uint_as_float(orr[8 * t + 4]) * inv, __uint_as_float(orr[8 * t + 5]) * inv);
        u.w = pack_bf16x2(__uint_as_float(orr[8 * t + 6]) * inv, __uint_as_float(orr[8 * t + 7]) * inv);
        *reinterpret_cast<uint4*>(orow + 8 * t) = u;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, FA_TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// "Dual" softmax: every softmax thread serves BOTH query tiles.  The time line of the kernel above (tools/attn_trace.py) shows each
// softmax warp busy for ~1500 of the 2430 cycles of a key tile and waiting for the rest (S ready, TMEM load, the P V MMA of the
// previous tile freeing its P buffer) -- and the two query-tile groups wait at the same time, so the MUFU pipe idles then.  Here a
// thread owns (query row r, 32-key quarter c) of tile A AND of tile B: per key tile it pulls both 32-score slices into registers
// (releasing S_A and S_B), then exponentiates one tile's slice, hands that P quarter to the issuer, and does the other tile's slice.
// By the time it returns to a tile, that tile's next S has long been computed and its P quarter long been multiplied, so in steady
// state no barrier wait blocks; odd quarters start with tile B, even ones with tile A, so P quarters reach both issuers evenly.
// TMEM as above; P quarter c of group g = 16 columns at 384 + 64 g + 16 c.  The P V product runs per quarter (K = 32: two MMAs).
// ------------------------------------------------------------------------------------------------------------------
constexpr int PD_SMEM = 2 * FA_Q_BYTES + PT_STAGES * FA_KV_BYTES + 1024 + 512 + 4096;   // + barriers + [2][4][128] partial row sums

template <int POLY, int MODE>   // MODE: bit 1 = no MUFU (bottleneck experiment, wrong results)
__global__ void __launch_bounds__(640, 1)
flash_attn_pd_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                     const __grid_constant__ CUtensorMap mapV, const __grid_constant__ FaParams p) {
  pdl_trigger();
  extern __shared__ uint8_t fa_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(fa_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                                   // [2] query tiles
  uint8_t* sKV = sQ + 2 * FA_Q_BYTES;                   // [PT_STAGES] {K, V}
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + PT_STAGES * FA_KV_BYTES);
  uint64_t* q_full = bars;                              // [1]
  uint64_t* kv_full = bars + 1;                         // [PT_STAGES]
  uint64_t* kv_empty = kv_full + PT_STAGES;             // [PT_STAGES] (count 2: both groups' P V MMAs)
  uint64_t* s_full = kv_empty + PT_STAGES;              // [group]
  uint64_t* s_empty = s_full + 2;                       // [group] (count 512: every softmax thread reads both S tiles)
  uint64_t* p_full = s_empty + 2;                       // [group][quarter] (count 128)
  uint64_t* p_empty = p_full + 8;                       // [group][quarter]
  uint64_t* o_full = p_empty + 8;                       // [group]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 2);
  float* sL = reinterpret_cast<float*>(bars + 64);      // [group][quarter][128] partial row sums
  static_assert(1 + 2 * PT_STAGES + 2 + 2 + 8 + 8 + 2 + 1 <= 64, "barrier block is 512 bytes");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * (2 * FA_BM);
  const int h = blockIdx.y, b = blockIdx.z;
  const int ntiles = (p.n_keys + FA_BN - 1) / FA_BN;
  const int nq_last = (p.n_keys - (ntiles - 1) * FA_BN + 31) >> 5;   // live 32-key quarters of the last tile (1..4)
  constexpr uint32_t TM_O = 256, TM_P = 384;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapQ);
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
    mbar_init(q_full, 1);
    for (int s = 0; s < PT_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 2); }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&s_full[g], 1);
      mbar_init(&s_empty[g], 512);
      mbar_init(&o_full[g], 1);
      for (int c = 0; c < 4; ++c) { mbar_init(&p_full[4 * g + c], 128); mbar_init(&p_empty[4 * g + c], 1); }
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, FA_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // provably warp-uniform (see elect_one in ptx.cuh)
  pdl_wait();

  if (warp == 0) {
    if (elect_one()) {
      // ---------------- TMA producer: both query tiles, then the K/V ring
      mbar_expect_tx(q_full, 2 * FA_Q_BYTES);
      for (int g = 0; g < 2; ++g) {
        if (p.q_heads_first) tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, h, row0 + g * FA_BM, b);
        else tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, row0 + g * FA_BM, h, b);
      }
      for (int j = 0; j < ntiles; ++j) {
        const int st = j % PT_STAGES;
        const uint32_t n = (uint32_t)(j / PT_STAGES);
        mbar_wait_sleep(&kv_empty[st], (n & 1u) ^ 1u, p.wait_ns);
        mbar_expect_tx(&kv_full[st], FA_KV_BYTES);
        uint8_t* dst = sKV + st * FA_KV_BYTES;
        if (p.kv_heads_first) {
          tma_load_4d(dst, &mapK, &kv_full[st], 0, h, j * FA_BN, b);
          tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, h, j * FA_BN, b);
        } else {
          tma_load_4d(dst, &mapK, &kv_full[st], 0, j * FA_BN, h, b);
          tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, j * FA_BN, h, b);
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    if (elect_one()) {
      // ---------------- MMA issuer of group g
      const int g = warp - 1;
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FA_BN >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint32_t idesc_pv = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(FA_D >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint64_t qdesc = make_sw128_kmajor_desc(smem_u32(sQ + g * FA_Q_BYTES));
      auto issue_s = [&](int j) {               // S_g(j) = Q_g K_j^T once every softmax thread has pulled S_g(j-1) into registers
        const int st = j % PT_STAGES;
        mbar_wait_sleep(&kv_full[st], (uint32_t)((j / PT_STAGES) & 1), p.wait_ns);
        mbar_wait_sleep(&s_empty[g], (uint32_t)((j & 1) ^ 1), p.wait_ns);
        tc_fence_after();
        const uint64_t bdesc = make_sw128_kmajor_desc(smem_u32(sKV + st * FA_KV_BYTES));
#pragma unroll
        for (int k = 0; k < FA_D / 16; ++k)
          umma_bf16(tmem_base + (uint32_t)(g * FA_BN), qdesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_s, k != 0 ? 1u : 0u);
        umma_commit(&s_full[g]);
      };
      mbar_wait_sleep(q_full, 0, p.wait_ns);
      issue_s(0);
      uint32_t acc = 0;
      for (int j = 0; j < ntiles; ++j) {
        if (j + 1 < ntiles) issue_s(j + 1);
        const int st = j % PT_STAGES;
        const uint32_t v_addr = smem_u32(sKV + st * FA_KV_BYTES + FA_K_BYTES);
        for (int u = 0; u < 4; ++u) {           // quarters in the order the softmax threads produce them for this group
          const int c = ((u & 1) << 1) | ((u >> 1) ^ g);   // g = 0: 0, 2, 1, 3;  g = 1: 1, 3, 0, 2
          if (j == ntiles - 1 && c >= nq_last) continue;
          mbar_wait_sleep(&p_full[4 * g + c], (uint32_t)(j & 1), p.wait_ns);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            // A: 16 keys = 8 packed columns of this quarter's P block; B: 16 key rows of V (MN-major, 2 KB)
            const uint32_t a_tmem = tmem_base + TM_P + (uint32_t)(g * 64 + c * 16 + k * 8);
            const uint64_t bdesc = make_sw128_mnmajor_desc(v_addr + (uint32_t)((c * 2 + k) * 16 * 128), 1024, 1024);
            umma_bf16_ts(tmem_base + TM_O + (uint32_t)(g * FA_D), a_tmem, bdesc, idesc_pv, acc);
            acc = 1u;
          }
          umma_commit(&p_empty[4 * g + c]);
        }
        umma_commit(&kv_empty[st]);             // one of the two arrivals that free K_j / V_j
      }
      umma_commit(&o_full[g]);
    }
  } else if (warp >= 4) {
    // ---------------- softmax / epilogue: thread = (query row r of BOTH tiles, 32-key quarter c)
    const int q = warp & 3;
    const int c = (warp - 4) >> 2;
    const int r = q * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const int g0 = c & 1, g1 = g0 ^ 1;                  // the tile this thread exponentiates first / second
    float l0 = 0.f, l1 = 0.f;                           // row sums of tile g0 / g1 over this quarter
    for (int j = 0; j < ntiles; ++j) {
      if (j == ntiles - 1 && c >= nq_last) break;       // no valid key in this quarter of the last tile
      const int kb = j * FA_BN + c * 32;
      const bool ragged = kb + 32 > p.n_keys;
      uint32_t s0[32], s1[32];
      mbar_wait_sleep(&s_full[g0], (uint32_t)(j & 1), p.wait_ns);
      tc_fence_after();
      tmem_ld32_nowait(tmem_base + lane_off + (uint32_t)(g0 * FA_BN + c * 32), s0);
      mbar_wait_sleep(&s_full[g1], (uint32_t)(j & 1), p.wait_ns);
      tc_fence_after();
      tmem_ld32_nowait(tmem_base + lane_off + (uint32_t)(g1 * FA_BN + c * 32), s1);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; ++i) { asm volatile("" : "+r"(s0[i])); asm volatile("" : "+r"(s1[i])); }   // pin behind the wait
      tc_fence_before();
      mbar_arrive(&s_empty[g0]);                        // this thread's share of both S tiles is in registers
      mbar_arrive(&s_empty[g1]);
      uint32_t pk[16];
      mbar_wait_sleep(&p_empty[4 * g0 + c], (uint32_t)((j & 1) ^ 1), p.wait_ns);   // P V of tile j-1 has read this quarter
      tc_fence_after();
      if (ragged) pt_chunk32<POLY, 1 | (MODE & 2), true>(s0, 0.f, kb, p.n_keys, pk, l0);
      else pt_chunk32<POLY, 1 | (MODE & 2), false>(s0, 0.f, kb, p.n_keys, pk, l0);
      tmem_st16(tmem_base + lane_off + TM_P + (uint32_t)(g0 * 64 + c * 16), pk);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&p_full[4 * g0 + c]);
      mbar_wait_sleep(&p_empty[4 * g1 + c], (uint32_t)((j & 1) ^ 1), p.wait_ns);
      tc_fence_after();
      if (ragged) pt_chunk32<POLY, 1 | (MODE & 2), true>(s1, 0.f, kb, p.n_keys, pk, l1);
      else pt_chunk32<POLY, 1 | (MODE & 2), false>(s1, 0.f, kb, p.n_keys, pk, l1);
      tmem_st16(tmem_base + lane_off + TM_P + (uint32_t)(g1 * 64 + c * 16), pk);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&p_full[4 * g1 + c]);
    }
    // ---- O / l -> global: the four quarter threads of a row add their sums; each stores 16 channels of both tiles
    mbar_wait_sleep(&o_full[0], 0, p.wait_ns);
    mbar_wait_sleep(&o_full[1], 0, p.wait_ns);
    tc_fence_after();
    sL[(g0 * 4 + c) * FA_BM + r] = l0;
    sL[(g1 * 4 + c) * FA_BM + r] = l1;
    asm volatile("bar.sync 1, 512;" ::: "memory");      // the 16 softmax warps
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      const float l = (sL[(g * 4 + 0) * FA_BM + r] + sL[(g * 4 + 1) * FA_BM + r]) + (sL[(g * 4 + 2) * FA_BM + r] + sL[(g * 4 + 3) * FA_BM + r]);
      const float inv = 1.f / l;
      uint32_t orr[16];
      tmem_ld16_nowait(tmem_base + lane_off + TM_O + (uint32_t)(g * FA_D + c * 16), orr);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 16; ++i) asm volatile("" : "+r"(orr[i]));
      const int row = row0 + g * FA_BM + r;
      if (row < p.rows) {
        __nv_bfloat16* orow = p.o + (long long)b * p.q_bs + (long long)h * p.q_hs + (long long)row * p.q_rs + c * 16;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          uint4 u;
          u.x = pack_bf16x2(__uint_as_float(orr[8 * t + 0]) * inv, __uint_as_float(orr[8 * t + 1]) * inv);
          u.y = pack_bf16x2(__uint_as_float(orr[8 * t + 2]) * inv, __uint_as_float(orr[8 * t + 3]) * inv);
          u.z = pack_bf16x2(__uint_as_float(orr[8 * t + 4]) * inv, __uint_as_float(orr[8 * t + 5]) * inv);
          u.w = pack_bf16x2(__uint_as_float(orr[8 * t + 6]) * inv, __uint_as_float(orr[8 * t + 7]) * inv);
          *reinterpret_cast<uint4*>(orow + 8 * t) = u;
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, FA_TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// PERSISTENT form of the kernel above (its measured default configuration: 16 softmax warps, scores preloaded, P = exp2(S), P in
// tensor memory).  tools/attn_keys_scan.py: a CTA of the one-shot kernel costs 5.4 us of launch / prologue / pipeline ramp / epilogue
// plus 1.15 us per key tile -- 12 % of the 64x64-level launch (33 tiles), 35 % of the 32x32-level one (9 tiles).  Here one CTA per SM
// walks the work items (256 query rows of one head of one sample) it_0 = blockIdx.x, it_0 + gridDim.x, ...: barriers, tensor memory
// and tensor-map prefetch are set up once, the K/V ring keeps streaming across item boundaries (the producer runs up to PT_STAGES
// tiles ahead, i.e. into the next item), the next item's Q tiles are fetched as soon as the last S MMA of the current item has read
// them, and S(0) of the next item is computed while the softmax warps still scale and store O of the current one.
// All barrier parities are derived from running counters (key tiles / handed-over P halves / items processed by THIS CTA).
// ------------------------------------------------------------------------------------------------------------------
struct FaPersist {
  int pairs_per_head;      // ceil(rows / 256)
  int n_heads;
  long long total_items;   // B * n_heads * pairs_per_head
};

template <int POLY, int MODE>   // MODE: bit 1 = no MUFU (bottleneck experiment, wrong results); bit 2 = per-CTA rotated key-tile order; bit 3 = S MMAs issued by a third thread
__global__ void __launch_bounds__(640, 1)
flash_attn_ptp_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                      const __grid_constant__ CUtensorMap mapV, const __grid_constant__ FaParams p, const __grid_constant__ FaPersist pp) {
  pdl_trigger();
  extern __shared__ uint8_t fa_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(fa_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                                   // [2] query tiles
  uint8_t* sKV = sQ + 2 * FA_Q_BYTES;                   // [PT_STAGES] {K, V}
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + PT_STAGES * FA_KV_BYTES);
  uint64_t* q_full = bars;                              // [1]
  uint64_t* q_empty = bars + 1;                         // [1] (count 2: the last S MMA of both groups)
  uint64_t* kv_full = bars + 2;                         // [PT_STAGES]
  uint64_t* kv_empty = kv_full + PT_STAGES;             // [PT_STAGES] (count 2: both groups' P V MMAs)
  uint64_t* s_full = kv_empty + PT_STAGES;              // [group]
  uint64_t* s_empty = s_full + 2;                       // [group] (count 256)
  uint64_t* p_full = s_empty + 2;                       // [group][half] (count 128)
  uint64_t* p_empty = p_full + 4;                       // [group][half]
  uint64_t* o_full = p_empty + 4;                       // [group]
  uint64_t* o_empty = o_full + 2;                       // [group] (count 8: one arrival per softmax warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_empty + 2);
  float* sL = reinterpret_cast<float*>(bars + 64);      // [group][sub][128] partial row sums
  static_assert(2 + 2 * PT_STAGES + 2 + 2 + 4 + 4 + 2 + 2 + 1 <= 64, "barrier block is 512 bytes");

  constexpr bool SPLIT = (MODE & 8) != 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (p.n_keys + FA_BN - 1) / FA_BN;
  const int dead = ((ntiles - 1) * FA_BN + 64 >= p.n_keys) ? 1 : 0;   // the last tile's second 64-key half holds no valid key
  constexpr uint32_t TM_O = 256, TM_P = 384;
  // The sum over key tiles has no running max, so its order is free: every CTA starts at a different tile.  The persistent CTAs start
  // together and stay in lock step; without the rotation all 148 SMs ask L2 for the same 32 KB K/V tile at the same moment.
  const int rot = (MODE & 4) ? (int)((blockIdx.x * 5u) % (uint32_t)ntiles) : 0;
  const int jd = (ntiles - 1 - rot + ntiles) % ntiles;       // loop position of the last (possibly half-dead, possibly ragged) tile

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapQ);
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
    mbar_init(q_full, 1);
    mbar_init(q_empty, SPLIT ? 1 : 2);
    for (int s = 0; s < PT_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 2); }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&s_full[g], 1);
      mbar_init(&s_empty[g], 256);
      mbar_init(&o_full[g], 1);
      mbar_init(&o_empty[g], 8);
      for (int i = 0; i < 2; ++i) { mbar_init(&p_full[2 * g + i], 128); mbar_init(&p_empty[2 * g + i], 1); }
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, FA_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // provably warp-uniform (see elect_one in ptx.cuh)
  pdl_wait();

  if (warp == 0) {
    if (elect_one()) {
      // ---------------- TMA producer
      uint32_t T = 0;                                   // key tiles loaded by this CTA so far
      int n = 0;
      for (long long it = blockIdx.x; it < pp.total_items; it += gridDim.x, ++n) {
        const int pair = (int)(it % pp.pairs_per_head);
        const int h = (int)((it / pp.pairs_per_head) % pp.n_heads), b = (int)(it / ((long long)pp.pairs_per_head * pp.n_heads));
        const int row0 = pair * (2 * FA_BM);
        if (n > 0) mbar_wait_sleep(q_empty, (uint32_t)((n - 1) & 1), p.wait_ns);   // the previous item's last S MMAs have read Q
        mbar_expect_tx(q_full, 2 * FA_Q_BYTES);
        for (int g = 0; g < 2; ++g) {
          if (p.q_heads_first) tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, h, row0 + g * FA_BM, b);
          else tma_load_4d(sQ + g * FA_Q_BYTES, &mapQ, q_full, 0, row0 + g * FA_BM, h, b);
        }
        for (int j = 0; j < ntiles; ++j, ++T) {
          const int st = (int)(T % PT_STAGES);
          mbar_wait_sleep(&kv_empty[st], ((T / PT_STAGES) & 1u) ^ 1u, p.wait_ns);
          mbar_expect_tx(&kv_full[st], FA_KV_BYTES);
          uint8_t* dst = sKV + st * FA_KV_BYTES;
          const int jt = j + rot < ntiles ? j + rot : j + rot - ntiles;
          if (p.kv_heads_first) {
            tma_load_4d(dst, &mapK, &kv_full[st], 0, h, jt * FA_BN, b);
            tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, h, jt * FA_BN, b);
          } else {
            tma_load_4d(dst, &mapK, &kv_full[st], 0, jt * FA_BN, h, b);
            tma_load_4d(dst + FA_K_BYTES, &mapV, &kv_full[st], 0, jt * FA_BN, h, b);
          }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    if (elect_one()) {
      // ---------------- MMA issuer of group g
      const int g = warp - 1;
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FA_BN >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint32_t idesc_pv = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(FA_D >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint64_t qdesc = make_sw128_kmajor_desc(smem_u32(sQ + g * FA_Q_BYTES));
      uint32_t T0 = 0, H1 = 0;                          // key tiles / second-half P hand-overs before the current item
      int n = 0;
      for (long long it = blockIdx.x; it < pp.total_items; it += gridDim.x, ++n, T0 += (uint32_t)ntiles, H1 += (uint32_t)(ntiles - dead)) {
        auto issue_s = [&](int j) {                     // S_g(j) = Q_g K_j^T once group g has pulled its previous S into registers
          const uint32_t T = T0 + (uint32_t)j;
          const int st = (int)(T % PT_STAGES);
          mbar_wait_sleep(&kv_full[st], (T / PT_STAGES) & 1u, p.wait_ns);
          mbar_wait_sleep(&s_empty[g], (T & 1u) ^ 1u, p.wait_ns);
          tc_fence_after();
          const uint64_t bdesc = make_sw128_kmajor_desc(smem_u32(sKV + st * FA_KV_BYTES));
#pragma unroll
          for (int k = 0; k < FA_D / 16; ++k)
            umma_bf16(tmem_base + (uint32_t)(g * FA_BN), qdesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_s, k != 0 ? 1u : 0u);
          umma_commit(&s_full[g]);
          if (j == ntiles - 1) umma_commit(q_empty);    // Q of this item is no longer needed by this group
        };
        if (!SPLIT) {
          mbar_wait_sleep(q_full, (uint32_t)(n & 1), p.wait_ns);
          issue_s(0);
        }
        for (int j = 0; j < ntiles; ++j) {
          if (!SPLIT && j + 1 < ntiles) issue_s(j + 1);
          const uint32_t T = T0 + (uint32_t)j;
          const int st = (int)(T % PT_STAGES);
          if (SPLIT) mbar_wait_sleep(&kv_full[st], (T / PT_STAGES) & 1u, p.wait_ns);   // V_j has landed (this thread did not issue S_j)
          const uint32_t v_addr = smem_u32(sKV + st * FA_KV_BYTES + FA_K_BYTES);
          for (int hf = 0; hf < 2; ++hf) {              // the first 64 keys are multiplied while the second 64 are exponentiated
            if (hf == 1 && dead && j == jd) break;
            const int pb = 2 * g + hf;
            const uint32_t ph = hf == 0 ? T : H1 + (uint32_t)(j - ((dead && j > jd) ? 1 : 0));
            mbar_wait_sleep(&p_full[pb], ph & 1u, p.wait_ns);
            if (j == 0 && hf == 0) mbar_wait_sleep(&o_empty[g], (uint32_t)((n & 1) ^ 1), p.wait_ns);   // the previous item's O has been read
            tc_fence_after();
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t a_tmem = tmem_base + TM_P + (uint32_t)(g * 64 + hf * 32 + k * 8);
              const uint64_t bdesc = make_sw128_mnmajor_desc(v_addr + (uint32_t)((hf * 4 + k) * 16 * 128), 1024, 1024);
              umma_bf16_ts(tmem_base + TM_O + (uint32_t)(g * FA_D), a_tmem, bdesc, idesc_pv, (j | hf | k) != 0 ? 1u : 0u);
            }
            umma_commit(&p_empty[pb]);
          }
          umma_commit(&kv_empty[st]);                   // one of the two arrivals that free K_j / V_j
        }
        umma_commit(&o_full[g]);
      }
    }
  } else if (SPLIT && warp == 3) {
    if (elect_one()) {
      // ---------------- S issuer of both groups
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FA_BN >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint64_t qdesc0 = make_sw128_kmajor_desc(smem_u32(sQ));
      const uint64_t kdesc0 = make_sw128_kmajor_desc(smem_u32(sKV));
      uint32_t T = 0;
      int n = 0;
      for (long long it = blockIdx.x; it < pp.total_items; it += gridDim.x, ++n) {
        mbar_wait_sleep(q_full, (uint32_t)(n & 1), p.wait_ns);
        for (int j = 0; j < ntiles; ++j, ++T) {
          const int st = (int)(T % PT_STAGES);
          mbar_wait_sleep(&kv_full[st], (T / PT_STAGES) & 1u, p.wait_ns);
          const uint64_t bdesc = kdesc0 + (uint64_t)(st * (FA_KV_BYTES >> 4));
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            mbar_wait_sleep(&s_empty[g], (T & 1u) ^ 1u, p.wait_ns);   // group g has pulled its previous S into registers
            tc_fence_after();
#pragma unroll
            for (int k = 0; k < FA_D / 16; ++k)
              umma_bf16(tmem_base + (uint32_t)(g * FA_BN), qdesc0 + (uint64_t)(g * (FA_Q_BYTES >> 4) + 2 * k), bdesc + (uint64_t)(2 * k), idesc_s, k != 0 ? 1u : 0u);
            umma_commit(&s_full[g]);
          }
          if (j == ntiles - 1) umma_commit(q_empty);    // Q of this item is no longer needed
        }
      }
    }
  } else if (warp >= 4) {
    // ---------------- softmax / epilogue: group g, thread = (query row of that group, 64-key half)
    const int idx = warp - 4;
    const int g = idx >> 3;
    const int sub = (idx >> 2) & 1;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const int pb = 2 * g + sub;
    const uint32_t p_col = tmem_base + lane_off + TM_P + (uint32_t)(g * 64 + sub * 32);
    float* sLg = sL + g * 2 * FA_BM;
    uint32_t T0 = 0, H1 = 0;
    int n = 0;
    for (long long it = blockIdx.x; it < pp.total_items; it += gridDim.x, ++n, T0 += (uint32_t)ntiles, H1 += (uint32_t)(ntiles - dead)) {
      const int pair = (int)(it % pp.pairs_per_head);
      const int h = (int)((it / pp.pairs_per_head) % pp.n_heads), b = (int)(it / ((long long)pp.pairs_per_head * pp.n_heads));
      const int row0 = pair * (2 * FA_BM);
      float l = 0.f;
      for (int j = 0; j < ntiles; ++j) {
        const uint32_t T = T0 + (uint32_t)j;
        const int key0 = (j + rot < ntiles ? j + rot : j + rot - ntiles) * FA_BN;
        mbar_wait_sleep(&s_full[g], T & 1u, p.wait_ns);
        tc_fence_after();
        if (sub == 1 && dead && j == jd) {              // nothing valid in this warp's half of the last tile: only release S
          tc_fence_before();
          mbar_arrive(&s_empty[g]);
          continue;
        }
        uint32_t sr[64];
        tmem_ld32_nowait(tmem_base + lane_off + (uint32_t)(g * FA_BN + sub * 64), sr);
        tmem_ld32_nowait(tmem_base + lane_off + (uint32_t)(g * FA_BN + sub * 64 + 32), sr + 32);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 64; ++i) asm volatile("" : "+r"(sr[i]));   // pin the destination registers behind the wait
        tc_fence_before();
        mbar_arrive(&s_empty[g]);                       // this thread's share of S_g is in registers
        const uint32_t ph = sub == 0 ? T : H1 + (uint32_t)(j - ((dead && j > jd) ? 1 : 0));
        mbar_wait_sleep(&p_empty[pb], (ph & 1u) ^ 1u, p.wait_ns);   // the P V MMAs of the previous tile have finished reading this half of P
        tc_fence_after();
        const bool ragged = key0 + FA_BN > p.n_keys;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          uint32_t pk[16];
          const int kb = key0 + sub * 64 + 32 * t;
          if (ragged) pt_chunk32<POLY, 1 | (MODE & 2), true>(sr + 32 * t, 0.f, kb, p.n_keys, pk, l);
          else pt_chunk32<POLY, 1 | (MODE & 2), false>(sr + 32 * t, 0.f, kb, p.n_keys, pk, l);
          tmem_st16(p_col + (uint32_t)(16 * t), pk);
        }
        tmem_st_wait();                                 // the stores have landed in tensor memory ...
        tc_fence_before();                              // ... and are ordered before the issuer's MMAs through the barrier
        mbar_arrive(&p_full[pb]);
      }
      // ---- O / l -> global: the two column-half threads of a row add their sums and each stores 32 channels
      mbar_wait_sleep(&o_full[g], (uint32_t)(n & 1), p.wait_ns);
      tc_fence_after();
      sLg[sub * FA_BM + r] = l;
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");         // the 8 softmax warps of this group
      l = sLg[r] + sLg[FA_BM + r];
      uint32_t orr[32];
      tmem_ld32_nowait(tmem_base + lane_off + TM_O + (uint32_t)(g * FA_D + sub * 32), orr);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; ++i) asm volatile("" : "+r"(orr[i]));
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[g]);          // O_g may be overwritten by the next item's first P V MMA
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");         // sLg is rewritten by the next item only after everybody has read it
      const float inv = 1.f / l;
      const int row = row0 + g * FA_BM + r;
      if (row < p.rows) {
        __nv_bfloat16* orow = p.o + (long long)b * p.q_bs + (long long)h * p.q_hs + (long long)row * p.q_rs + sub * 32;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          uint4 u;
          u.x = pack_bf16x2(__uint_as_float(orr[8 * t + 0]) * inv, __uint_as_float(orr[8 * t + 1]) * inv);
          u.y = pack_bf16x2(__uint_as_float(orr[8 * t + 2]) * inv, __uint_as_float(orr[8 * t + 3]) * inv);
          u.z = pack_bf16x2(__uint_as_float(orr[8 * t + 4]) * inv, __uint_as_float(orr[8 * t + 5]) * inv);
          u.w = pack_bf16x2(__uint_as_float(orr[8 * t + 6]) * inv, __uint_as_float(orr[8 * t + 7]) * inv);
          *reinterpret_cast<uint4*>(orow + 8 * t) = u;
        }
      }
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, FA_TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Few-keys (cross-) attention on tcgen05: <= 64 keys per head (the 39 context rows of CrossAttention).  The work is memory bound
// (q in, o out: 268 MB at the 64x64 level), so the kernel is PERSISTENT: one CTA per SM walks a contiguous range of work items
// (sample b, 128-row query tile, head h); the K and V rows of all heads of the current sample stay resident in shared memory
// (2 x 64 KB, reloaded when b changes), Q tiles stream through a 4-stage TMA ring, and three TMEM "slots" (S 64 + P 32 + O 64 columns)
// keep three items in flight:   S = Q K_h^T  (M128 x N64 x K64)  ->  4 worker warps: tcgen05.ld, P = exp2(S) (bounded cosine-sim logits,
// keys >= n_keys masked), row sum, P -> tensor memory  ->  O = P V_h  (A operand from TMEM)  ->  same warps: O / l -> bf16 -> one
// 128-byte row store per thread.  Replaces the mma.sync kernel (2.3 TB/s; its mma.sync + MUFU work alone is ~45 us per launch).
// ------------------------------------------------------------------------------------------------------------------
constexpr int XA_NS = 3;                           // TMEM slots / items in flight
constexpr int XA_QS = 4;                           // Q ring stages
constexpr int XA_KEYS = 64;                        // key tile (rows beyond n_keys are zero-filled by TMA and masked)
constexpr int XA_KV_HEAD_BYTES = XA_KEYS * 64 * 2; // one head's K (or V) tile: 8 KB
constexpr int XA_MAX_HEADS = 8;
constexpr int XA_SMEM = XA_QS * FA_Q_BYTES + 2 * XA_MAX_HEADS * XA_KV_HEAD_BYTES + 1024 + 512;

struct XaParams {
  __nv_bfloat16* o;
  long long q_bs;          // elements between samples in q / o
  int q_rs, q_hs;          // row / head strides of q and o (elements)
  int rows, n_keys, B, heads;
  int tiles_per_sample;    // ceil(rows / 128)
  int items_per_cta;
  uint32_t wait_ns;
};

__global__ void __launch_bounds__(64 + 128 * XA_NS, 1)
cross_attn_tc_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapV,
                     const __grid_constant__ XaParams p) {
  pdl_trigger();
  extern __shared__ uint8_t fa_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(fa_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                                        // [XA_QS] query tiles
  uint8_t* sK = sQ + XA_QS * FA_Q_BYTES;                     // [heads] K tiles of the current sample
  uint8_t* sV = sK + XA_MAX_HEADS * XA_KV_HEAD_BYTES;        // [heads] V tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + XA_MAX_HEADS * XA_KV_HEAD_BYTES);
  uint64_t* q_full = bars;                       // [XA_QS]
  uint64_t* q_empty = q_full + XA_QS;            // [XA_QS]
  uint64_t* kv_full = q_empty + XA_QS;           // [1]
  uint64_t* kv_empty = kv_full + 1;              // [1]
  uint64_t* s_full = kv_empty + 1;               // [XA_NS]
  uint64_t* p_full = s_full + XA_NS;             // [XA_NS]
  uint64_t* o_full = p_full + XA_NS;             // [XA_NS]
  uint64_t* slot_free = o_full + XA_NS;          // [XA_NS]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(slot_free + XA_NS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long total_items = (long long)p.B * p.tiles_per_sample * p.heads;
  const long long item0 = (long long)blockIdx.x * p.items_per_cta;
  const long long item1 = item0 + p.items_per_cta < total_items ? item0 + p.items_per_cta : total_items;
  const int n_items = item1 > item0 ? (int)(item1 - item0) : 0;
  const int per_sample = p.tiles_per_sample * p.heads;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapQ);
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
    for (int s = 0; s < XA_QS; ++s) { mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 1); }
    mbar_init(kv_full, 1);
    mbar_init(kv_empty, 1);
    for (int s = 0; s < XA_NS; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 4);       // one arrival per worker warp of the slot
      mbar_init(&o_full[s], 1);
      mbar_init(&slot_free[s], 4);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // provably warp-uniform (see elect_one in ptx.cuh)
  pdl_wait();
  // TMEM columns: accumulators on 64-column boundaries (S_s at 128 s, O_s at 128 s + 64), the packed P tiles behind them (384 + 32 s)
  constexpr uint32_t SLOT_COLS = 128, P_BASE = 384;

  if (warp == 0) {
    if (elect_one()) {
      // ---------------- TMA producer: K/V of all heads whenever the sample changes, then one Q tile per item
      int cur_b = -1, epoch = 0;
      for (int i = 0; i < n_items; ++i) {
        const long long it = item0 + i;
        const int b = (int)(it / per_sample), rem = (int)(it % per_sample);
        const int tile = rem / p.heads, h = rem % p.heads;
        if (b != cur_b) {
          mbar_wait_sleep(kv_empty, (uint32_t)((epoch & 1) ^ 1), p.wait_ns);      // every MMA that read the previous sample's K/V has completed
          mbar_expect_tx(kv_full, (uint32_t)(2 * p.heads * XA_KV_HEAD_BYTES));
          for (int hh = 0; hh < p.heads; ++hh) {
            tma_load_4d(sK + hh * XA_KV_HEAD_BYTES, &mapK, kv_full, 0, hh, 0, b);
            tma_load_4d(sV + hh * XA_KV_HEAD_BYTES, &mapV, kv_full, 0, hh, 0, b);
          }
          cur_b = b;
          ++epoch;
        }
        const int st = i % XA_QS;
        mbar_wait_sleep(&q_empty[st], (uint32_t)(((i / XA_QS) & 1) ^ 1), p.wait_ns);
        mbar_expect_tx(&q_full[st], FA_Q_BYTES);
        tma_load_4d(sQ + st * FA_Q_BYTES, &mapQ, &q_full[st], 0, h, tile * FA_BM, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      // ---------------- MMA issuer
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(XA_KEYS >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      const uint32_t idesc_pv = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(FA_D >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      int epoch = 0, kv_b = -1;
      auto item_b = [&](int i) { return (int)((item0 + i) / per_sample); };
      auto item_h = [&](int i) { return (int)((item0 + i) % p.heads); };   // per_sample is a multiple of heads
      auto issue_s = [&](int i) {
        const int b = item_b(i), h = item_h(i), st = i % XA_QS, slot = i % XA_NS;
        if (b != kv_b) {
          mbar_wait_sleep(kv_full, (uint32_t)(epoch & 1), p.wait_ns);
          kv_b = b;
          ++epoch;
        }
        mbar_wait_sleep(&q_full[st], (uint32_t)((i / XA_QS) & 1), p.wait_ns);
        mbar_wait_sleep(&slot_free[slot], (uint32_t)(((i / XA_NS) & 1) ^ 1), p.wait_ns);   // the workers have stored the item that used this slot
        tc_fence_after();
        const uint64_t adesc = make_sw128_kmajor_desc(smem_u32(sQ + st * FA_Q_BYTES));
        const uint64_t bdesc = make_sw128_kmajor_desc(smem_u32(sK + h * XA_KV_HEAD_BYTES));
#pragma unroll
        for (int k = 0; k < FA_D / 16; ++k)
          umma_bf16(tmem_base + (uint32_t)(slot * SLOT_COLS), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_s, k != 0 ? 1u : 0u);
        umma_commit(&s_full[slot]);
        umma_commit(&q_empty[st]);
      };
      if (n_items > 0) issue_s(0);
      for (int i = 0; i < n_items; ++i) {
        const bool next_same_sample = i + 1 < n_items && item_b(i + 1) == item_b(i);
        if (next_same_sample) issue_s(i + 1);              // scores of the next item while the workers exponentiate this one
        const int slot = i % XA_NS, h = item_h(i);
        mbar_wait_sleep(&p_full[slot], (uint32_t)((i / XA_NS) & 1), p.wait_ns);
        tc_fence_after();
        const uint32_t v_addr = smem_u32(sV + h * XA_KV_HEAD_BYTES);
#pragma unroll
        for (int k = 0; k < XA_KEYS / 16; ++k) {
          const uint32_t a_tmem = tmem_base + P_BASE + (uint32_t)(slot * 32 + k * 8);
          const uint64_t bdesc = make_sw128_mnmajor_desc(v_addr + (uint32_t)(k * 16 * 128), 1024, 1024);
          umma_bf16_ts(tmem_base + (uint32_t)(slot * SLOT_COLS + 64), a_tmem, bdesc, idesc_pv, k != 0 ? 1u : 0u);
        }
        umma_commit(&o_full[slot]);
        if (i + 1 < n_items && !next_same_sample) {
          umma_commit(kv_empty);                            // all MMAs of this sample are issued: its K/V may be replaced once they complete
          issue_s(i + 1);
        }
      }
    }
  } else {
    // ---------------- workers: slot = (warp - 2) / 4, thread = one query row of every item of its slot
    const int slot = (warp - 2) >> 2;
    const int q4 = warp & 3;
    const int r = q4 * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q4 * 32) << 16;
    const uint32_t t_s = tmem_base + lane_off + (uint32_t)(slot * SLOT_COLS);
    const uint32_t t_p = tmem_base + lane_off + P_BASE + (uint32_t)(slot * 32);
    for (int i = slot; i < n_items; i += XA_NS) {
      const long long it = item0 + i;
      const int b = (int)(it / per_sample), rem = (int)(it % per_sample);
      const int tile = rem / p.heads, h = rem % p.heads;
      const uint32_t par = (uint32_t)((i / XA_NS) & 1);
      mbar_wait_sleep(&s_full[slot], par, p.wait_ns);
      tc_fence_after();
      float l = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < XA_KEYS; c0 += 32) {
        uint32_t sr[32], pk[16];
        tmem_ld32_nowait(t_s + (uint32_t)c0, sr);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) asm volatile("" : "+r"(sr[j]));
        pt_chunk32<0, 1, true>(sr, 0.f, c0, p.n_keys, pk, l);
        tmem_st16(t_p + (uint32_t)(c0 >> 1), pk);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[slot]);
      mbar_wait_sleep(&o_full[slot], par, p.wait_ns);
      tc_fence_after();
      const float inv = 1.f / l;
      const int row = tile * FA_BM + r;
      __nv_bfloat16* orow = p.o + (long long)b * p.q_bs + (long long)row * p.q_rs + (long long)h * p.q_hs;
#pragma unroll
      for (int c0 = 0; c0 < FA_D; c0 += 32) {
        uint32_t orr[32];
        tmem_ld32_nowait(t_s + 64u + (uint32_t)c0, orr);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) asm volatile("" : "+r"(orr[j]));
        if (row < p.rows) {
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            uint4 u;
            u.x = pack_bf16x2(__uint_as_float(orr[8 * t + 0]) * inv, __uint_as_float(orr[8 * t + 1]) * inv);
            u.y = pack_bf16x2(__uint_as_float(orr[8 * t + 2]) * inv, __uint_as_float(orr[8 * t + 3]) * inv);
            u.z = pack_bf16x2(__uint_as_float(orr[8 * t + 4]) * inv, __uint_as_float(orr[8 * t + 5]) * inv);
            u.w = pack_bf16x2(__uint_as_float(orr[8 * t + 6]) * inv, __uint_as_float(orr[8 * t + 7]) * inv);
            *reinterpret_cast<uint4*>(orow + c0 + 8 * t) = u;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&slot_free[slot]);
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512u);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Linear cross-attention (LinearCrossAttention.forward, imagen_pytorch.py:836-874):
//   out = softmax_d(q) @ C,   C[d, e] = 8 * sum_j softmax_j(k)[j, d] * v[j, e]      (per sample row and head)
// Unlike CrossAttention there is no per-pixel score matrix: the keys enter only through the dim_head x dim_head matrix C.
// linear_xattn_context_kernel builds C once per step (the time-token K/V rows change every step) and stores it bf16 as
// [B][heads][64 d][64 e], the layout of a V tile, so that the main kernel loads it with the same TMA map / MN-major
// descriptor as cross_attn_tc_kernel's V.  Head channels >= dim_head (zero-padded heads) get C rows of exact zeros.
// ------------------------------------------------------------------------------------------------------------------
constexpr int LX_CTX_THREADS = 256;
constexpr int LX_CTX_SMEM = 2 * 64 * 64 * 4 + 2 * 64 * 4;   // one 64-token chunk of softmax_j(k) and of v (fp32) + column max / scale

__global__ void __launch_bounds__(LX_CTX_THREADS)
linear_xattn_context_kernel(const __nv_bfloat16* __restrict__ k, const __nv_bfloat16* __restrict__ v, long long kv_bs, int kv_rs, int n_keys,
                            int dim_head, __nv_bfloat16* __restrict__ ctx) {
  pdl_trigger();
  extern __shared__ float lx_smem[];
  float* sW = lx_smem;               // [64 tokens][64 d]: exp(k - max_d) * 8 / sum_d
  float* sV = sW + 64 * 64;          // [64 tokens][64 e]
  float* sMax = sV + 64 * 64;        // [64]
  float* sScale = sMax + 64;         // [64]
  const int h = blockIdx.x, b = blockIdx.y, heads = gridDim.x, tid = threadIdx.x;
  const __nv_bfloat16* kb = k + (long long)b * kv_bs + h * 64;
  const __nv_bfloat16* vb = v + (long long)b * kv_bs + h * 64;
  pdl_wait();
  // column statistics of k over the tokens (softmax over dim -2), fp32 with a true max: the logits are unbounded
  if (tid < 64) {
    float m = -INFINITY;
    for (int j = 0; j < n_keys; ++j) m = fmaxf(m, __bfloat162float(kb[(long long)j * kv_rs + tid]));
    float s = 0.f;
    for (int j = 0; j < n_keys; ++j) s += __expf(__bfloat162float(kb[(long long)j * kv_rs + tid]) - m);
    sMax[tid] = m;
    sScale[tid] = tid < dim_head ? 8.f / s : 0.f;   // CrossAttention's scale = 8 on q, folded into C (q @ C is linear)
  }
  const int e = tid & 63, d0 = tid >> 6;            // this thread: C[d0 + 4 i][e], i < 16
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  for (int j0 = 0; j0 < n_keys; j0 += 64) {
    const int nj = n_keys - j0 < 64 ? n_keys - j0 : 64;
    __syncthreads();                                 // statistics ready / previous chunk consumed
    for (int idx = tid; idx < nj * 64; idx += LX_CTX_THREADS) {
      const int j = idx >> 6, c = idx & 63;
      const long long off = (long long)(j0 + j) * kv_rs + c;
      sW[idx] = __expf(__bfloat162float(kb[off]) - sMax[c]) * sScale[c];
      sV[idx] = __bfloat162float(vb[off]);
    }
    __syncthreads();
    for (int j = 0; j < nj; ++j) {
      const float vv = sV[j * 64 + e];
#pragma unroll
      for (int i = 0; i < 16; ++i) acc[i] = fmaf(sW[j * 64 + d0 + 4 * i], vv, acc[i]);
    }
  }
  __nv_bfloat16* cb = ctx + ((long long)b * heads + h) * 64 * 64;
#pragma unroll
  for (int i = 0; i < 16; ++i) cb[(d0 + 4 * i) * 64 + e] = __float2bfloat16_rn(acc[i]);
}

// Main kernel, persistent like cross_attn_tc_kernel: one CTA per SM walks a contiguous range of work items (sample b, 128-row query
// tile, head h).  The C tiles of all heads of the current sample stay resident in shared memory (8 x 8 KB, reloaded when b changes),
// q tiles stream through a TMA ring, and LX_NS tensor-memory slots (O 64 columns + P 32 columns) keep LX_NS items in flight:
//   4 worker warps per slot: q row from shared memory -> softmax over the first dim_head channels in fp32 (one thread per row) ->
//   P (bf16, exact zeros in padded channels) -> tensor memory  ->  O = P C (TS-form tcgen05.mma, M128 x N64 x K64)  ->
//   the same warps: tcgen05.ld O -> bf16 -> one 128-byte row store per thread.
// The softmax already normalises each row and C carries the 8, so O needs no further scaling.
constexpr int LX_NS = 4;                               // TMEM slots / items in flight
constexpr int LX_QS = 6;                               // q ring stages
constexpr int LX_CTX_BYTES = 64 * 64 * 2;              // one head's C tile: 8 KB
constexpr int LX_MAX_HEADS = 8;
constexpr int LX_SMEM = LX_QS * FA_Q_BYTES + LX_MAX_HEADS * LX_CTX_BYTES + 1024 + 512;

struct LxParams {
  __nv_bfloat16* o;
  long long q_bs;          // elements between samples in q / o
  int q_rs;                // row stride of q and o (elements); head h starts at column 64 h
  int rows, B, heads, dim_head;
  int tiles_per_sample;    // ceil(rows / 128)
  int items_per_cta;
  uint32_t wait_ns;
};

__global__ void __launch_bounds__(64 + 128 * LX_NS, 1)
linear_cross_attn_tc_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapC, const __grid_constant__ LxParams p) {
  pdl_trigger();
  extern __shared__ uint8_t fa_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(fa_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                                        // [LX_QS] q tiles
  uint8_t* sC = sQ + LX_QS * FA_Q_BYTES;                     // [heads] C tiles of the current sample
  uint64_t* bars = reinterpret_cast<uint64_t*>(sC + LX_MAX_HEADS * LX_CTX_BYTES);
  uint64_t* q_full = bars;                       // [LX_QS]
  uint64_t* q_empty = q_full + LX_QS;            // [LX_QS]
  uint64_t* c_full = q_empty + LX_QS;            // [1]
  uint64_t* c_empty = c_full + 1;                // [1]
  uint64_t* p_full = c_empty + 1;                // [LX_NS]
  uint64_t* o_full = p_full + LX_NS;             // [LX_NS]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + LX_NS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long total_items = (long long)p.B * p.tiles_per_sample * p.heads;
  const long long item0 = (long long)blockIdx.x * p.items_per_cta;
  const long long item1 = item0 + p.items_per_cta < total_items ? item0 + p.items_per_cta : total_items;
  const int n_items = item1 > item0 ? (int)(item1 - item0) : 0;
  const int per_sample = p.tiles_per_sample * p.heads;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapQ);
    tma_prefetch_desc(&mapC);
    for (int s = 0; s < LX_QS; ++s) { mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 4); }   // q_empty: one arrival per worker warp
    mbar_init(c_full, 1);
    mbar_init(c_empty, 1);
    for (int s = 0; s < LX_NS; ++s) {
      mbar_init(&p_full[s], 4);
      mbar_init(&o_full[s], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  pdl_wait();
  // TMEM columns: O of slot s at 64 s, the packed P tiles behind them (256 + 32 s)
  constexpr uint32_t P_BASE = 64 * LX_NS;

  if (warp == 0) {
    if (elect_one()) {
      // ---------------- TMA producer: C of all heads whenever the sample changes, then one q tile per item
      int cur_b = -1, epoch = 0;
      for (int i = 0; i < n_items; ++i) {
        const long long it = item0 + i;
        const int b = (int)(it / per_sample), rem = (int)(it % per_sample);
        const int tile = rem / p.heads, h = rem % p.heads;
        if (b != cur_b) {
          mbar_wait_sleep(c_empty, (uint32_t)((epoch & 1) ^ 1), p.wait_ns);      // every MMA that read the previous sample's C has completed
          mbar_expect_tx(c_full, (uint32_t)(p.heads * LX_CTX_BYTES));
          for (int hh = 0; hh < p.heads; ++hh) tma_load_4d(sC + hh * LX_CTX_BYTES, &mapC, c_full, 0, 0, hh, b);
          cur_b = b;
          ++epoch;
        }
        const int st = i % LX_QS;
        mbar_wait_sleep(&q_empty[st], (uint32_t)(((i / LX_QS) & 1) ^ 1), p.wait_ns);
        mbar_expect_tx(&q_full[st], FA_Q_BYTES);
        tma_load_4d(sQ + st * FA_Q_BYTES, &mapQ, &q_full[st], 0, h, tile * FA_BM, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      // ---------------- MMA issuer: O = P C per item, P from tensor memory
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(FA_D >> 3) << 17) | ((uint32_t)(FA_BM >> 4) << 24);
      int epoch = 0, c_b = -1;
      for (int i = 0; i < n_items; ++i) {
        const long long it = item0 + i;
        const int b = (int)(it / per_sample), h = (int)(it % p.heads);   // per_sample is a multiple of heads
        const int slot = i % LX_NS;
        if (b != c_b) {
          mbar_wait_sleep(c_full, (uint32_t)(epoch & 1), p.wait_ns);
          c_b = b;
          ++epoch;
        }
        mbar_wait_sleep(&p_full[slot], (uint32_t)((i / LX_NS) & 1), p.wait_ns);
        tc_fence_after();
        const uint32_t c_addr = smem_u32(sC + h * LX_CTX_BYTES);
#pragma unroll
        for (int k = 0; k < FA_D / 16; ++k) {
          const uint32_t a_tmem = tmem_base + P_BASE + (uint32_t)(slot * 32 + k * 8);
          const uint64_t bdesc = make_sw128_mnmajor_desc(c_addr + (uint32_t)(k * 16 * 128), 1024, 1024);
          umma_bf16_ts(tmem_base + (uint32_t)(slot * 64), a_tmem, bdesc, idesc, k != 0 ? 1u : 0u);
        }
        umma_commit(&o_full[slot]);
        const bool next_same_sample = i + 1 < n_items && (int)((it + 1) / per_sample) == b;
        if (i + 1 < n_items && !next_same_sample) umma_commit(c_empty);   // this sample's C may be replaced once its MMAs complete
      }
    }
  } else {
    // ---------------- workers: slot = (warp - 2) / 4, thread = one query row of every item of its slot
    const int slot = (warp - 2) >> 2;
    const int q4 = warp & 3;
    const int r = q4 * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q4 * 32) << 16;
    const uint32_t t_o = tmem_base + lane_off + (uint32_t)(slot * 64);
    const uint32_t t_p = tmem_base + lane_off + P_BASE + (uint32_t)(slot * 32);
    constexpr float LOG2E_F = 1.4426950408889634f;
    for (int i = slot; i < n_items; i += LX_NS) {
      const long long it = item0 + i;
      const int b = (int)(it / per_sample), rem = (int)(it % per_sample);
      const int tile = rem / p.heads, h = rem % p.heads;
      const int st = i % LX_QS;
      mbar_wait_sleep(&q_full[st], (uint32_t)((i / LX_QS) & 1), p.wait_ns);
      // this thread's q row: 8 x 16-byte chunks, chunk c of row r at position c ^ (r & 7) (128-byte swizzle)
      const uint8_t* qrow = sQ + st * FA_Q_BYTES + r * 128;
      float x[64];
#pragma unroll
      for (int c = 0; c < 8; ++c) unpack8(*reinterpret_cast<const uint4*>(qrow + ((c ^ (r & 7)) << 4)), x + 8 * c);
      __syncwarp();
      if (lane == 0) mbar_arrive(&q_empty[st]);
      // softmax over the head width (dim -1), fp32 with a true max: q is unbounded
      float m = -INFINITY;
#pragma unroll
      for (int d = 0; d < 64; ++d)
        if (d < p.dim_head) m = fmaxf(m, x[d]);
      const float mb = m * LOG2E_F;
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < 64; ++d) {
        x[d] = d < p.dim_head ? ex2_approx(fmaf(x[d], LOG2E_F, -mb)) : 0.f;
        s += x[d];
      }
      const float inv = 1.f / s;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(x[32 * half + 2 * j] * inv, x[32 * half + 2 * j + 1] * inv);
        tmem_st16(t_p + (uint32_t)(16 * half), pk);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[slot]);
      mbar_wait_sleep(&o_full[slot], (uint32_t)((i / LX_NS) & 1), p.wait_ns);
      tc_fence_after();
      const int row = tile * FA_BM + r;
      __nv_bfloat16* orow = p.o + (long long)b * p.q_bs + (long long)row * p.q_rs + (long long)h * 64;
#pragma unroll
      for (int c0 = 0; c0 < FA_D; c0 += 32) {
        uint32_t orr[32];
        tmem_ld32_nowait(t_o + (uint32_t)c0, orr);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) asm volatile("" : "+r"(orr[j]));
        if (row < p.rows) {
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            uint4 u;
            u.x = pack_bf16x2(__uint_as_float(orr[8 * t + 0]), __uint_as_float(orr[8 * t + 1]));
            u.y = pack_bf16x2(__uint_as_float(orr[8 * t + 2]), __uint_as_float(orr[8 * t + 3]));
            u.z = pack_bf16x2(__uint_as_float(orr[8 * t + 4]), __uint_as_float(orr[8 * t + 5]));
            u.w = pack_bf16x2(__uint_as_float(orr[8 * t + 6]), __uint_as_float(orr[8 * t + 7]));
            *reinterpret_cast<uint4*>(orow + c0 + 8 * t) = u;
          }
        }
      }
      tc_fence_before();   // the O reads are complete before the next P of this slot lets the issuer overwrite O
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512u);
  }
}

// 4-D map over [B][rows x heads][64]: dim0 = 64 head channels, dims 1/2 = (rows, heads) ordered by ascending stride
// (heads_first: the 8 heads of a row are adjacent, as in the cross-attention q / k / v layout), dim3 = batch.
int encode_rows_map(CUtensorMap* map, const void* base, int rows, int n_heads, int B, long long rs, long long hs, long long bs, int box_rows,
                    bool heads_first, const char* what) {
  EncodeTiledFn enc = get_encode_fn();
  B200_REQUIRE(enc != nullptr, "attention: cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[4], strides[3];
  cuuint32_t box[4] = {(cuuint32_t)FA_D, 1, 1, 1};
  dims[0] = FA_D;
  if (heads_first) {
    dims[1] = (cuuint64_t)n_heads; strides[0] = (cuuint64_t)hs * 2;
    dims[2] = (cuuint64_t)rows;    strides[1] = (cuuint64_t)rs * 2;
    box[2] = (cuuint32_t)box_rows;
  } else {
    dims[1] = (cuuint64_t)rows;    strides[0] = (cuuint64_t)rs * 2;
    dims[2] = (cuuint64_t)n_heads; strides[1] = n_heads > 1 ? (cuuint64_t)hs * 2 : (cuuint64_t)rows * rs * 2;   // extent-1 dims still need a legal stride
    box[1] = (cuuint32_t)box_rows;
  }
  dims[3] = (cuuint64_t)B;
  strides[2] = B > 1 ? (cuuint64_t)bs * 2 : strides[1] * dims[2];
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B200_REQUIRE(r == CUDA_SUCCESS, "attention: cuTensorMapEncodeTiled(%s) failed with %d (rows=%d heads=%d B=%d rs=%lld hs=%lld bs=%lld)", what, (int)r,
               rows, n_heads, B, rs, hs, bs);
  return B200_OK;
}

}  // namespace

// called by b200_attention (attention.cu) for <= 64 keys with a usable logit bound and heads-adjacent layouts
int b200_cross_attention_tc(const void* q, void* o, int64_t q_bs, int64_t q_hs, int32_t q_rs, int32_t rows, const void* k, const void* v,
                            int64_t kv_bs, int64_t kv_hs, int32_t kv_rs, int32_t n_keys, int B, int n_heads, cudaStream_t st) {
  CUtensorMap mq, mk, mv;
  int rc;
  if ((rc = encode_rows_map(&mq, q, rows, n_heads, B, q_rs, q_hs, q_bs, FA_BM, true, "Q")) != B200_OK) return rc;
  if ((rc = encode_rows_map(&mk, k, n_keys, n_heads, B, kv_rs, kv_hs, kv_bs, XA_KEYS, true, "K")) != B200_OK) return rc;
  if ((rc = encode_rows_map(&mv, v, n_keys, n_heads, B, kv_rs, kv_hs, kv_bs, XA_KEYS, true, "V")) != B200_OK) return rc;
  XaParams p;
  p.o = reinterpret_cast<__nv_bfloat16*>(o);
  p.q_bs = q_bs; p.q_rs = q_rs; p.q_hs = (int)q_hs; p.rows = rows; p.n_keys = n_keys; p.B = B; p.heads = n_heads;
  p.tiles_per_sample = (rows + FA_BM - 1) / FA_BM;
  const long long total = (long long)B * p.tiles_per_sample * n_heads;
  const int sms = sm_count();
  long long per = (total + sms - 1) / sms;
  per = (per + n_heads - 1) / n_heads * n_heads;                 // whole query tiles per CTA: the K/V reload boundaries fall between tiles
  p.items_per_cta = (int)per;
  {
    static const uint32_t wns = [] { const char* ev = getenv("B200_IMAGEN_FA_WAIT_NS"); return (uint32_t)(ev ? atoi(ev) : FA_DEFAULT_WAIT_NS); }();
    p.wait_ns = wns;
  }
  const int grid = (int)((total + per - 1) / per);
  B200_SMEM_OPT_IN(cross_attn_tc_kernel, XA_SMEM);
  B200_CUDA_OK(b200_launch(cross_attn_tc_kernel, dim3(grid), dim3(64 + 128 * XA_NS), XA_SMEM, st, mq, mk, mv, p));
  return B200_OK;
}

extern "C" int b200_linear_xattn_context(const void* k, const void* v, int64_t kv_bs, int32_t kv_rs, int32_t n_keys, int B, int n_heads,
                                         int32_t dim_head, void* ctx, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  B200_REQUIRE(k && v && ctx, "linear cross-attention context: null pointer");
  B200_REQUIRE(n_keys > 0 && B > 0 && B <= 65535 && n_heads > 0 && n_heads <= LX_MAX_HEADS && dim_head > 0 && dim_head <= 64,
               "linear cross-attention context: bad shape keys=%d B=%d heads=%d dim_head=%d", n_keys, B, n_heads, dim_head);
  B200_REQUIRE(kv_rs >= n_heads * 64 && kv_bs >= (int64_t)n_keys * kv_rs, "linear cross-attention context: strides too small (rs=%d bs=%lld)",
               kv_rs, (long long)kv_bs);
  B200_SMEM_OPT_IN(linear_xattn_context_kernel, LX_CTX_SMEM);
  B200_CUDA_OK(b200_launch(linear_xattn_context_kernel, dim3(n_heads, B), dim3(LX_CTX_THREADS), LX_CTX_SMEM, st,
                           reinterpret_cast<const __nv_bfloat16*>(k), reinterpret_cast<const __nv_bfloat16*>(v), (long long)kv_bs, (int)kv_rs,
                           (int)n_keys, (int)dim_head, reinterpret_cast<__nv_bfloat16*>(ctx)));
  return B200_OK;
}

extern "C" int b200_linear_cross_attention(const void* q, void* o, int64_t q_bs, int32_t q_rs, int32_t rows, const void* ctx, int B, int n_heads,
                                           int32_t dim_head, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  B200_REQUIRE(q && o && ctx, "linear cross-attention: null pointer");
  B200_REQUIRE(rows > 0 && B > 0 && n_heads > 0 && n_heads <= LX_MAX_HEADS && dim_head > 0 && dim_head <= 64,
               "linear cross-attention: bad shape rows=%d B=%d heads=%d dim_head=%d", rows, B, n_heads, dim_head);
  B200_REQUIRE((q_rs & 7) == 0 && (q_bs & 7) == 0 && q_rs >= n_heads * 64 && q_bs >= (int64_t)rows * q_rs,
               "linear cross-attention: strides must be multiples of 8 elements and cover heads x 64 channels (rs=%d bs=%lld)", q_rs, (long long)q_bs);
  CUtensorMap mq, mc;
  int rc;
  if ((rc = encode_rows_map(&mq, q, rows, n_heads, B, q_rs, 64, q_bs, FA_BM, true, "Q")) != B200_OK) return rc;
  if ((rc = encode_rows_map(&mc, ctx, 64, n_heads, B, 64, 64 * 64, (long long)n_heads * 64 * 64, 64, false, "C")) != B200_OK) return rc;
  LxParams p;
  p.o = reinterpret_cast<__nv_bfloat16*>(o);
  p.q_bs = q_bs; p.q_rs = q_rs; p.rows = rows; p.B = B; p.heads = n_heads; p.dim_head = dim_head;
  p.tiles_per_sample = (rows + FA_BM - 1) / FA_BM;
  const long long total = (long long)B * p.tiles_per_sample * n_heads;
  const int sms = sm_count();
  long long per = (total + sms - 1) / sms;
  per = (per + n_heads - 1) / n_heads * n_heads;                 // whole query tiles per CTA: the C reload boundaries fall between tiles
  p.items_per_cta = (int)per;
  {
    static const uint32_t wns = [] { const char* ev = getenv("B200_IMAGEN_FA_WAIT_NS"); return (uint32_t)(ev ? atoi(ev) : FA_DEFAULT_WAIT_NS); }();
    p.wait_ns = wns;
  }
  const int grid = (int)((total + per - 1) / per);
  B200_SMEM_OPT_IN(linear_cross_attn_tc_kernel, LX_SMEM);
  B200_CUDA_OK(b200_launch(linear_cross_attn_tc_kernel, dim3(grid), dim3(64 + 128 * LX_NS), LX_SMEM, st, mq, mc, p));
  return B200_OK;
}

// called by b200_attention (attention.cu) when the caller supplies a usable logit bound
int b200_attention_tc(const void* q, void* o, int64_t q_bs, int64_t q_hs, int32_t q_rs, int32_t rows, const void* k, const void* v,
                      int64_t kv_bs, int64_t kv_hs, int32_t kv_rs, int32_t n_keys, int B, int n_heads, float max_logit, cudaStream_t st) {
  CUtensorMap mq, mk, mv;
  int rc;
  const bool q_hf = n_heads > 1 && q_hs < q_rs, kv_hf = n_heads > 1 && kv_hs < kv_rs;
  if ((rc = encode_rows_map(&mq, q, rows, n_heads, B, q_rs, q_hs, q_bs, FA_BM, q_hf, "Q")) != B200_OK) return rc;
  if ((rc = encode_rows_map(&mk, k, n_keys, n_heads, B, kv_rs, kv_hs, kv_bs, FA_BN, kv_hf, "K")) != B200_OK) return rc;
  if ((rc = encode_rows_map(&mv, v, n_keys, n_heads, B, kv_rs, kv_hs, kv_bs, FA_BN, kv_hf, "V")) != B200_OK) return rc;
  FaParams p;
  p.o = reinterpret_cast<__nv_bfloat16*>(o);
  p.q_bs = q_bs; p.q_hs = q_hs; p.q_rs = q_rs; p.rows = rows; p.n_keys = n_keys; p.max_logit = max_logit;
  p.q_heads_first = q_hf ? 1 : 0; p.kv_heads_first = kv_hf ? 1 : 0;
  {
    static const uint32_t wns = [] { const char* ev = getenv("B200_IMAGEN_FA_WAIT_NS"); return (uint32_t)(ev ? atoi(ev) : FA_DEFAULT_WAIT_NS); }();
    p.wait_ns = wns;
  }
  p.trace = nullptr;
  p.trace_cta = 0;
  static const char* trace_path = getenv("B200_IMAGEN_FA_TRACE");   // development: dump one CTA's barrier time line of the next launch(es)
  static long long* trace_dev = nullptr;
  constexpr size_t TRACE_WORDS = 20 * 64 * 8;
  if (trace_path) {
    if (!trace_dev) B200_CUDA_OK(cudaMalloc(&trace_dev, TRACE_WORDS * sizeof(long long)));
    B200_CUDA_OK(cudaMemsetAsync(trace_dev, 0, TRACE_WORDS * sizeof(long long), st));
    p.trace = trace_dev;
    const char* c = getenv("B200_IMAGEN_FA_TRACE_CTA");
    p.trace_cta = c ? atoi(c) : 1000;
  }
  // Kernel variant: the defaults were chosen from B200 measurements (profiles/r02_attention_*); B200_IMAGEN_FA_VARIANT selects one of
  // the kept alternatives for tools/sweep_attention.py, B200_IMAGEN_FA_PERSISTENT=0 keeps the one-shot kernel for short key sequences.
  static const int variant = [] { const char* e = getenv("B200_IMAGEN_FA_VARIANT"); return e ? atoi(e) : -1; }();
  static const bool persistent_on = [] { const char* e = getenv("B200_IMAGEN_FA_PERSISTENT"); return !e || atoi(e) != 0; }();
  const int ntiles = (n_keys + FA_BN - 1) / FA_BN;
  const dim3 grid2((rows + 2 * FA_BM - 1) / (2 * FA_BM), n_heads, B);
#define PP_LAUNCH(POLY, SUB)                                                                                                     \
  {                                                                                                                                \
    B200_SMEM_OPT_IN((flash_attn_pp_kernel<POLY, SUB>), PP_SMEM);                                                                  \
    B200_CUDA_OK(b200_launch(flash_attn_pp_kernel<POLY, SUB>, grid2, dim3(128 + 256 * SUB), PP_SMEM, st, mq, mk, mv, p));           \
  }
#define PT_LAUNCH(POLY, SUB, ORDER, MODE)                                                                                        \
  {                                                                                                                                \
    B200_SMEM_OPT_IN((flash_attn_pt_kernel<POLY, SUB, ORDER, MODE>), PT_SMEM);                                                     \
    B200_CUDA_OK(b200_launch(flash_attn_pt_kernel<POLY, SUB, ORDER, MODE>, grid2, dim3(128 + 256 * SUB), PT_SMEM, st, mq, mk, mv, p)); \
  }
#define PTP_LAUNCH(POLY, MODE)                                                                                                   \
  {                                                                                                                                \
    B200_SMEM_OPT_IN((flash_attn_ptp_kernel<POLY, MODE>), PT_SMEM);                                                                \
    FaPersist pp;                                                                                                                  \
    pp.pairs_per_head = (rows + 2 * FA_BM - 1) / (2 * FA_BM);                                                                      \
    pp.n_heads = n_heads;                                                                                                          \
    pp.total_items = (long long)B * n_heads * pp.pairs_per_head;                                                                   \
    const long long ctas = pp.total_items < (long long)sm_count() ? pp.total_items : (long long)sm_count();                         \
    B200_CUDA_OK(b200_launch(flash_attn_ptp_kernel<POLY, MODE>, dim3((unsigned)ctas), dim3(640), PT_SMEM, st, mq, mk, mv, p, pp));  \
  }
  // MODE bits of flash_attn_pt_kernel: 1 no "- C", 2/4 ablations, 8 warp-elected arrivals, 16 score preload, 32 chunked P hand-over,
  // 64 late P-buffer wait, 512 time-line trace, 1024 S MMAs on a third issuer thread
  switch (variant) {
    case -1:                                     // product path
      if (persistent_on && ntiles <= FA_PERSISTENT_MAX_TILES) PTP_LAUNCH(4, 8)
      else PT_LAUNCH(4, 2, false, 17 + 1024 + 64)
      break;
    // the measured trail (times of the 64x64-level launch; profiles/r02_attention_*): each variant adds one change to the previous one
    case 12: PP_LAUNCH(0, 2); break;             // round-1 default: P through shared memory, 16 softmax warps (1.66 ms)
    case 20: PT_LAUNCH(0, 2, false, 0); break;   // P in tensor memory (1.53 ms)
    case 41: PT_LAUNCH(8, 2, false, 1); break;   // P = exp2(S), 1/8 polynomial exp2, suspend-hinted waits (1.42 ms)
    case 60: PT_LAUNCH(8, 2, false, 41); break;  // P handed over in 32-key chunks, warp-elected arrivals (1.37 ms)
    case 59: PT_LAUNCH(8, 2, false, 17); break;  // scores preloaded, S released before the first exponential (1.23 ms)
    case 65: PT_LAUNCH(6, 2, false, 17); break;  // 1/6 polynomial (1.20 ms; 1.17 ms once issued under elect.sync)
    case 82: PT_LAUNCH(6, 2, true, 17); break;   // MUFU token between the two query-tile groups (1.41 ms: slower)
    case 112: PT_LAUNCH(4, 2, false, 17 + 1024); break;        // S MMAs of both groups on a third issuer thread, 1/4 polynomial (1.12 ms)
    case 118: PT_LAUNCH(4, 2, false, 17 + 1024 + 64); break;   // + late P-buffer wait = the one-shot product path (1.12 ms)
    case 69: PT_LAUNCH(0, 2, false, 19); break;                // bottleneck experiment: preload, no MUFU (1.10 -> 0.88 ms with elect.sync; wrong results)
    case 114: PT_LAUNCH(0, 2, false, 19 + 1024); break;        // bottleneck experiment: third issuer thread, no MUFU (0.80 ms)
    case 81: PT_LAUNCH(6, 2, false, 17 + 512); break;          // variant 65 + time-line trace (tools/attn_trace.py)
    case 115: PT_LAUNCH(4, 2, false, 17 + 1024 + 512); break;  // variant 112 + time-line trace
#define PD_LAUNCH(POLY, MODE)                                                                                                    \
  {                                                                                                                                \
    B200_SMEM_OPT_IN((flash_attn_pd_kernel<POLY, MODE>), PD_SMEM);                                                                 \
    B200_CUDA_OK(b200_launch(flash_attn_pd_kernel<POLY, MODE>, grid2, dim3(640), PD_SMEM, st, mq, mk, mv, p));                      \
  }
    case 100: PD_LAUNCH(6, 0); break;            // dual softmax: every thread serves both query tiles (1.30 ms)
    case 104: PD_LAUNCH(0, 2); break;            // bottleneck experiment: dual, no MUFU
#undef PD_LAUNCH
    case 90: PTP_LAUNCH(6, 0); break;            // persistent CTAs at any length (1.16 ms)
    case 121: PTP_LAUNCH(4, 8); break;           // persistent + third issuer thread = the product path for short key sequences (1.19 ms)
    case 123: PTP_LAUNCH(0, 10); break;          // bottleneck experiment: persistent, third issuer thread, no MUFU (0.80 ms)
    default: B200_REQUIRE(false, "attention: unknown B200_IMAGEN_FA_VARIANT=%d", variant);
  }
#undef PTP_LAUNCH
#undef PT_LAUNCH
#undef PP_LAUNCH
  B200_LAUNCH_OK();
  if (trace_path && p.trace) {
    static long long host[TRACE_WORDS];
    B200_CUDA_OK(cudaStreamSynchronize(st));
    B200_CUDA_OK(cudaMemcpy(host, trace_dev, sizeof(host), cudaMemcpyDeviceToHost));
    if (FILE* f = fopen(trace_path, "wb")) {
      fwrite(host, sizeof(long long), TRACE_WORDS, f);
      fclose(f);
    }
  }
  return B200_OK;
}
