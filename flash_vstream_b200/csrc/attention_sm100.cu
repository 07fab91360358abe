// attention_sm100.cu — fvs_attention / fvs_attention80: per-frame multi-head self-attention on tcgen05, head_dim 64, or
// head_dim 80 = 64 "main" + 16 "extra" dims (kX variant, the Qwen2-VL vision tower): the extra dims travel as 16-column
// SWIZZLE_32B tiles next to the 64-column SWIZZLE_128B ones, cost one more K=16 MMA per S tile and one N=16 MMA per P V
// step, and live in their own column block of the activation ([main | extra] layout, see include/fvs_b200.h).
//
// One CTA per (128-query tile, head, frame); 2 CTAs co-reside per SM (~86 KB smem, 256 TMEM columns each).
//   warp 0      : TMA producer — Q tile once, then 64-row K/V tiles through a 4-stage ring (SWIZZLE_128B boxes cut from
//                 the packed [frames, tokens, 3*H*64] QKV activation by 3-D tensor maps; rows past `tokens` are
//                 zero-filled by the TMA, so frames never bleed into each other)
//   warp 1      : MMA issuer (converged warp, one elect.sync lane issues) — S_j = Q K_j^T into one of TWO TMEM score
//                 buffers; O += P_j V_j (P from TMEM, V MN-major straight from its TMA tile) and L += P_j 1 (row sums
//                 against a constant tile of ones) accumulate in TMEM
//   warp 2      : TMEM allocator;  warp 3: builds the ones tile
//   warps 4..11 : softmax, two threads per query row (warps 4-7: columns [0,32) of each 64-wide KV tile, warps 8-11:
//                 [32,64)).  SINGLE-PASS online softmax with LAZY rescaling: scores are read from TMEM exactly once
//                 (TMEM->RF moves only 16 fp32/clk/SM — as scarce as the 16 ex2/clk/SM SFU rate — so a second read of S
//                 would double the kernel's bound); P = exp2((S - m) * scale*log2e) uses the running row maximum m, and
//                 the TMEM accumulators O|L are rescaled (tcgen05.ld/st read-modify-write) only when a tile raises the
//                 maximum by more than 2^8, which after the first tile is rare.  The result is exact: O and L always
//                 carry the same scale, and O/L is formed at the end.
// P never touches shared memory: the softmax threads write the rounded P tile with tcgen05.st over the first 32 columns of
// the S buffer they just drained, and the P V / row-sum MMAs take it as their TMEM A operand (tcgen05.mma [d], [a], b-desc).
// S_{j+2} overwrites those columns, so the MMA issue order is S_0, S_1, then [P_j V_j, S_{j+2}] for j = 0, 1, ... in the
// (in-order) tensor pipe.  That keeps the softmax chain free of shared-memory stores and proxy fences.  DESIGN.md §3.2 has
// the measurements that chose this design over P in shared memory, a persistent schedule and the other variants that were
// built, measured and removed.
// tokens = 577 for ViT-L/14-336: 10 KV tiles, the last one 16 wide (1 valid key).
// Replaces HF CLIPAttention reached from multimodal_encoder/clip_encoder.py:50 (SURVEY.md §2.2 K2).
#include "fvs_common.h"
#include "fvs_kernels.h"
#include "fvs_ptx.cuh"

namespace fvs {
namespace attn {

constexpr int HD = 64;          // head dim
constexpr int BQ = 128;         // query rows per CTA
constexpr int BKV = 64;         // kv rows per tile
constexpr int kKVStages = 4;
constexpr int kThreads = 384;
constexpr int kSoftmaxThreads = 256;
constexpr int Q_BYTES = BQ * HD * 2;      // 16 KB
constexpr int KV_BYTES = BKV * HD * 2;    // 8 KB: [64 rows][64 x 16-bit], 128 B per row
constexpr int STG_BYTES = BQ * HD * 2;    // 16 KB: [128 rows][64 x 16-bit] O tile staged for the TMA store
constexpr int ONES_BYTES = 2048;          // [16 rows][64 x 16-bit] of 1.0 (B operand of the row-sum MMA)
constexpr int XCHG_BYTES = 2 * 2 * 128 * 4;  // [tile parity][column group][row] partial maxima
constexpr uint32_t TMEM_COLS = 256;  // S0: [0,64)  S1: [64,128)  O: [128,192) (+[192,208) extra dims)  L (row sums): 16 columns after O
constexpr uint32_t TMEM_O_OFF = 128;
constexpr int XD = 16;                    // extra head dims of the head_dim-80 variant
constexpr int QX_BYTES = BQ * XD * 2;     // 4 KB: [128 rows][16 x 16-bit], 32 B per row (SWIZZLE_32B)
constexpr int KVX_BYTES = BKV * XD * 2;   // 2 KB
template <bool kX> struct Lay {
  static constexpr int Q_TOTAL = Q_BYTES + (kX ? QX_BYTES : 0);
  static constexpr int KV_STAGE = KV_BYTES + (kX ? KVX_BYTES : 0);     // 8 KB | 10 KB, both multiples of 1024
  // The staging region is 2 * STG_BYTES although the O tile uses only its first half: the layout is kept byte-identical
  // to the build that DESIGN.md §3.2 measured.
  static constexpr int TILES = Q_TOTAL + kKVStages * KV_STAGE + 2 * STG_BYTES + ONES_BYTES + XCHG_BYTES;
  static constexpr int BYTES = TILES + 256 + 1024;
  static constexpr uint32_t L_OFF = kX ? 208 : 192;
};
constexpr float kRescaleThreshold = 8.0f;  // log2 units: rescale O|L only if the row maximum grew by more than 2^8

template <bool kBF16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if (kBF16) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}

template <bool kBF16, bool kX>
__global__ void __launch_bounds__(kThreads, 2)
attention_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_kv,
                 const __grid_constant__ CUtensorMap tmap_ctx, const __grid_constant__ CUtensorMap tmap_qx,
                 const __grid_constant__ CUtensorMap tmap_kvx, const __grid_constant__ CUtensorMap tmap_ctxx, int tokens,
                 int heads, float scale_log2e) {
  using L_ = Lay<kX>;
  constexpr uint32_t TMEM_L_OFF = L_::L_OFF;
  // SWIZZLE_128B tiles need 1024-byte alignment.  The alignment is declared (not rounded up by hand through an integer
  // cast): the pointer keeps its shared address space, so the compiler emits 32-bit STS/LDS instead of generic ST/LD.
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint8_t* smem_q = smem;
  uint8_t* smem_qx = smem_q + Q_BYTES;                    // kX: [128][32 B] extra dims of Q (later: staging of the extra ctx dims)
  uint8_t* smem_kv = smem_q + L_::Q_TOTAL;                // [kKVStages][8 KB main (+ 2 KB extra)]
  uint8_t* smem_stg = smem_kv + kKVStages * L_::KV_STAGE; // 16 KB O staging tile (+ 16 KB unused, see Lay)
  uint8_t* smem_ones = smem_stg + 2 * STG_BYTES;          // 2 KB of 1.0
  float* smem_x = reinterpret_cast<float*>(smem_ones + ONES_BYTES);  // [2][2][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L_::TILES);
  uint64_t* q_full = bars;                 // 1
  uint64_t* kv_full = bars + 1;            // [4]
  uint64_t* kv_empty = bars + 5;           // [4]
  uint64_t* s_full = bars + 9;             // [2] MMA -> softmax: S tile ready in TMEM buffer b
  uint64_t* s_empty = bars + 11;           // [2] softmax -> MMA: S buffer b drained to registers (256 arrivals)
  uint64_t* p_full = bars + 13;            // [2] softmax -> MMA: P written over S buffer b (256 arrivals)
  uint64_t* pv_done = bars + 15;           // [2] MMA -> softmax: P_j V_j (and everything before it) retired
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 17);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * BQ;
  const int head = blockIdx.y;
  const int frame = blockIdx.z;
  const int nkv = (tokens + BKV - 1) / BKV;
  const int last_cols = ((tokens - (nkv - 1) * BKV) + 15) & ~15;  // width of the last KV tile, multiple of 16
  const int q_col = head * HD;
  const int k_col = heads * HD + head * HD;
  const int v_col = 2 * heads * HD + head * HD;
  // extra-dim column blocks follow the three main blocks: [q main | k main | v main | q extra | k extra | v extra]
  const int xq_col = 3 * heads * HD + head * XD;
  const int xk_col = xq_col + heads * XD;
  const int xv_col = xk_col + heads * XD;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_kv);
    tma_prefetch_desc(&tmap_ctx);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < kKVStages; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&s_full[b], 1);
      mbar_init(&s_empty[b], kSoftmaxThreads);
      mbar_init(&p_full[b], kSoftmaxThreads);
      mbar_init(&pv_done[b], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<TMEM_COLS>(tmem_ptr_smem);
    tmem_relinquish();
  }
  if (warp == 3) {  // constant tile of ones (layout-independent: every element is 1.0)
    const uint32_t one2 = kBF16 ? 0x3F803F80u : 0x3C003C00u;
    for (int i = lane; i < ONES_BYTES / 16; i += 32)
      reinterpret_cast<uint4*>(smem_ones)[i] = make_uint4(one2, one2, one2, one2);
    fence_proxy_async_smem();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // register re-balancing between warpgroups: the 4 service warps need almost nothing, the 8 softmax warps hold a
  // 32-column score slice per thread (launch: 384 x 80 registers; after: 128 x 64 + 256 x 88 = 30720 = the CTA's launch allocation — setmaxnreg.inc can only take what .dec released inside the same CTA)
  if (warp < 4) reg_dealloc<64>(); else reg_alloc<88>();

  pdl_trigger();  // PDL: the setup above overlapped the QKV GEMM's tail; its output is read from here on
  pdl_wait();

  if (warp == 0 && lane == 0) {
    // ------------------------------------------------------------------ TMA producer
    mbar_arrive_expect_tx(q_full, L_::Q_TOTAL);
    tma_load_3d(smem_q, &tmap_q, q_full, q_col, q0, frame);
    if (kX) tma_load_3d(smem_qx, &tmap_qx, q_full, xq_col, q0, frame);
    int stage = 0;
    uint32_t phase = 0;
    auto load_tile = [&](int col, int xcol, int row) {
      mbar_wait(&kv_empty[stage], phase ^ 1);
      mbar_arrive_expect_tx(&kv_full[stage], L_::KV_STAGE);
      tma_load_3d(smem_kv + stage * L_::KV_STAGE, &tmap_kv, &kv_full[stage], col, row, frame);
      if (kX) tma_load_3d(smem_kv + stage * L_::KV_STAGE + KV_BYTES, &tmap_kvx, &kv_full[stage], xcol, row, frame);
      if (++stage == kKVStages) { stage = 0; phase ^= 1; }
    };
    // consumption order of the MMA thread: K0, K1, then (V_j, K_{j+2}) for j = 0, 1, ...
    load_tile(k_col, xk_col, 0);
    if (nkv > 1) load_tile(k_col, xk_col, BKV);
    for (int j = 0; j < nkv; ++j) {
      load_tile(v_col, xv_col, j * BKV);
      if (j + 2 < nkv) load_tile(k_col, xk_col, (j + 2) * BKV);
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    // The WHOLE warp runs this control flow and one lane issues: with a single-lane role every descriptor is a per-thread
    // value that has to be moved into the uniform registers tcgen05.mma reads (R2UR + ELECT per operand, ~15 dependent
    // instructions per MMA).  At N = 64 an MMA is only 32-48 clk of tensor work, so that serial issue stream — not the
    // tensor pipe, the SFU or TMEM — was what paced the kernel (ncu: softmax warps 30 % of their time waiting for S;
    // removing MUFU.EX2 altogether gained 2 %, removing MMAs 1.6 % each).  Warp-uniform descriptor arithmetic stays in
    // the uniform datapath; descriptors are kept as (lo, hi) words so a k step is one 32-bit add.
    constexpr uint32_t idesc_pv = umma_idesc_f16(BQ, HD, kBF16, false, /*B = V is MN-major*/ true);
    constexpr uint32_t idesc_l = umma_idesc_f16(BQ, 16, kBF16, false, false);
    constexpr uint32_t idesc_pvx = umma_idesc_f16(BQ, XD, kBF16, false, /*B = V extra is MN-major*/ true);
    constexpr uint32_t idesc_s_full = umma_idesc_f16(BQ, BKV, kBF16, false, false);
    const uint32_t idesc_s_last = umma_idesc_f16(BQ, last_cols, kBF16, false, false);
    // descriptor words (see umma_desc_sw128 / umma_desc_sw32): hi = SBO | version | layout, lo = address >> 4 | LBO << 16
    constexpr uint32_t HI_K = uint32_t(umma_desc_sw128(0, 1024, 16) >> 32);      // K-major SWIZZLE_128B (Q, K, ones)
    constexpr uint32_t HI_V = uint32_t(umma_desc_sw128(0, 1024, 1024) >> 32);    // MN-major SWIZZLE_128B (V)
    constexpr uint32_t HI_X = uint32_t(umma_desc_sw32(0, 256, 256) >> 32);       // SWIZZLE_32B (extra dims)
    constexpr uint32_t LBO_K = uint32_t(umma_desc_sw128(0, 1024, 16));
    constexpr uint32_t LBO_V = uint32_t(umma_desc_sw128(0, 1024, 1024));
    constexpr uint32_t LBO_X = uint32_t(umma_desc_sw32(0, 256, 256));
    auto desc = [](uint32_t lo, uint32_t hi) { return (uint64_t(hi) << 32) | lo; };
    const uint32_t q_lo = (smem_u32(smem_q) >> 4) | LBO_K;
    const uint32_t qx_lo = (smem_u32(smem_qx) >> 4) | LBO_X;
    const uint32_t ones_lo = (smem_u32(smem_ones) >> 4) | LBO_K;
    const uint32_t kv_lo0 = smem_u32(smem_kv) >> 4;           // + stage * (KV_STAGE >> 4)
    const uint32_t o_tmem = tmem_base + TMEM_O_OFF;
    const uint32_t l_tmem = tmem_base + TMEM_L_OFF;
    int stage = 0;
    uint32_t phase = 0;

    auto issue_s = [&](int j) {  // S_j -> TMEM buffer (j & 1)
      const int b = j & 1;
      mbar_wait(&kv_full[stage], phase);
      if (j >= 2) mbar_wait(&s_empty[b], ((j - 2) >> 1) & 1);  // softmax has drained S_{j-2} from this buffer
      tc_fence_after_sync();
      const uint32_t idesc_s = (j == nkv - 1) ? idesc_s_last : idesc_s_full;
      const uint32_t k_lo = kv_lo0 + stage * (L_::KV_STAGE >> 4);
      const uint32_t s_tmem = tmem_base + b * BKV;
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
          umma_f16_ss(s_tmem, desc(q_lo + 2 * k, HI_K), desc((k_lo | LBO_K) + 2 * k, HI_K), idesc_s, k != 0 ? 1u : 0u);
        if (kX)   // dims 64..79: one more K = 16 step from the SWIZZLE_32B tiles
          umma_f16_ss(s_tmem, desc(qx_lo, HI_X), desc((k_lo + (KV_BYTES >> 4)) | LBO_X, HI_X), idesc_s, 1u);
        umma_commit(&kv_empty[stage]);
        umma_commit(&s_full[b]);
      }
      __syncwarp();
      if (++stage == kKVStages) { stage = 0; phase ^= 1; }
    };
    auto issue_pv_step = [&](uint32_t p_tmem, uint32_t v_lo, int k, uint32_t acc) {
      // A = P[:, 16k..16k+16) from TMEM: 8 columns of packed pairs at the head of S buffer b; B = V[16k..16k+16, 0..64):
      // MN-major, 16 kv rows = two 8-row groups (SBO = 1024 B apart), 2048 B per k step
      const uint32_t a_tmem = p_tmem + 8 * k;
      umma_f16_ts(o_tmem, a_tmem, desc((v_lo | LBO_V) + 128 * k, HI_V), idesc_pv, acc);
      if (kX)   // O[:, 64..80) += P V_extra: B = V_extra[16k..16k+16, 0..16) MN-major, two 8-row groups 256 B apart
        umma_f16_ts(o_tmem + HD, a_tmem, desc(((v_lo + (KV_BYTES >> 4)) | LBO_X) + 32 * k, HI_X), idesc_pvx, acc);
      umma_f16_ts(l_tmem, a_tmem, desc(ones_lo, HI_K), idesc_l, acc);  // row sums of the rounded P
    };

    // Issue order: S_0, S_1, then [P_j V_j, S_{j+2}]: S_{j+2} overwrites the TMEM columns P_j lives in, so it has to
    // follow P_j V_j in the (in-order) tensor pipe.
    mbar_wait(q_full, 0);
    issue_s(0);
    if (nkv > 1) issue_s(1);
    for (int j = 0; j < nkv; ++j) {
      const int b = j & 1;
      mbar_wait(&kv_full[stage], phase);          // V_j landed
      mbar_wait(&p_full[b], (j >> 1) & 1);        // P_j written (and any O|L rescale finished)
      tc_fence_after_sync();
      const uint32_t v_lo = kv_lo0 + stage * (L_::KV_STAGE >> 4);
      const uint32_t p_tmem = tmem_base + b * BKV;  // TMEM address of P_j (aliases the drained S buffer)
      if (elect_one()) {
        if (j < nkv - 1 || last_cols == BKV) {
          issue_pv_step(p_tmem, v_lo, 0, j != 0 ? 1u : 0u);
#pragma unroll
          for (int k = 1; k < BKV / 16; ++k) issue_pv_step(p_tmem, v_lo, k, 1u);
        } else {
          for (int k = 0; k < last_cols / 16; ++k) issue_pv_step(p_tmem, v_lo, k, (j | k) != 0 ? 1u : 0u);
        }
        umma_commit(&kv_empty[stage]);
        umma_commit(&pv_done[b]);
      }
      __syncwarp();
      if (++stage == kKVStages) { stage = 0; phase ^= 1; }
      if (j + 2 < nkv) issue_s(j + 2);            // behind P_j V_j: S_{j+2} overwrites the TMEM columns P_j lives in
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ softmax: 2 threads per query row
    const int quad = warp & 3;
    const int grp = (warp - 4) >> 2;          // 0: columns [0,32) of each KV tile / O dims [0,32) ; 1: [32,64)
    const int r = quad * 32 + lane;           // query row inside the tile == TMEM lane
    const int rsw = r & 7;                    // swizzle phase of this row
    const uint32_t lane_addr = uint32_t(quad * 32) << 16;
    float m_run = -INFINITY;                  // running row maximum of the raw scores (identical in both threads of a row)
    float* const xs_mine = smem_x + grp * 128 + r;
    float* const xs_peer = smem_x + (grp ^ 1) * 128 + r;
    const uint32_t s_addr0 = tmem_base + lane_addr + grp * 32;

    for (int j = 0; j < nkv; ++j) {
      const int b = j & 1;
      // Columns of this tile that are real keys for this thread (<= 0: none).  The load below always fetches 32 columns:
      // on the (narrower) last tile the surplus columns hold stale scores that the masks discard, and the P columns they
      // produce lie beyond the K extent the P V MMA reads.  Keeping the code path uniform avoids register shuffles.
      const int myvalid = tokens - j * BKV - grp * 32;
      mbar_wait(&s_full[b], (j >> 1) & 1);
      tc_fence_after_sync();
      uint32_t v[32];
      tmem_ld_32x32b_x32(s_addr0 + b * BKV, v);
      tmem_ld_wait_dep(v);
      tc_fence_before_sync();
      mbar_arrive(&s_empty[b]);               // S buffer b may be overwritten by S_{j+2}

      // ---- tile maximum of this row (over both column groups).  On the (narrower) last tile the columns past the
      // sequence end hold stale scores: they are forced to -inf here and their P entries to zero below.
      const bool full = myvalid >= 32;
      if (!full) {
#pragma unroll
        for (int e = 0; e < 32; ++e)
          if (e >= myvalid) v[e] = 0xff800000u;   // -inf
      }
      float tmax = -INFINITY;
#pragma unroll
      for (int e = 0; e < 32; ++e) tmax = fmaxf(tmax, __uint_as_float(v[e]));
      xs_mine[b * 256] = tmax;                // exchange slot of this tile parity
      named_bar_sync(2 + quad, 64);           // the two warps that share these 32 rows
      tmax = fmaxf(tmax, xs_peer[b * 256]);

      // ---- lazy rescale of the TMEM accumulators
      const bool grow = (tmax - m_run) * scale_log2e > kRescaleThreshold;  // true at j == 0 (m_run = -inf)
      if (j == 0) {
        m_run = tmax;
      } else if (__any_sync(0xffffffffu, grow)) {
        const float m_new = grow ? tmax : m_run;
        const float factor = grow ? ex2_approx((m_run - m_new) * scale_log2e) : 1.0f;
        mbar_wait(&pv_done[(j - 1) & 1], ((j - 1) >> 1) & 1);   // every P V up to tile j-1 has retired
        tc_fence_after_sync();
        // O columns of this thread in two 16-column halves (keeps the register footprint of this rare path small);
        // column group 0 also rescales the row sums L, which carry the same scale
        const uint32_t o_addr = tmem_base + lane_addr + TMEM_O_OFF + grp * 32;
#pragma unroll 1
        for (int h = 0; h < 3; ++h) {
          if (h == 2 && grp != 0 && !kX) break;
          // third block: column group 0 rescales the row sums L, column group 1 (kX) the 16 extra O dims
          const uint32_t a = (h < 2) ? o_addr + h * 16
                                     : tmem_base + lane_addr + (grp == 0 ? TMEM_L_OFF : TMEM_O_OFF + HD);
          uint32_t o[16];
          tmem_ld_32x32b_x16(a, o);
          tmem_ld_wait_dep(o);
#pragma unroll
          for (int e = 0; e < 16; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * factor);
          tmem_st_32x32b_x16(a, o);
        }
        tmem_st_wait();
        m_run = m_new;
      }

      // ---- P_j = exp2((S - m_run) * scale*log2e) -> TMEM, packed pairs over the head of S buffer b (this thread's 32 columns
      // -> 16 TMEM columns at 16 * grp).  The partner thread of the row has loaded ITS scores before the pair barrier above,
      // so overwriting its columns is safe; S_{j+2} is only issued behind P_j V_j.  Masked columns carry -inf, so ex2 gives
      // exactly 0 (no separate masking pass); a thread with no valid column at all (second column group of a narrow last
      // tile) just writes zeros.
      {
        const float neg_max_scaled = -m_run * scale_log2e;
        uint32_t w[16];
#pragma unroll
        for (int e = 0; e < 32; e += 2)
          w[e >> 1] = myvalid <= 0 ? 0u
                                   : pack2<kBF16>(ex2_approx(fmaf(__uint_as_float(v[e]), scale_log2e, neg_max_scaled)),
                                                  ex2_approx(fmaf(__uint_as_float(v[e + 1]), scale_log2e, neg_max_scaled)));
        tmem_st_32x32b_x16(tmem_base + lane_addr + b * BKV + grp * 16, w);
        tmem_st_wait();
      }
      tc_fence_before_sync();                 // orders the tcgen05.st of P and of a rescale before the MMA thread's P V
      mbar_arrive(&p_full[b]);
    }

    // ---- epilogue: O / L -> 16-bit -> swizzled staging tile -> TMA store; each thread 32 of the 64 dims
    mbar_wait(&pv_done[(nkv - 1) & 1], ((nkv - 1) >> 1) & 1);
    tc_fence_after_sync();
    uint32_t o[32], lsum[16];
    tmem_ld_32x32b_x32(tmem_base + lane_addr + TMEM_O_OFF + grp * 32, o);
    tmem_ld_32x32b_x16(tmem_base + lane_addr + TMEM_L_OFF, lsum);
    tmem_ld_wait_dep(o);
    tmem_ld_wait_dep(lsum);
    const float inv = 1.0f / __uint_as_float(lsum[0]);
    uint8_t* stg = smem_stg + r * 128;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint4 w;
      w.x = pack2<kBF16>(__uint_as_float(o[i * 8 + 0]) * inv, __uint_as_float(o[i * 8 + 1]) * inv);
      w.y = pack2<kBF16>(__uint_as_float(o[i * 8 + 2]) * inv, __uint_as_float(o[i * 8 + 3]) * inv);
      w.z = pack2<kBF16>(__uint_as_float(o[i * 8 + 4]) * inv, __uint_as_float(o[i * 8 + 5]) * inv);
      w.w = pack2<kBF16>(__uint_as_float(o[i * 8 + 6]) * inv, __uint_as_float(o[i * 8 + 7]) * inv);
      *reinterpret_cast<uint4*>(stg + (((grp * 4 + i) ^ rsw) << 4)) = w;
    }
    if (kX && grp == 1) {   // the 16 extra dims: SWIZZLE_32B staging in the (now idle) Q-extra tile
      uint32_t ox[16];
      tmem_ld_32x32b_x16(tmem_base + lane_addr + TMEM_O_OFF + HD, ox);
      tmem_ld_wait_dep(ox);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint4 w;
        w.x = pack2<kBF16>(__uint_as_float(ox[c * 8 + 0]) * inv, __uint_as_float(ox[c * 8 + 1]) * inv);
        w.y = pack2<kBF16>(__uint_as_float(ox[c * 8 + 2]) * inv, __uint_as_float(ox[c * 8 + 3]) * inv);
        w.z = pack2<kBF16>(__uint_as_float(ox[c * 8 + 4]) * inv, __uint_as_float(ox[c * 8 + 5]) * inv);
        w.w = pack2<kBF16>(__uint_as_float(ox[c * 8 + 6]) * inv, __uint_as_float(ox[c * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(smem_qx + r * 32 + ((c ^ ((r >> 2) & 1)) << 4)) = w;
      }
    }
    fence_proxy_async_smem();
    named_bar_sync(1, kSoftmaxThreads);
    if (threadIdx.x == 128) {
      tma_store_3d(&tmap_ctx, smem_stg, head * HD, q0, frame);  // rows >= tokens are clipped by the map
      if (kX) tma_store_3d(&tmap_ctxx, smem_qx, heads * HD + head * XD, q0, frame);
      tma_store_commit();
      tma_store_wait_all<0>();
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after_sync();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

}  // namespace attn

template <bool kBF16, bool kX>
static int attention_launch_t(const AttnMaps& m, dim3 grid, int tokens, int heads, float scale_log2e, cudaStream_t stream) {
  using namespace attn;
  static bool done = false;
  if (!done) {
    FVS_CUDA_OK(cudaFuncSetAttribute(attention_kernel<kBF16, kX>, cudaFuncAttributeMaxDynamicSharedMemorySize, Lay<kX>::BYTES));
    done = true;
  }
  FVS_CUDA_OK(launch_ex(attention_kernel<kBF16, kX>, grid, dim3(kThreads), Lay<kX>::BYTES, stream, 1, /*pdl=*/true, m.q, m.kv,
                        m.ctx, m.qx, m.kvx, m.ctxx, tokens, heads, scale_log2e));
  return FVS_OK;
}

int attention_launch(const AttnMaps& m, int frames, int tokens, int heads, float scale, int dtype, cudaStream_t stream,
                     int head_dim) {
  using namespace attn;
  const float scale_log2e = scale * 1.4426950408889634f;
  dim3 grid((tokens + BQ - 1) / BQ, heads, frames);
  const bool bf = dtype == FVS_BF16, x80 = head_dim == 80;
  const int prof = prof_begin(FVS_PROF_ATTENTION, 4.0 * frames * double(heads) * tokens * double(tokens) * head_dim, stream);
  const int r = x80 ? (bf ? attention_launch_t<true, true>(m, grid, tokens, heads, scale_log2e, stream)
                          : attention_launch_t<false, true>(m, grid, tokens, heads, scale_log2e, stream))
                    : (bf ? attention_launch_t<true, false>(m, grid, tokens, heads, scale_log2e, stream)
                          : attention_launch_t<false, false>(m, grid, tokens, heads, scale_log2e, stream));
  if (r) return r;
  prof_end(prof, stream);
  FVS_CHECK_LAUNCH("attention_kernel");
  return FVS_OK;
}

// head_dim 64: qkv [frames*tokens, 3*H*64], ctx [.., H*64].  head_dim 80: qkv [.., 3*H*80] laid out as
// [q main H*64 | k main | v main | q extra H*16 | k extra | v extra], ctx [.., H*80] as [main H*64 | extra H*16].
int attention_make_maps(AttnMaps* m, const void* qkv, void* ctx, int frames, int tokens, int heads, int head_dim) {
  using namespace attn;
  const uint64_t wq = uint64_t(3) * heads * head_dim, wc = uint64_t(heads) * head_dim;
  int r;
  if ((r = make_tmap_3d(&m->q, qkv, frames, tokens, wq, wq, uint64_t(tokens) * wq, BQ, HD, 1))) return r;
  if ((r = make_tmap_3d(&m->kv, qkv, frames, tokens, wq, wq, uint64_t(tokens) * wq, BKV, HD, 1))) return r;
  if ((r = make_tmap_3d(&m->ctx, ctx, frames, tokens, wc, wc, uint64_t(tokens) * wc, BQ, HD, 1))) return r;
  if (head_dim == 80) {
    if ((r = make_tmap_3d(&m->qx, qkv, frames, tokens, wq, wq, uint64_t(tokens) * wq, BQ, XD, 2))) return r;
    if ((r = make_tmap_3d(&m->kvx, qkv, frames, tokens, wq, wq, uint64_t(tokens) * wq, BKV, XD, 2))) return r;
    if ((r = make_tmap_3d(&m->ctxx, ctx, frames, tokens, wc, wc, uint64_t(tokens) * wc, BQ, XD, 2))) return r;
  } else {
    m->qx = m->q; m->kvx = m->kv; m->ctxx = m->ctx;
  }
  return FVS_OK;
}

}  // namespace fvs

static int attention_entry(const void* qkv, void* ctx, int frames, int tokens, int heads, float scale, int dtype,
                           fvs_stream_t stream, int head_dim, const char* who) {
  using namespace fvs;
  FVS_REQUIRE(qkv && ctx, "%s: null pointer", who);
  FVS_REQUIRE(frames > 0 && tokens > 0 && heads > 0, "%s: bad shape", who);
  FVS_REQUIRE(frames <= 65535 && heads <= 65535, "%s: grid too large", who);
  FVS_REQUIRE(dtype == FVS_F16 || dtype == FVS_BF16, "%s: dtype must be f16 or bf16", who);
  FVS_REQUIRE(scale > 0.f, "%s: scale must be positive", who);
  AttnMaps m;
  int r = attention_make_maps(&m, qkv, ctx, frames, tokens, heads, head_dim);
  if (r) return r;
  return attention_launch(m, frames, tokens, heads, scale, dtype, static_cast<cudaStream_t>(stream), head_dim);
}

extern "C" int fvs_attention(const void* qkv, void* ctx, int frames, int tokens, int heads, float scale, int dtype,
                             fvs_stream_t stream) {
  return attention_entry(qkv, ctx, frames, tokens, heads, scale, dtype, stream, 64, "fvs_attention");
}

extern "C" int fvs_attention80(const void* qkv, void* ctx, int frames, int tokens, int heads, float scale, int dtype,
                               fvs_stream_t stream) {
  return attention_entry(qkv, ctx, frames, tokens, heads, scale, dtype, stream, 80, "fvs_attention80");
}
