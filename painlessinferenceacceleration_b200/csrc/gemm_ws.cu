// Weight-streaming GEMM for the verify forward (sm_100a: TMA + tcgen05 + TMEM).
//
//   Y[t, n] = sum_k X[t, k] * W[n, k]        X: [TOK <= 64 draft rows, K] bf16,  W: [N, K] bf16 (nn.Linear weight)
//
// i.e. the q/k/v/o/gate/up/down/lm_head projections of the reference's patched forward
// (models/llama/modeling_llama.py:254-256, :303, :185-186, :769) at the draft's row count.  With <= 64 rows the
// GEMM is a pure weight stream (arithmetic intensity = rows FLOP/B << ridge), so the kernel is built around HBM:
//   * swap-AB: 128 weight rows are the UMMA M dimension, the 64 tokens the UMMA N dimension; D[128 x 64] fp32 lives in
//     64 TMEM columns, so the big operand (W) is read exactly once and only the small one (X, <= 1.4 MB, L2 resident)
//     is re-read per tile;
//   * one CTA per (128-row weight tile, K split): warp 0 = TMA producer over a 4-stage mbarrier ring of
//     {W tile 128x64 (16 KB), X tile 64x64 (8 KB)} SWIZZLE_128B boxes, warp 1 = single-thread tcgen05.mma issuer
//     (4 x UMMA 128x64x16 per stage), warps 2-5 = epilogue (tcgen05.ld -> bf16 / fp32 store).  ~100 KB of shared
//     memory per CTA so that two CTAs share an SM and one CTA's prologue/epilogue hides behind the other's stream;
//   * projections with few weight tiles (o_proj, down_proj: N = 4096 -> 32 tiles) split K across CTAs and write fp32
//     partial slices that the consumer (k_rmsnorm_partials) sums in a fixed order - deterministic, no atomics.
#include <cuda.h>
#include <cuda_bf16.h>

#include <new>

#include "common.cuh"

namespace pia {
namespace gemm {

constexpr int BMW = 128;   // weight rows per tile (UMMA M)
constexpr int BK = 64;     // k elements per stage (one 128-byte swizzle row)
constexpr int TOK = 64;    // token rows (UMMA N)
constexpr int NTHREADS = 192;
constexpr int W_BYTES = BMW * BK * 2, X_BYTES = TOK * BK * 2, STAGE_BYTES = W_BYTES + X_BYTES;
constexpr int XCH_BYTES = TOK * 64 * 2;  // bf16 [64 tokens][64 rows] exchange tile of the SiLU*up epilogue
constexpr int smem_total(int nstage) { return nstage * STAGE_BYTES + 256 + XCH_BYTES + 1024; }
constexpr int TMEM_COLS = 64;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t addr, uint32_t *v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(addr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// K-major SWIZZLE_128B operand descriptor (cute::UMMA::SmemDescriptor): 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t kmajor_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;           // LBO (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32; // SBO
  d |= (uint64_t)1 << 46;           // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;           // SWIZZLE_128B
  return d;
}
// bf16 x bf16 -> fp32, M = 128, N = TOK, both operands K-major
constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TOK >> 3) << 17) | ((uint32_t)(BMW >> 4) << 24);

struct Params {
  int N, K, n_split, chunks_per_split, n_chunks, rows, tiled;
  int groups, w_group_rows, x_group_chunks;  // grouped GEMM (gridDim.z = groups): group g uses weight rows
                                             // [g*w_group_rows, +N) and activation columns [g*x_group_chunks*64, +K)
  long long out_group_stride;                // elements between the groups' [rows_cap, N] outputs
  int cluster;              // > 1: the K splits of a tile are one thread-block cluster and reduce through DSMEM (bf16 out)
  int silu;                 // 1: tile rows are 64 gate rows + 64 up rows of the same columns -> out = silu(g) * u
  int no_pdl;               // 1: plain kernel boundary - do not let the successor start early either
  __nv_bfloat16 *out_bf16;  // [rows_cap, N]  (or [rows_cap, N/2] with silu)   (n_split == 1)
  float *out_f32;           // [n_split, TOK, N] slices  (n_split > 1)
  // fp8-weight plans only
  const float *scale;             // [groups, N] per-output-channel dequantisation scales
  const __nv_bfloat16 *bias;      // [N] or nullptr
  int w_group_tiles;              // 128-row weight tiles per group (tiled fp8 blocks are [groups][tiles][chunks])
};

// ------------------------------------------------------------------------------------------------ fp8 weights
// FP8 = true: W is e4m3 with one fp32 scale per output channel, Y[t, n] = bf16(s[n] * sum_k X[t, k] Wq[n, k] (+ b[n])).
// A stage is one 128 x 128 e4m3 box (16 KB: half the bytes of the bf16 stage's 128 x 64) plus the two 64-k activation
// boxes of the same 128 k.  tcgen05.mma kind::f16 needs bf16 operands, so the four epilogue warps - idle until the
// accumulator is complete - dequantise each weight half-tile (thread = weight row) into a SWIZZLE_128B K-major bf16
// half-tile in shared memory (two slots, recycled by tcgen05.commit), fence the generic->async proxy and hand it to
// the MMA warp, which runs exactly the bf16 kernel's UMMA sequence on it.  The conversion is exact (every e4m3 value is
// a bf16 value), so with the scale applied in the epilogue the only roundings are the fp32 MMA accumulation and the
// final bf16 store.  Chosen over writing the bf16 tile to TMEM (tcgen05.st + TS-form MMA): the shared-memory form keeps
// the MMA descriptors, the accumulator and the split-K / cluster code of the bf16 path unchanged, and the swizzled
// layout makes the row-per-thread loads and stores bank-conflict free.
// Activations stay bf16 on purpose: at <= 256 token rows the GEMM is bound by HBM bytes, not by the MMA rate, so
// quantising X to e4m3 for kind::f8f6f4 would change the numerics (W8A8) for no gain in time.
// TOKN (the UMMA N = token rows per launch) is 64 (decode, decoding_length <= 64), 128 (decode up to 128 nodes) or
// 256 (prefill passes); shared memory per TOKN is sized so that TOKN = 64 keeps two CTAs per SM.
constexpr int F8_BK = 128;                 // k per fp8 stage (one 128-byte swizzle row of e4m3)
constexpr int F8_W = BMW * F8_BK;          // 16 KB e4m3 weight box
constexpr int F8_CONV = BMW * BK * 2;      // one bf16 half tile (128 rows x 64 k)
constexpr int f8_stage(int tokn) { return F8_W + 2 * tokn * BK * 2; }
constexpr int f8_smem_total(int nstage, int tokn) { return nstage * f8_stage(tokn) + 2 * F8_CONV + 256 + 1024; }
constexpr uint32_t idesc_tok(int tokn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(tokn >> 3) << 17) | ((uint32_t)(BMW >> 4) << 24);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// two e4m3 bytes at bits 15:8 and 31:24 of t -> bf16x2, exactly: sign and the 7 exponent/mantissa bits move into a
// bf16 with exponent bias 127 instead of 7, and the multiply by 2^120 rebiases (bf16 keeps e4m3's subnormals, the
// product is exact and -0 keeps the sign of zero)
__device__ __forceinline__ uint32_t e4m3x2_to_bf16x2(uint32_t t) {
  const uint32_t v = (t & 0x80008000u) | ((t >> 4) & 0x07F007F0u);
  uint32_t r;
  asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(v), "r"(0x7B807B80u), "r"(0x80008000u));
  return r;
}

// NSTAGE = 4: ~100 KB of shared memory, two CTAs per SM (grids with more CTAs than SMs);
// NSTAGE = 8: ~200 KB, one CTA per SM with twice the bytes in flight (grids that do not fill the SMs twice) -
// HBM only saturates with >= ~10 MB of loads in flight chip-wide.
// FP8: NSTAGE = 2 at TOKN = 64 (~97 KB, two CTAs per SM), otherwise one CTA per SM (see f8_smem_total).
template <int NSTAGE, int TOKN = TOK, bool FP8 = false>
__global__ void __launch_bounds__(NTHREADS, (FP8 ? (TOKN == 64 && NSTAGE <= 2) : NSTAGE <= 4) ? 2 : 1)
k_gemm_ws(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x, Params p) {
  constexpr int SMEM_BAR = FP8 ? NSTAGE * f8_stage(TOKN) + 2 * F8_CONV : NSTAGE * STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *sm = smem_raw + (base - smem_u32(smem_raw));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bar_full = base + SMEM_BAR, bar_empty = bar_full + 8 * NSTAGE, bar_acc = bar_empty + 8 * NSTAGE;
  const uint32_t conv_full = bar_acc + 8, conv_empty = conv_full + 16;  // fp8: the two bf16 half-tile slots
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(sm + SMEM_BAR + 16 * NSTAGE + (FP8 ? 48 : 16));
  constexpr int TMEM_N = FP8 ? TOKN : TMEM_COLS;
  // grid = (tiles, splits), or (splits, tiles) when the splits of a tile form a cluster (clusters run along x)
  const int tile = p.cluster ? blockIdx.y : blockIdx.x, split = p.cluster ? blockIdx.x : blockIdx.y;
  const int n0 = tile * BMW;
  const int grp = blockIdx.z;  // 0 unless the plan is a grouped GEMM (one group = one MoE expert)
  const int xk0 = grp * p.x_group_chunks;
  const int c0 = split * p.chunks_per_split;
  int c1 = c0 + p.chunks_per_split;
  if (c1 > p.n_chunks) c1 = p.n_chunks;
  const int nch = c1 - c0;

  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_acc, 1);
    if constexpr (FP8) {
      for (int h = 0; h < 2; ++h) { mbar_init(conv_full + 8 * h, 128); mbar_init(conv_empty + 8 * h, 1); }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();  // warp 0 reconverges before the block barrier below
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_N));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (!p.no_pdl) pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // Barriers + TMEM are set up while the previous kernel drains, and - the weights being immutable - the first
  // NSTAGE weight tiles are already streaming from HBM before griddepcontrol.wait: only the activation tiles (and
  // the output stores) depend on the predecessor, so its run time hides this kernel's pipeline fill.

  if constexpr (FP8) {
    constexpr int XH = TOKN * BK * 2, STG = f8_stage(TOKN), CONV0 = NSTAGE * STG, QT = TOKN / 4;
    constexpr uint32_t IDESC8 = idesc_tok(TOKN);
    if (warp == 0) {
      if (lane == 0) {
        const int blk0 = (grp * p.w_group_tiles + tile) * p.n_chunks + c0;
        auto load_x = [&](int i, int s) {  // the two 64-k activation boxes of fp8 chunk c0 + i
          const uint32_t xd = base + s * STG + F8_W;
          const int kc = xk0 + 2 * (c0 + i);
          tma_load_2d(xd, &map_x, bar_full + 8 * s, kc * BK, 0);
          tma_load_2d(xd + XH, &map_x, bar_full + 8 * s, (kc + 1) * BK, 0);
        };
        const int pre = nch < NSTAGE ? nch : NSTAGE;
        for (int i = 0; i < pre; ++i) {
          mbar_expect_tx(bar_full + 8 * i, STG);
          tma_load_3d(base + i * STG, &map_w, bar_full + 8 * i, 0, 0, blk0 + i);
        }
        pdl_wait();
        for (int i = 0; i < pre; ++i) load_x(i, i);
        for (int i = pre; i < nch; ++i) {
          const int s = i % NSTAGE, ph = (i / NSTAGE) & 1;
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          mbar_expect_tx(bar_full + 8 * s, STG);
          tma_load_3d(base + s * STG, &map_w, bar_full + 8 * s, 0, 0, blk0 + i);
          load_x(i, s);
        }
      }
      __syncwarp();
      if (p.cluster) { cluster_sync_all(); cluster_sync_all(); }
    } else if (warp == 1) {
      if (lane == 0) {
        for (int i = 0; i < nch; ++i) {
          const int s = i % NSTAGE, ph = (i / NSTAGE) & 1;
          mbar_wait(bar_full + 8 * s, ph);  // activation boxes landed
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            mbar_wait(conv_full + 8 * h, i & 1);  // bf16 half tile h written and fenced
            tc_fence_after();
            const uint32_t wa = base + CONV0 + h * F8_CONV, xa = base + s * STG + F8_W + h * XH;
#pragma unroll
            for (int j = 0; j < BK / 16; ++j)
              umma_bf16(tmem, kmajor_desc(wa + j * 32), kmajor_desc(xa + j * 32), IDESC8, (i | h | j) != 0);
            umma_commit(conv_empty + 8 * h);
          }
          umma_commit(bar_empty + 8 * s);
        }
        umma_commit(bar_acc);
      }
      __syncwarp();
      if (p.cluster) { cluster_sync_all(); cluster_sync_all(); }
    } else {
      const int q = warp & 3;
      const int r = q * 32 + lane, r7 = r & 7;
      // dequantise: thread = weight row r; 16-byte chunk c of a swizzled 128-byte row sits at chunk c ^ (r & 7)
      for (int i = 0; i < nch; ++i) {
        const int s = i % NSTAGE, ph = (i / NSTAGE) & 1;
        mbar_wait(bar_full + 8 * s, ph);
        const uint8_t *src = sm + s * STG + r * 128;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          mbar_wait(conv_empty + 8 * h, (i & 1) ^ 1);
          uint8_t *dst = sm + CONV0 + h * F8_CONV + r * 128;
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const uint4 f = *reinterpret_cast<const uint4 *>(src + (((h * 4 + c4) ^ r7) << 4));
            uint4 lo, hi;
            lo.x = e4m3x2_to_bf16x2(__byte_perm(f.x, 0, 0x1404)); lo.y = e4m3x2_to_bf16x2(__byte_perm(f.x, 0, 0x3424));
            lo.z = e4m3x2_to_bf16x2(__byte_perm(f.y, 0, 0x1404)); lo.w = e4m3x2_to_bf16x2(__byte_perm(f.y, 0, 0x3424));
            hi.x = e4m3x2_to_bf16x2(__byte_perm(f.z, 0, 0x1404)); hi.y = e4m3x2_to_bf16x2(__byte_perm(f.z, 0, 0x3424));
            hi.z = e4m3x2_to_bf16x2(__byte_perm(f.w, 0, 0x1404)); hi.w = e4m3x2_to_bf16x2(__byte_perm(f.w, 0, 0x3424));
            *reinterpret_cast<uint4 *>(dst + (((2 * c4) ^ r7) << 4)) = lo;
            *reinterpret_cast<uint4 *>(dst + (((2 * c4 + 1) ^ r7) << 4)) = hi;
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          mbar_arrive(conv_full + 8 * h);
        }
      }
      // epilogue: scale per weight row (= TMEM lane), bias, one rounding; 32 token columns at a time
      pdl_wait();
      if (nch > 0) { mbar_wait(bar_acc, 0); tc_fence_after(); }
      const uint32_t a = tmem + ((uint32_t)(q * 32) << 16);
      const float *scale = p.scale + (long long)grp * p.N;
      uint32_t v[32];
      auto load32 = [&](int cc) {
        if (nch > 0) { tmem_ld32(a + cc * 32, v); tmem_ld_wait(); }
        else {
#pragma unroll
          for (int t = 0; t < 32; ++t) v[t] = 0u;
        }
      };
      if (p.cluster) {
        // as the bf16 path: fp32 rows pushed to the owner CTA's (dead) stage ring, summed there in split order, then
        // scaled, biased and rounded once
        const int cs = p.cluster, RS = BMW / cs;
        cluster_sync_all();
        {
          const int owner = r / RS, rl = r % RS;
          const uint32_t dst = map_to_cta(base + (uint32_t)((split * QT) * RS + rl) * 16, owner);
          for (int cc = 0; cc < TOKN / 32; ++cc) {
            load32(cc);
#pragma unroll
            for (int u = 0; u < 8; ++u)
              st_cluster_f4(dst + (uint32_t)((cc * 8 + u) * RS) * 16, __uint_as_float(v[4 * u]), __uint_as_float(v[4 * u + 1]),
                            __uint_as_float(v[4 * u + 2]), __uint_as_float(v[4 * u + 3]));
          }
        }
        cluster_sync_all();
        {
          const int e = (warp - 2) * 32 + lane;
          const int rl = e % RS, tg = e / RS;
          const int qpt = QT * RS / BMW;               // token quads per thread
          const int n_out = n0 + split * RS + rl;
          const float4 *buf = reinterpret_cast<const float4 *>(sm);
          __nv_bfloat16 *ob = p.out_bf16 + grp * p.out_group_stride;
          const float sc = scale[n_out], bb = p.bias ? __bfloat162float(p.bias[n_out]) : 0.f;
          for (int tq = tg * qpt; tq < (tg + 1) * qpt; ++tq) {
            float4 acc = buf[tq * RS + rl];
            for (int src = 1; src < cs; ++src) {
              const float4 b = buf[(src * QT + tq) * RS + rl];
              acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
            }
            const int t0 = 4 * tq;
            if (t0 < p.rows) ob[(long long)t0 * p.N + n_out] = __float2bfloat16_rn(sc * acc.x + bb);
            if (t0 + 1 < p.rows) ob[(long long)(t0 + 1) * p.N + n_out] = __float2bfloat16_rn(sc * acc.y + bb);
            if (t0 + 2 < p.rows) ob[(long long)(t0 + 2) * p.N + n_out] = __float2bfloat16_rn(sc * acc.z + bb);
            if (t0 + 3 < p.rows) ob[(long long)(t0 + 3) * p.N + n_out] = __float2bfloat16_rn(sc * acc.w + bb);
          }
        }
      } else {
        const int n = n0 + r;  // N % 128 == 0: every row is in range
        const float sc = scale[n];
        // fp32 slices: every slice is scaled, the bias goes into slice 0 only
        const float bb = (p.bias && split == 0) ? __bfloat162float(p.bias[n]) : 0.f;
        for (int cc = 0; cc < TOKN / 32; ++cc) {
          load32(cc);
          if (p.n_split == 1) {
            __nv_bfloat16 *o = p.out_bf16 + grp * p.out_group_stride + n;
#pragma unroll
            for (int t = 0; t < 32; ++t)
              if (cc * 32 + t < p.rows) o[(long long)(cc * 32 + t) * p.N] = __float2bfloat16_rn(sc * __uint_as_float(v[t]) + bb);
          } else {
            float *o = p.out_f32 + (long long)split * TOKN * p.N + n;
#pragma unroll
            for (int t = 0; t < 32; ++t)
              if (cc * 32 + t < p.rows) o[(long long)(cc * 32 + t) * p.N] = sc * __uint_as_float(v[t]) + bb;
          }
        }
      }
      tc_fence_before();
    }
  } else
  if (warp == 0) {
    if (lane == 0) {
      auto load_w = [&](int i, int s) {
        const uint32_t wd = base + s * STAGE_BYTES;
        if (p.tiled) tma_load_3d(wd, &map_w, bar_full + 8 * s, 0, 0, tile * p.n_chunks + c0 + i);
        else tma_load_2d(wd, &map_w, bar_full + 8 * s, (c0 + i) * BK, grp * p.w_group_rows + n0);
      };
      const int pre = nch < NSTAGE ? nch : NSTAGE;
      for (int i = 0; i < pre; ++i) {  // all stages start empty
        mbar_expect_tx(bar_full + 8 * i, STAGE_BYTES);
        load_w(i, i);
      }
      pdl_wait();
      for (int i = 0; i < pre; ++i) tma_load_2d(base + i * STAGE_BYTES + W_BYTES, &map_x, bar_full + 8 * i, (xk0 + c0 + i) * BK, 0);
      for (int i = pre; i < nch; ++i) {
        const int s = i % NSTAGE, ph = (i / NSTAGE) & 1;
        mbar_wait(bar_empty + 8 * s, ph ^ 1);
        mbar_expect_tx(bar_full + 8 * s, STAGE_BYTES);
        load_w(i, s);
        tma_load_2d(base + s * STAGE_BYTES + W_BYTES, &map_x, bar_full + 8 * s, (xk0 + c0 + i) * BK, 0);
      }
    }
    __syncwarp();
    if (p.cluster) { cluster_sync_all(); cluster_sync_all(); }
  } else if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < nch; ++i) {
        const int s = i % NSTAGE, ph = (i / NSTAGE) & 1;
        mbar_wait(bar_full + 8 * s, ph);
        tc_fence_after();
        const uint32_t wa = base + s * STAGE_BYTES, xa = wa + W_BYTES;
#pragma unroll
        for (int j = 0; j < BK / 16; ++j)
          umma_bf16(tmem, kmajor_desc(wa + j * 32), kmajor_desc(xa + j * 32), IDESC, (i | j) != 0);
        umma_commit(bar_empty + 8 * s);
      }
      umma_commit(bar_acc);
    }
    __syncwarp();
    if (p.cluster) { cluster_sync_all(); cluster_sync_all(); }
  } else {
    // epilogue: thread = one weight row n (TMEM lane), 64 token values in registers
    pdl_wait();  // output stores (and the WAR hazard on the output buffer) are ordered after the predecessor
    const int q = warp & 3;
    const int n = n0 + q * 32 + lane;
    uint32_t v[64];
    if (nch > 0) {
      mbar_wait(bar_acc, 0);
      tc_fence_after();
      const uint32_t a = tmem + ((uint32_t)(q * 32) << 16);
      tmem_ld32(a, v);
      tmem_ld32(a + 32, v + 32);
      tmem_ld_wait();
    } else {
#pragma unroll
      for (int t = 0; t < 64; ++t) v[t] = 0u;
    }
    if (p.cluster) {
      // split-K inside a cluster: after everyone has left its main loop (barrier A: the pipeline stages of every CTA
      // are dead) each thread pushes its fp32 row - 16 token quads, quad-major so that the lanes of a warp write
      // consecutive 16-byte words - into the CTA that owns that row slice, barrier B, and the owner adds the
      // cluster's partials in split order (deterministic) and writes bf16.  No fp32 round trip through HBM/L2.
      const int cs = p.cluster, RS = BMW / cs;      // rows per owner CTA: 64 (2 splits) or 32 (4 splits)
      cluster_sync_all();
      {
        const int row = q * 32 + lane;
        const int owner = row / RS, rl = row % RS;
        const uint32_t dst = map_to_cta(base + (uint32_t)((split * 16) * RS + rl) * 16, owner);
#pragma unroll
        for (int tq = 0; tq < 16; ++tq)
          st_cluster_f4(dst + (uint32_t)(tq * RS) * 16, __uint_as_float(v[4 * tq]), __uint_as_float(v[4 * tq + 1]),
                        __uint_as_float(v[4 * tq + 2]), __uint_as_float(v[4 * tq + 3]));
      }
      cluster_sync_all();
      {
        const int e = (warp - 2) * 32 + lane;       // 0..127
        const int rl = e % RS, tg = e / RS;         // row of this CTA's slice, token group
        const int qpt = RS / 8;                     // token quads per thread: 16 / (128 / RS)
        const int n_out = n0 + split * RS + rl;     // this CTA's rank in the cluster == its split index
        const float4 *buf = reinterpret_cast<const float4 *>(sm);
        __nv_bfloat16 *ob = p.out_bf16 + grp * p.out_group_stride;
        if (n_out < p.N) {
          for (int tq = tg * qpt; tq < (tg + 1) * qpt; ++tq) {
            float4 a = buf[(0 * 16 + tq) * RS + rl];
            for (int src = 1; src < cs; ++src) {
              const float4 b = buf[(src * 16 + tq) * RS + rl];
              a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
            }
            const int t0 = 4 * tq;
            if (t0 < p.rows) ob[(long long)t0 * p.N + n_out] = __float2bfloat16_rn(a.x);
            if (t0 + 1 < p.rows) ob[(long long)(t0 + 1) * p.N + n_out] = __float2bfloat16_rn(a.y);
            if (t0 + 2 < p.rows) ob[(long long)(t0 + 2) * p.N + n_out] = __float2bfloat16_rn(a.z);
            if (t0 + 3 < p.rows) ob[(long long)(t0 + 3) * p.N + n_out] = __float2bfloat16_rn(a.w);
          }
        }
      }
    } else
    if (p.silu) {
      // act(gate) * up (modeling_llama.py:185-186) in the epilogue: lanes 0-63 (warps q = 0, 1) hold gate rows, lanes
      // 64-127 (q = 2, 3) the up rows of the same 64 output columns.  Each warp pair splits the 64 tokens: the gate warp
      // finishes tokens 0-31 (it receives the up values through shared memory), the up warp tokens 32-63 (it receives the
      // gate values), so all four warps share the exponentials.  Rounding points as in eager bf16 (and k_silu_mul):
      // GEMM out -> bf16, silu -> bf16, product -> bf16.
      __nv_bfloat16 *xu = reinterpret_cast<__nv_bfloat16 *>(sm + SMEM_BAR + 256);  // up   [32 tokens 0-31 ][64 rows]
      __nv_bfloat16 *xg = xu + 32 * 64;                                             // gate [32 tokens 32-63][64 rows]
      const int rr = (q & 1) * 32 + lane;
      if (q >= 2) {
#pragma unroll
        for (int t = 0; t < 32; ++t) xu[t * 64 + rr] = __float2bfloat16_rn(__uint_as_float(v[t]));
      } else {
#pragma unroll
        for (int t = 0; t < 32; ++t) xg[t * 64 + rr] = __float2bfloat16_rn(__uint_as_float(v[32 + t]));
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const int col = tile * 64 + rr;
      const int inter = p.N >> 1;
      if (col < inter) {
        const int tb = q < 2 ? 0 : 32;
#pragma unroll
        for (int t = 0; t < 32; ++t) {
          if (tb + t < p.rows) {
            const float g = q < 2 ? __bfloat162float(__float2bfloat16_rn(__uint_as_float(v[t]))) : __bfloat162float(xg[t * 64 + rr]);
            const float u = q < 2 ? __bfloat162float(xu[t * 64 + rr]) : __bfloat162float(__float2bfloat16_rn(__uint_as_float(v[32 + t])));
            const float sg = __bfloat162float(__float2bfloat16_rn(g / (1.f + expf(-g))));
            p.out_bf16[(long long)(tb + t) * inter + col] = __float2bfloat16_rn(sg * u);
          }
        }
      }
    } else
    if (n < p.N) {
      if (p.n_split == 1) {
#pragma unroll
        for (int t = 0; t < TOK; ++t)
          if (t < p.rows) p.out_bf16[grp * p.out_group_stride + (long long)t * p.N + n] = __float2bfloat16_rn(__uint_as_float(v[t]));
      } else {
        float *o = p.out_f32 + (long long)split * TOK * p.N;
#pragma unroll
        for (int t = 0; t < TOK; ++t)
          if (t < p.rows) o[(long long)t * p.N + n] = __uint_as_float(v[t]);
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_N));
  }
}


// ------------------------------------------------------------------------------------------------ stream-K
// Work = n_tiles x n_chunks (tile, k-chunk) units, cut into gridDim.x equal contiguous ranges: every SM streams
// the same number of bytes whatever N is (qkv: 96 tiles, o/down: 32 tiles on 148 SMs).  A tile whose chunks span
// several CTAs is finished by the CTA that holds its FIRST chunk (it reaches that tile last in its own range, so the
// other contributors - which meet the tile first in theirs - are normally done already): contributors store their
// fp32 partial to a workspace slot and bump the tile's flag, the owner adds the slots in slot order (deterministic)
// and writes bf16.  All CTAs are co-resident (grid <= #SMs, one CTA per SM), so the owner's wait cannot deadlock.
struct SkParams {
  int N, n_tiles, n_chunks, rows, max_contrib;
  long long units;
  __nv_bfloat16 *out;   // [rows_cap, N]
  float *ws;            // [n_tiles][max_contrib][128][64]
  int *flags;           // [n_tiles], zero between launches
};

__device__ __forceinline__ long long sk_begin(long long b, long long U, int G) { return b * U / G; }
__device__ __forceinline__ int sk_cta_of(long long x, long long U, int G) {
  int b = (int)(x * G / U);
  while (b + 1 < G && sk_begin(b + 1, U, G) <= x) ++b;
  while (b > 0 && sk_begin(b, U, G) > x) --b;
  return b;
}

constexpr int SK_STAGES = 8;
constexpr int SK_SMEM_BAR = SK_STAGES * STAGE_BYTES;
constexpr int SK_SMEM_TOTAL = SK_SMEM_BAR + 256 + 1024;
constexpr int SK_TMEM_COLS = 128;  // two 64-column accumulators

__global__ void __launch_bounds__(NTHREADS, 1)
k_gemm_sk(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x, SkParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *sm = smem_raw + (base - smem_u32(smem_raw));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bar_full = base + SK_SMEM_BAR, bar_empty = bar_full + 8 * SK_STAGES, bar_acc_full = bar_empty + 8 * SK_STAGES,
                 bar_acc_empty = bar_acc_full + 16;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(sm + SK_SMEM_BAR + 16 * SK_STAGES + 48);
  const int G = gridDim.x, b = blockIdx.x;
  const long long u0 = sk_begin(b, p.units, G), u1 = sk_begin(b + 1, p.units, G);

  if (tid == 0) {
    for (int s = 0; s < SK_STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_acc_full, 1); mbar_init(bar_acc_full + 8, 1);
    mbar_init(bar_acc_empty, 128); mbar_init(bar_acc_empty + 8, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();  // warp 0 reconverges before the block barrier below
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(SK_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      int i = 0;
      for (long long u = u0; u < u1; ++u, ++i) {
        const int tile = (int)(u / p.n_chunks), ch = (int)(u % p.n_chunks);
        const int s = i % SK_STAGES, ph = (i / SK_STAGES) & 1;
        mbar_wait(bar_empty + 8 * s, ph ^ 1);
        mbar_expect_tx(bar_full + 8 * s, STAGE_BYTES);
        const uint32_t wd = base + s * STAGE_BYTES, xd = wd + W_BYTES;
        tma_load_3d(wd, &map_w, bar_full + 8 * s, 0, 0, tile * p.n_chunks + ch);
        tma_load_2d(xd, &map_x, bar_full + 8 * s, ch * BK, 0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int i = 0, seg = 0;
      long long u = u0;
      while (u < u1) {
        const int tile = (int)(u / p.n_chunks);
        long long ue = (long long)(tile + 1) * p.n_chunks;
        if (ue > u1) ue = u1;
        const int buf = seg & 1;
        mbar_wait(bar_acc_empty + 8 * buf, ((seg >> 1) & 1) ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d = tmem + buf * 64;
        bool first = true;
        for (; u < ue; ++u, ++i) {
          const int s = i % SK_STAGES, ph = (i / SK_STAGES) & 1;
          mbar_wait(bar_full + 8 * s, ph);
          tc_fence_after();
          const uint32_t wa = base + s * STAGE_BYTES, xa = wa + W_BYTES;
#pragma unroll
          for (int j = 0; j < BK / 16; ++j) {
            umma_bf16(d, kmajor_desc(wa + j * 32), kmajor_desc(xa + j * 32), IDESC, !(first && j == 0));
          }
          first = false;
          umma_commit(bar_empty + 8 * s);
        }
        umma_commit(bar_acc_full + 8 * buf);
        ++seg;
      }
    }
  } else {
    // epilogue warps: thread = one weight row of the tile (TMEM lane), 64 token values
    const int q = warp & 3;
    const int r = q * 32 + lane;
    int seg = 0;
    long long u = u0;
    uint32_t v[64];
    while (u < u1) {
      const int tile = (int)(u / p.n_chunks);
      const long long ts = (long long)tile * p.n_chunks;
      long long ue = ts + p.n_chunks;
      if (ue > u1) ue = u1;
      const int buf = seg & 1;
      mbar_wait(bar_acc_full + 8 * buf, (seg >> 1) & 1);
      tc_fence_after();
      const uint32_t a = tmem + buf * 64 + ((uint32_t)(q * 32) << 16);
      tmem_ld32(a, v);
      tmem_ld32(a + 32, v + 32);
      tmem_ld_wait();
      tc_fence_before();
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_acc_empty + 8 * buf) : "memory");
      const bool head = (u == ts), whole = head && (ue == ts + p.n_chunks);
      const int n = tile * BMW + r;
      if (!head) {
        // contributor: slot = how many CTA ranges after the owner's this one is
        const int owner = sk_cta_of(ts, p.units, G);
        const int slot = b - owner - 1;
        float4 *dst = reinterpret_cast<float4 *>(p.ws + (((long long)tile * p.max_contrib + slot) * BMW + r) * TOK);
#pragma unroll
        for (int t = 0; t < 16; ++t)
          dst[t] = make_float4(__uint_as_float(v[4 * t]), __uint_as_float(v[4 * t + 1]), __uint_as_float(v[4 * t + 2]),
                               __uint_as_float(v[4 * t + 3]));
        __threadfence();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (r == 0) atomicAdd(&p.flags[tile], 1);
      } else {
        if (!whole) {
          // owner: wait for the other contributors of this tile, then add their slots in order
          const int last = sk_cta_of(ts + p.n_chunks - 1, p.units, G);
          const int contributors = last - b;
          if (r == 0) {
            while (atomicAdd(&p.flags[tile], 0) < contributors) __nanosleep(64);
            p.flags[tile] = 0;  // self-reset for the next launch
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");
          __threadfence();
          for (int c = 0; c < contributors; ++c) {
            const float4 *src = reinterpret_cast<const float4 *>(p.ws + (((long long)tile * p.max_contrib + c) * BMW + r) * TOK);
#pragma unroll
            for (int t = 0; t < 16; ++t) {
              const float4 x = __ldcg(src + t);
              v[4 * t] = __float_as_uint(__uint_as_float(v[4 * t]) + x.x);
              v[4 * t + 1] = __float_as_uint(__uint_as_float(v[4 * t + 1]) + x.y);
              v[4 * t + 2] = __float_as_uint(__uint_as_float(v[4 * t + 2]) + x.z);
              v[4 * t + 3] = __float_as_uint(__uint_as_float(v[4 * t + 3]) + x.w);
            }
          }
        }
        if (n < p.N) {
#pragma unroll
          for (int t = 0; t < TOK; ++t)
            if (t < p.rows) p.out[(long long)t * p.N + n] = __float2bfloat16_rn(__uint_as_float(v[t]));
        }
      }
      u = ue;
      ++seg;
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(SK_TMEM_COLS));
  }
}

}  // namespace gemm
}  // namespace pia

using namespace pia;
using namespace pia::gemm;

struct pia_gemm_plan {
  CUtensorMap map_w, map_x;
  Params p;
  int nstage;
  int no_pdl;  // 1: launched without the programmatic-dependent-launch attribute (a plain kernel boundary, like cuBLAS)
  // stream-K mode
  int stream_k, sk_grid;
  SkParams sk;
  int fp8, tok, x_rows;  // fp8-weight plan: token rows per launch (UMMA N) and rows of the activation buffer
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    void *ptr = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

// weights pre-tiled in HBM: [N/128 * K/64] contiguous 16 KB blocks of 128 rows x 64 k (one TMA box each), so a CTA
// streams one contiguous slab instead of 128 strided 128-byte pieces per stage
static int encode_tiled_w(CUtensorMap *m, const void *base, uint64_t n_blocks) {
  EncodeTiledFn fn = get_encode();
  PIA_REQUIRE(fn, "cuTensorMapEncodeTiled not available in this driver");
  cuuint64_t dims[3] = {(cuuint64_t)BK, (cuuint64_t)BMW, n_blocks};
  cuuint64_t strides[2] = {(cuuint64_t)BK * 2, (cuuint64_t)BK * BMW * 2};
  cuuint32_t box[3] = {BK, BMW, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return PIA_ERR_CUDA; }
  return PIA_OK;
}

static int encode_2d(CUtensorMap *m, const void *base, uint64_t inner, uint64_t outer, uint32_t box_inner,
                     uint32_t box_outer, CUtensorMapL2promotion promo) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    void *ptr = nullptr;
    PIA_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres));
    PIA_REQUIRE(ptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available in this driver");
    fn = (EncodeTiledFn)ptr;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {inner * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return PIA_ERR_CUDA; }
  return PIA_OK;
}

extern "C" int pia_gemm_plan_create(const void *d_w, int N, int K, const void *d_x, int x_rows, int split_k,
                                    int w_tiled, pia_gemm_plan_t **out) {
  PIA_REQUIRE(d_w && d_x && out, "null argument");
  PIA_REQUIRE(N > 0 && K > 0 && K % BK == 0, "K must be a multiple of %d", BK);
  PIA_REQUIRE(x_rows >= TOK, "the activation buffer must hold at least %d rows", TOK);
  PIA_REQUIRE((reinterpret_cast<uintptr_t>(d_w) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_x) & 15) == 0, "operands must be 16-byte aligned");
  pia_gemm_plan *g = new (std::nothrow) pia_gemm_plan();
  PIA_REQUIRE(g, "out of host memory");
  const int n_chunks = K / BK;
  const int want_stream_k = (split_k == -1);
  const int want_cluster = (split_k == -2 || split_k == -4 || split_k == -8) ? -split_k : 0;
  if (split_k < -1 && !want_cluster) { delete g; set_error("cluster split-K supports 2, 4 or 8 CTAs"); return PIA_ERR_INVALID; }
  if (want_cluster) split_k = want_cluster;
  if (split_k < 1) split_k = 1;
  if (split_k > n_chunks) split_k = n_chunks;
  g->p.N = N; g->p.K = K; g->p.n_chunks = n_chunks;
  g->p.chunks_per_split = (n_chunks + split_k - 1) / split_k;
  g->p.n_split = (n_chunks + g->p.chunks_per_split - 1) / g->p.chunks_per_split;
  g->p.rows = TOK; g->p.out_bf16 = nullptr; g->p.out_f32 = nullptr; g->p.silu = 0;
  g->p.groups = 1; g->p.w_group_rows = 0; g->p.x_group_chunks = 0; g->p.out_group_stride = 0;
  g->p.cluster = 0;
  if (want_cluster) {
    if (g->p.n_split != want_cluster) { delete g; set_error("K = %d is too short for %d cluster splits", K, want_cluster); return PIA_ERR_INVALID; }
    g->p.cluster = want_cluster;
  }
  g->p.tiled = w_tiled ? 1 : 0;
  if (w_tiled && N % BMW != 0) { delete g; set_error("a tiled weight needs N %% %d == 0", BMW); return PIA_ERR_INVALID; }
  int rc = w_tiled ? encode_tiled_w(&g->map_w, d_w, (uint64_t)(N / BMW) * n_chunks)
                   : encode_2d(&g->map_w, d_w, (uint64_t)K, (uint64_t)N, BK, BMW, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
  if (rc == PIA_OK) rc = encode_2d(&g->map_x, d_x, (uint64_t)K, (uint64_t)x_rows, BK, TOK, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
  if (rc == PIA_OK) {
    int n_sm = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    const int ctas = ((N + BMW - 1) / BMW) * g->p.n_split;
    g->nstage = ctas <= n_sm ? 8 : 4;
    cudaError_t e = cudaFuncSetAttribute(k_gemm_ws<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_total(4));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_gemm_ws<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_total(8));
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); rc = PIA_ERR_CUDA; }
  }
  g->stream_k = 0; g->no_pdl = 0;
  if (rc == PIA_OK && want_stream_k) {
    // stream-K over the HBM-tiled weight: grid = min(#SMs, units), fix-up workspace owned by the plan
    if (!w_tiled) { delete g; set_error("stream-K needs the tiled weight layout"); return PIA_ERR_INVALID; }
    int n_sm = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    SkParams &k = g->sk;
    k.N = N; k.n_tiles = N / BMW; k.n_chunks = n_chunks; k.rows = TOK;
    k.units = (long long)k.n_tiles * n_chunks;
    g->sk_grid = (int)(k.units < n_sm ? k.units : n_sm);
    const long long per = (k.units + g->sk_grid - 1) / g->sk_grid;
    k.max_contrib = (int)((n_chunks + per - 1) / per) + 1;
    k.out = nullptr;
    cudaError_t e = cudaMalloc((void **)&k.ws, sizeof(float) * (size_t)k.n_tiles * k.max_contrib * BMW * TOK);
    if (e == cudaSuccess) e = cudaMalloc((void **)&k.flags, sizeof(int) * k.n_tiles);
    if (e == cudaSuccess) e = cudaMemset(k.flags, 0, sizeof(int) * k.n_tiles);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_gemm_sk, cudaFuncAttributeMaxDynamicSharedMemorySize, SK_SMEM_TOTAL);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { set_error("stream-K plan: %s", cudaGetErrorString(e)); delete g; return PIA_ERR_CUDA; }
    g->stream_k = 1;
    g->p.n_split = 1;
  }
  if (rc != PIA_OK) { delete g; return rc; }
  *out = g;
  return PIA_OK;
}

extern "C" int pia_gemm_plan_destroy(pia_gemm_plan_t *g) {
  if (g) {
    if (g->stream_k) { cudaFree(g->sk.ws); cudaFree(g->sk.flags); }
    delete g;
  }
  return PIA_OK;
}
extern "C" int pia_gemm_plan_set_pdl(pia_gemm_plan_t *g, int on) {
  PIA_REQUIRE(g, "null plan");
  g->no_pdl = on ? 0 : 1;
  return PIA_OK;
}
extern "C" int pia_gemm_plan_splits(const pia_gemm_plan_t *g) { return g ? (g->p.cluster ? 1 : g->p.n_split) : 0; }
extern "C" int pia_gemm_plan_set_silu(pia_gemm_plan_t *g, int on) {
  PIA_REQUIRE(g && !g->fp8 && g->p.n_split == 1 && !g->stream_k && g->p.N % BMW == 0, "the SiLU*up epilogue needs split_k == 1 and N %% 128 == 0");
  g->p.silu = on ? 1 : 0;
  return PIA_OK;
}

// Grouped GEMM (MoE experts, mixtral/modeling_mixtral.py:692-759): out[g] = X[:, g*K:(g+1)*K] @ W[g]^T for `groups`
// stacked weights W [groups*N, K] (row-major) and activations X [x_rows, groups*K]; one launch, gridDim.z = groups.
extern "C" int pia_gemm_plan_create_grouped(const void *d_w, int groups, int N, int K, const void *d_x, int x_rows,
                                            pia_gemm_plan_t **out) {
  PIA_REQUIRE(d_w && d_x && out, "null argument");
  PIA_REQUIRE(groups >= 1 && groups <= 65535 && N > 0 && N % BMW == 0 && K > 0 && K % BK == 0,
              "grouped GEMM needs N %% %d == 0 and K %% %d == 0", BMW, BK);
  PIA_REQUIRE(x_rows >= TOK, "the activation buffer must hold at least %d rows", TOK);
  PIA_REQUIRE((reinterpret_cast<uintptr_t>(d_w) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_x) & 15) == 0, "operands must be 16-byte aligned");
  pia_gemm_plan *g = new (std::nothrow) pia_gemm_plan();
  PIA_REQUIRE(g, "out of host memory");
  const int n_chunks = K / BK;
  g->p.N = N; g->p.K = K; g->p.n_chunks = n_chunks; g->p.chunks_per_split = n_chunks; g->p.n_split = 1;
  g->p.rows = TOK; g->p.out_bf16 = nullptr; g->p.out_f32 = nullptr; g->p.silu = 0; g->p.tiled = 0; g->p.cluster = 0;
  g->p.groups = groups; g->p.w_group_rows = N; g->p.x_group_chunks = n_chunks; g->p.out_group_stride = (long long)TOK * N;
  g->stream_k = 0; g->no_pdl = 0;
  int rc = encode_2d(&g->map_w, d_w, (uint64_t)K, (uint64_t)groups * N, BK, BMW, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
  if (rc == PIA_OK) rc = encode_2d(&g->map_x, d_x, (uint64_t)groups * K, (uint64_t)x_rows, BK, TOK, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
  if (rc == PIA_OK) {
    int n_sm = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    g->nstage = (N / BMW) * groups <= n_sm ? 8 : 4;
    cudaError_t e = cudaFuncSetAttribute(k_gemm_ws<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_total(4));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_gemm_ws<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_total(8));
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); rc = PIA_ERR_CUDA; }
  }
  if (rc != PIA_OK) { delete g; return rc; }
  *out = g;
  return PIA_OK;
}

// e4m3 weights pre-tiled by tile_weight_fp8: [blocks] contiguous 16 KB boxes of 128 rows x 128 k bytes
static int encode_tiled_w_fp8(CUtensorMap *m, const void *base, uint64_t n_blocks) {
  EncodeTiledFn fn = get_encode();
  PIA_REQUIRE(fn, "cuTensorMapEncodeTiled not available in this driver");
  cuuint64_t dims[3] = {(cuuint64_t)F8_BK, (cuuint64_t)BMW, n_blocks};
  cuuint64_t strides[2] = {(cuuint64_t)F8_BK, (cuuint64_t)F8_BK * BMW};
  cuuint32_t box[3] = {F8_BK, BMW, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return PIA_ERR_CUDA; }
  return PIA_OK;
}

// the fp8 instantiations: (stages, token rows)
template <int NS, int T>
static cudaError_t f8_attr() {
  return cudaFuncSetAttribute(k_gemm_ws<NS, T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, f8_smem_total(NS, T));
}
template <int NS, int T>
static cudaError_t f8_launch(const pia_gemm_plan *g, const Params &p, cudaStream_t st) {
  const int smem = f8_smem_total(NS, T);
  if (p.cluster)
    return launch_kernel_cluster(k_gemm_ws<NS, T, true>, dim3(p.n_split, p.N / BMW), dim3(NTHREADS), smem, st,
                                 (unsigned)p.cluster, g->map_w, g->map_x, p);
  return launch_kernel(k_gemm_ws<NS, T, true>, dim3(p.N / BMW, p.n_split, p.groups), dim3(NTHREADS), smem, st, g->map_w,
                       g->map_x, p);
}

static int fp8_plan_create(const void *d_w, const float *d_scale, const void *d_bias, int groups, int N, int K,
                           const void *d_x, int x_rows, int split_k, pia_gemm_plan_t **out) {
  PIA_REQUIRE(d_w && d_scale && d_x && out, "null argument");
  PIA_REQUIRE(groups >= 1 && groups <= 65535, "groups %d outside [1, 65535]", groups);
  PIA_REQUIRE(N > 0 && K > 0 && N % BMW == 0 && K % F8_BK == 0, "fp8 weights need N %% %d == 0 and K %% %d == 0 (N = %d, K = %d)",
              BMW, F8_BK, N, K);
  PIA_REQUIRE(x_rows >= 1 && x_rows <= 256, "the activation buffer of an fp8 plan holds 1..256 rows, not %d", x_rows);
  PIA_REQUIRE((reinterpret_cast<uintptr_t>(d_w) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_x) & 15) == 0 &&
              (reinterpret_cast<uintptr_t>(d_scale) & 3) == 0 && (reinterpret_cast<uintptr_t>(d_bias) & 1) == 0,
              "operands must be aligned (weights / activations 16 bytes)");
  const int n_chunks = K / F8_BK;
  const int want_cluster = (split_k == -2 || split_k == -4 || split_k == -8) ? -split_k : 0;
  PIA_REQUIRE(split_k >= 1 || want_cluster, "fp8 plans take split_k >= 1 or a cluster split of -2, -4 or -8");
  PIA_REQUIRE(groups == 1 || split_k == 1, "grouped fp8 plans do not split K");
  if (want_cluster) split_k = want_cluster;
  if (split_k > n_chunks) split_k = n_chunks;
  pia_gemm_plan *g = new (std::nothrow) pia_gemm_plan();
  PIA_REQUIRE(g, "out of host memory");
  g->fp8 = 1;
  g->tok = x_rows <= 64 ? 64 : x_rows <= 128 ? 128 : 256;
  g->x_rows = x_rows;
  Params &p = g->p;
  p.N = N; p.K = K; p.n_chunks = n_chunks;
  p.chunks_per_split = (n_chunks + split_k - 1) / split_k;
  p.n_split = (n_chunks + p.chunks_per_split - 1) / p.chunks_per_split;
  p.rows = g->tok; p.out_bf16 = nullptr; p.out_f32 = nullptr; p.silu = 0; p.tiled = 1; p.cluster = 0;
  p.groups = groups; p.w_group_rows = N; p.x_group_chunks = K / BK; p.out_group_stride = (long long)g->tok * N;
  p.scale = d_scale; p.bias = (const __nv_bfloat16 *)d_bias; p.w_group_tiles = N / BMW;
  g->stream_k = 0; g->no_pdl = 0;
  if (want_cluster) {
    if (p.n_split != want_cluster) { delete g; set_error("K = %d is too short for %d cluster splits", K, want_cluster); return PIA_ERR_INVALID; }
    p.cluster = want_cluster;
  }
  int rc = encode_tiled_w_fp8(&g->map_w, d_w, (uint64_t)groups * (N / BMW) * n_chunks);
  if (rc == PIA_OK) rc = encode_2d(&g->map_x, d_x, (uint64_t)groups * K, (uint64_t)x_rows, BK, g->tok, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
  if (rc == PIA_OK) {
    int n_sm = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    const int ctas = (N / BMW) * p.n_split * groups;
    g->nstage = g->tok == 64 ? (ctas <= n_sm ? 5 : 2) : g->tok == 128 ? 4 : 2;
    cudaError_t e = g->tok == 64 ? (g->nstage == 5 ? f8_attr<5, 64>() : f8_attr<2, 64>())
                  : g->tok == 128 ? f8_attr<4, 128>() : f8_attr<2, 256>();
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); rc = PIA_ERR_CUDA; }
  }
  if (rc != PIA_OK) { delete g; return rc; }
  *out = g;
  return PIA_OK;
}

extern "C" int pia_gemm_plan_create_fp8(const void *d_w_tiled_f8, const float *d_scale, const void *d_bias, int N, int K,
                                        const void *d_x, int x_rows, int split_k, pia_gemm_plan_t **out) {
  return fp8_plan_create(d_w_tiled_f8, d_scale, d_bias, 1, N, K, d_x, x_rows, split_k, out);
}

extern "C" int pia_gemm_plan_create_grouped_fp8(const void *d_w_tiled_f8, const float *d_scale, int groups, int N, int K,
                                                const void *d_x, int x_rows, pia_gemm_plan_t **out) {
  return fp8_plan_create(d_w_tiled_f8, d_scale, nullptr, groups, N, K, d_x, x_rows, 1, out);
}

struct PdlScope { int on; explicit PdlScope(int off) : on(off) { if (on) ++pia::g_pdl_off; } ~PdlScope() { if (on) --pia::g_pdl_off; } };

extern "C" int pia_gemm_run(pia_gemm_plan_t *g, int rows, void *d_out, void *stream) {
  PIA_REQUIRE(g && d_out, "null argument");
  if (g->fp8) {
    PIA_REQUIRE(rows >= 1 && rows <= g->x_rows, "rows %d outside [1,%d]", rows, g->x_rows);
    PdlScope pdl_scope(g->no_pdl);
    Params p = g->p;
    p.rows = rows; p.no_pdl = g->no_pdl;
    if (p.n_split == 1 || p.cluster) p.out_bf16 = (__nv_bfloat16 *)d_out; else p.out_f32 = (float *)d_out;
    cudaStream_t st = (cudaStream_t)stream;
    const cudaError_t e = g->tok == 64 ? (g->nstage == 5 ? f8_launch<5, 64>(g, p, st) : f8_launch<2, 64>(g, p, st))
                        : g->tok == 128 ? f8_launch<4, 128>(g, p, st) : f8_launch<2, 256>(g, p, st);
    PIA_CUDA_CHECK(e);
    count_launch();
    return PIA_OK;
  }
  PIA_REQUIRE(rows >= 1 && rows <= TOK, "rows %d outside [1,%d]", rows, TOK);
  PdlScope pdl_scope(g->no_pdl);
  if (g->stream_k) {
    SkParams k = g->sk;
    k.rows = rows;
    k.out = (__nv_bfloat16 *)d_out;
    PIA_CUDA_CHECK(launch_kernel(k_gemm_sk, dim3(g->sk_grid), dim3(NTHREADS), SK_SMEM_TOTAL, (cudaStream_t)stream, g->map_w, g->map_x, k));
    count_launch();
    return PIA_OK;
  }
  Params p = g->p;
  p.rows = rows; p.no_pdl = g->no_pdl;
  if (p.n_split == 1 || p.cluster) p.out_bf16 = (__nv_bfloat16 *)d_out; else p.out_f32 = (float *)d_out;
  if (p.cluster) {
    dim3 cgrid(p.n_split, (p.N + BMW - 1) / BMW);
    if (g->nstage == 8) PIA_CUDA_CHECK(launch_kernel_cluster(k_gemm_ws<8>, cgrid, dim3(NTHREADS), smem_total(8), (cudaStream_t)stream, (unsigned)p.cluster, g->map_w, g->map_x, p));
    else PIA_CUDA_CHECK(launch_kernel_cluster(k_gemm_ws<4>, cgrid, dim3(NTHREADS), smem_total(4), (cudaStream_t)stream, (unsigned)p.cluster, g->map_w, g->map_x, p));
    count_launch();
    return PIA_OK;
  }
  dim3 grid((p.N + BMW - 1) / BMW, p.n_split, p.groups);
  if (g->nstage == 8) PIA_CUDA_CHECK(launch_kernel(k_gemm_ws<8>, grid, dim3(NTHREADS), smem_total(8), (cudaStream_t)stream, g->map_w, g->map_x, p));
  else PIA_CUDA_CHECK(launch_kernel(k_gemm_ws<4>, grid, dim3(NTHREADS), smem_total(4), (cudaStream_t)stream, g->map_w, g->map_x, p));
  count_launch();
  return PIA_OK;
}
