// Tree-masked attention for the LOOKAHEAD verify forward (sm_100a: TMA + tcgen05 + TMEM).
//
// Takes over the eager attention of the reference's patched models
//   models/llama/modeling_llama.py:243-308 (QK^T/sqrt(d) + mask, fp32 softmax, PV) with the lookahead mask of
//   :584-588 and common/pretrained_model.py:725-734 ([n, P+n] = visible prefix || tree mask).
// The mask is never materialised: prefix keys [pad_len, P) are visible to every row, the n draft keys follow the
// row's ancestor bit set (uint64 words, produced by the trie kernel) held in registers.
//
// One CTA = (KV split, head group).  A head group is up to two query heads of ONE KV head packed into a single
// UMMA M=128 tile: 2 query heads x 64 draft rows under GQA, 1 head otherwise (rows 64..127 idle for MHA/64).  With an
// odd group size G the last group of each KV head holds its single leftover head (rows 64..127 idle as for MHA), so a
// pair never straddles two KV heads: group g -> KV head g / ceil(G/2), heads hkv*G + 2j (+1), j = g % ceil(G/2).
// Warp roles (320 threads):  warp 0 = TMA producer (K/V tiles of 128 keys, 2-stage ring),
//                            warp 1 = TMEM owner + single-thread tcgen05.mma issuer,
//                            warps 2-9 = softmax / accumulate, two threads per row (TMEM lane == row; each
//                            takes 64 S columns and 64 O columns, row max / sum exchanged through smem).
// Per 128-key tile:  S = Q K^T (8 x UMMA 128x128x16 SS, fp32 in TMEM, double buffered)
//                    -> hidden keys to -inf (one 32-bit visibility word per 32 keys), online softmax in fp32
//                    -> P (bf16 pairs) back to TMEM (tcgen05.st, double buffered) = the A operand of
//                    -> O_tile = P V (8 x UMMA TS form, V consumed MN-major straight from the TMA tile)
//                    -> acc = acc * alpha + O_tile in registers, one tile late, so that PV(i) and QK^T(i+1) run on
//                       the tensor core while the softmax warps are busy with tile i+1.
// The KV range is split across the CTAs of a thread-block cluster (one wave of clusters, split count decided on the
// device from the live length): a single-split CTA normalises and writes bf16 directly; otherwise every thread
// pushes its partial row (acc, m, l) into the shared memory of the CTA that owns the row (DSMEM) and each CTA
// combines its row slice locally - no workspace in HBM, no separate combine launch.
// HBM-bound by design (arithmetic intensity = rows per KV byte: 64 FLOP/B for MHA, 256 for GQA-4;
// DESIGN.md gives the roofline).
#include <cuda.h>
#include <cuda_bf16.h>

#include <stdlib.h>

#include <new>

#include "common.cuh"

namespace pia {
namespace attn {

constexpr int BM = 128;      // rows per CTA (UMMA M)
constexpr int BN = 128;      // keys per tile (UMMA N of QK^T, K extent of PV)
constexpr int HD = 128;      // head dim
constexpr int NSTAGE = 2;
constexpr int NTHREADS = 320;   // warp 0 TMA, warp 1 MMA, warps 2-9 softmax (two warps per TMEM lane quadrant)
constexpr int SUB = 128 * 128;             // bytes of one [128 rows x 64 bf16] swizzle-128B sub-tile
constexpr int TILE_BYTES = 2 * SUB;        // one 128 x 128 bf16 operand tile
constexpr int SMEM_Q = 0, SMEM_K = TILE_BYTES, SMEM_V = SMEM_K + NSTAGE * TILE_BYTES;  // P lives in TMEM
constexpr int SMEM_BAR = SMEM_V + NSTAGE * TILE_BYTES;
constexpr int MRG_ACC = 0;                        // [n_split * RS][128] fp32 partial rows pushed by the cluster (over dead Q/P/KV tiles)
constexpr int MRG_ML = 112 * 1024;                // [n_split * RS] (m, l) pairs
constexpr int SMEM_XCH = SMEM_BAR + 256;           // row max / row sum exchange between the two column halves
// merge buffers that never alias a live tile (used when the CTA's rows fit: <= 64 rows): peers may push their
// partial rows as soon as they are done, without first waiting for this CTA to leave its tile loop
constexpr int MRG_DED_ACC = SMEM_XCH + 3 * 1024, MRG_DED_ACC_BYTES = (64 + 8) * 128 * 4,  // ns * ceil(64 / ns) <= 64 + MAX_SPLIT - 1 rows
               MRG_DED_ML = MRG_DED_ACC + MRG_DED_ACC_BYTES;
constexpr int SMEM_TOTAL = MRG_DED_ML + 1024 + 1024;  // + alignment slack
constexpr int TMEM_COLS = 512;
constexpr int TM_S0 = 0, TM_S1 = 128, TM_O = 256, TM_P0 = 384, TM_P1 = 448;  // fp32 S x2, fp32 O, bf16x2-packed P x2
constexpr int MAX_SPLIT = 8;            // KV splits per head group (merge keeps all partial rows in flight)

// ------------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
// A operand from TMEM (P, bf16 pairs packed in 32-bit columns, lane == row), B from shared memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t addr, const uint32_t *v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
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
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void st_cluster_f2(uint32_t addr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout), SWIZZLE_128B, version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // LayoutType::SWIZZLE_128B
  return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): bf16 x bf16 -> fp32, M=128, N=128
__device__ __forceinline__ constexpr uint32_t make_idesc(int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(BN >> 3) << 17) |
         ((uint32_t)(BM >> 4) << 24);
}

union Pack8 { uint4 u; __nv_bfloat16 h[8]; };
__device__ __forceinline__ float bfr(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
// x * cos + rotate_half(x) * sin for 8 elements, every product / sum rounded to bf16 (k_rope_kv_append's arithmetic,
// modeling_llama.py:167-168); `lower` = these elements lie in the first half of the head (partner enters negated)
__device__ __forceinline__ uint4 rope8(uint4 xa, uint4 xb, uint4 cs, uint4 sn, bool lower) {
  Pack8 a, b, c, s, o;
  a.u = xa; b.u = xb; c.u = cs; s.u = sn;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float x = __bfloat162float(a.h[j]);
    const float r = lower ? -__bfloat162float(b.h[j]) : __bfloat162float(b.h[j]);
    o.h[j] = __float2bfloat16_rn(bfr(x * __bfloat162float(c.h[j])) + bfr(r * __bfloat162float(s.h[j])));
  }
  return o.u;
}

struct Params {
  const __nv_bfloat16 *q;  // [max_nodes, Hq, HD]
  const unsigned long long *mask;
  pia_slots_t sl;          // request slots: blockIdx.z = slot (rows, n, P, pad and KV planes of that slot)
  int slot_planes;         // KV planes between consecutive slots' caches (0: shared cache)
  int plane0;              // first plane of the cache slot 0 addresses
  int layer, n_q_heads, n_kv_heads, np, mask_words, heads_per_cta, max_seq, n_split, tiles_per_cta;
  int groups_per_kv;       // head groups per KV head: ceil(G / heads_per_cta)
  float scale_log2;
  // fused mode (pia_tree_attn_fused_fwd): RoPE + KV append happen here.  Q and the draft nodes' K / V come straight from
  // the fused projection output, the draft keys are one extra tile built in shared memory, the cache only holds [0, P)
  int fused;
  const __nv_bfloat16 *qkv;      // [rows, (Hq + 2 Hkv) * HD]
  const __nv_bfloat16 *cos_t, *sin_t;  // [max_pos, HD / 2] bf16 (as k_rope_kv_append)
  int max_pos;
  __nv_bfloat16 *kc_layer, *vc_layer;  // this layer's [Hkv, max_seq, HD] planes of the cache slot 0 addresses
  __nv_bfloat16 *out;            // [max_nodes, Hq, HD]
  unsigned long long *dbg;       // optional per-CTA phase timestamps (pia_attn_plan_set_debug)
};

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define DBG(ev) do { if (p.dbg) p.dbg[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + (ev)] = gtime(); } while (0)

__global__ void __launch_bounds__(NTHREADS, 1)
k_tree_attn(const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v, Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *sm = smem_raw + (base - smem_u32(smem_raw));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  const uint32_t bar0 = base + SMEM_BAR;
  const uint32_t bar_kv_full = bar0, bar_kv_empty = bar0 + 8 * NSTAGE, bar_s_full = bar0 + 16 * NSTAGE,
                 bar_p_full = bar_s_full + 16, bar_o_full = bar_p_full + 16, bar_q_full = bar_o_full + 8,
                 bar_o_free = bar_q_full + 8, bar_draft = bar_o_free + 8,
                 bar_v_full = bar0 + 128;  // V tiles complete on their own barriers: QK^T starts as soon as K has landed
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(sm + SMEM_BAR + 16 * NSTAGE + 64);

  pdl_launch_dependents();
  if (tid == 0) {  // the two TMA descriptors are fetched while the barriers / TMEM are set up
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<unsigned long long>(&map_k)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<unsigned long long>(&map_v)) : "memory");
  }
  // Programmatic dependent launch: this CTA may be running while its predecessor (RoPE + KV append of the same layer)
  // still is.  What is read BEFORE griddepcontrol.wait is safe to read early: d_n / d_prefix_len / d_pad_len / the mask
  // rows were written before the first kernel of the layer chain (trie get and the previous step's accept are launched
  // without the PDL attribute, prefill meta is a stream-ordered copy), and cache rows below P were written by earlier
  // steps.  Only Q, the rows [P, P + n) of this layer's K/V planes and the output buffer depend on the predecessor: the
  // TMA producer waits before its first tile that reaches row P, the softmax warps wait before they read Q.
  const int split = blockIdx.x, group = blockIdx.y;
  const int slot = blockIdx.z;
  const int n = p.sl.d_n[slot], P = p.sl.d_prefix_len[slot];
  const int pad_len = p.sl.d_pad_len ? p.sl.d_pad_len[slot] : 0;
  if (n <= 0) return;      // idle slot: every CTA of its clusters takes this exit
  const long long row0 = (long long)slot * p.sl.rows_per_slot;  // first activation / mask row of the slot
  const int L = P + n;
  const int G = p.n_q_heads / p.n_kv_heads;
  const int hkv = group / p.groups_per_kv, jg = group % p.groups_per_kv;  // jg == 0: the KV head's first group
  const int hq0 = hkv * G + jg * p.heads_per_cta;
  const int heads_here = min(p.heads_per_cta, G - jg * p.heads_per_cta);  // 1 for the leftover head of an odd G
  // tiles: plain mode = the keys [0, L) of the cache; fused mode = the prefix tiles [0, P) of the cache + ONE draft tile
  // (the n draft keys, rotated and staged in shared memory by the softmax warps of the CTA that owns the last tile)
  const bool fused = p.fused != 0;
  const int Tp = (P + BN - 1) / BN;
  const int tiles_total = fused ? Tp + 1 : (L + BN - 1) / BN;
  // Work split decided on the device from the live length: tiles_per_cta tiles per CTA (more only when the
  // plan's split limit is reached); a single split writes the final output directly (no partials, no merge).
  const int rows_used = heads_here * p.np;               // 64 (one head, 64 nodes) or 128
  const bool ded = (rows_used + MAX_SPLIT) * HD * 4 <= MRG_DED_ACC_BYTES;
  int ns = (tiles_total + p.tiles_per_cta - 1) / p.tiles_per_cta;
  if (ns > p.n_split) ns = p.n_split;
  if (ns < 1) ns = 1;
  if (split >= ns) {
    if (ns > 1) { cluster_sync_all(); cluster_sync_all(); }
    return;
  }
  const int tps = (tiles_total + ns - 1) / ns;
  const int t0 = split * tps;
  int t1 = t0 + tps;
  if (t1 > tiles_total) t1 = tiles_total;
  const int ntile = t1 - t0;  // >= 1 for split < ns except possibly the last one
  // the CTA that owns the last tile takes the draft tile FIRST (slot 0 of the ring is free at kernel start; the order of
  // tiles does not matter to the online softmax) and its prefix tiles after it
  const bool has_draft = fused && ntile > 0 && t1 == tiles_total;
  auto tile_of = [&](int i) -> int { return has_draft ? (i == 0 ? Tp : t0 + i - 1) : t0 + i; };
  // cluster barrier A ("every CTA of the cluster is running and its merge buffers may be written"): with dedicated
  // merge buffers the arrive happens right here and the wait just before the push (it has long completed by then);
  // with aliased buffers (128-row tiles) A is a full barrier after the tile loop
  if (ns > 1 && ded) cluster_arrive();
  auto barrier_a = [&]() { if (ded) cluster_wait(); else cluster_sync_all(); };
  const int mrg_acc = ded ? MRG_DED_ACC : MRG_ACC, mrg_ml = ded ? MRG_DED_ML : MRG_ML;
  const int mrg_stride = ded ? 64 + MAX_SPLIT : 128 + MAX_SPLIT;  // slots per chunk column
  const bool is_sm_warp = warp >= 2;
  const int half = is_sm_warp ? (warp - 2) >> 2 : 0;     // which 64 columns of S / O this softmax warp owns
  const int row = ((warp & 3) << 5) | lane;              // TMEM lane == row (a warp may only touch its quadrant)
  const bool warp_active = is_sm_warp && (((warp & 3) << 5) < rows_used);
  const int hs = row / p.np, node = row % p.np;
  const bool row_live = warp_active && node < n;
  if (tid == 0) DBG(0);

  // ---- setup
  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) { mbar_init(bar_kv_full + 8 * s, 1); mbar_init(bar_kv_empty + 8 * s, 1); mbar_init(bar_v_full + 8 * s, 1); }
    mbar_init(bar_s_full, 1); mbar_init(bar_s_full + 8, 1);
    mbar_init(bar_p_full, 2 * rows_used); mbar_init(bar_p_full + 8, 2 * rows_used);
    mbar_init(bar_o_free, 2 * rows_used);
    mbar_init(bar_o_full, 1);
    mbar_init(bar_q_full, 2 * rows_used);
    mbar_init(bar_draft, NTHREADS - 64);  // all eight softmax warps stage the draft tile
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();  // warp 0 reconverges before the (warp-aligned) block barrier below (synccheck: divergent lane 0)
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (tid == 0) DBG(1);

  if (warp == 0) {
    // ================================================================ TMA producer
    if (lane == 0 && ntile > 0) {
      const int plane = p.plane0 + slot * p.slot_planes + p.layer * p.n_kv_heads + hkv;
      // rows the predecessor may still be appending start at P - or, when the slots share one cache (the chain chunks
      // of a prefill pass: chunk c's prefix holds what the same RoPE launch appends for chunks < c), at the smallest P
      int p_safe = P;
      if (p.slot_planes == 0) for (int b2 = 0; b2 < p.sl.batch; ++b2) p_safe = min(p_safe, p.sl.d_prefix_len[b2]);
      bool waited = false;
      for (int i = 0; i < ntile; ++i) {
        const int s = i % NSTAGE, ph = (i / NSTAGE) & 1;
        if (has_draft && i == 0) {  // staged by the softmax warps (bar_draft); this arrive only keeps the phases aligned
          mbar_arrive(bar_kv_full);
          mbar_arrive(bar_v_full);
          continue;
        }
        const int key0 = tile_of(i) * BN;
        // fused mode: every TMA tile lies below P (a ragged last tile drags in rows >= P that are stale or being
        // appended by this very launch - finite bf16 either way, and masked), nothing to wait for
        if (!fused && !waited && key0 + BN > p_safe) { pdl_wait(); waited = true; }
        mbar_wait(bar_kv_empty + 8 * s, ph ^ 1);
        const uint32_t kd = base + SMEM_K + s * TILE_BYTES, vd = base + SMEM_V + s * TILE_BYTES;
        mbar_expect_tx(bar_kv_full + 8 * s, TILE_BYTES);
        tma_load_3d(kd, &map_k, bar_kv_full + 8 * s, 0, key0, plane);
        tma_load_3d(kd + SUB, &map_k, bar_kv_full + 8 * s, 64, key0, plane);
        mbar_expect_tx(bar_v_full + 8 * s, TILE_BYTES);
        tma_load_3d(vd, &map_v, bar_v_full + 8 * s, 0, key0, plane);
        tma_load_3d(vd + SUB, &map_v, bar_v_full + 8 * s, 64, key0, plane);
        if (i == 0) DBG(2);
      }
    }
    __syncwarp();
    if (ns > 1) { barrier_a(); cluster_sync_all(); }
  } else if (warp == 1) {
    // ================================================================ MMA issuer (one thread)
    if (lane == 0 && ntile > 0) {
      constexpr uint32_t IDESC_QK = make_idesc(0), IDESC_PV = make_idesc(1);
      mbar_wait(bar_q_full, 0);
      auto issue_qk = [&](int i) {
        const int s = i % NSTAGE, ph = (i / NSTAGE) & 1;
        mbar_wait(bar_kv_full + 8 * s, ph);
        if (has_draft && i == 0) mbar_wait(bar_draft, 0);
        tc_fence_after();
        const uint32_t qa = base + SMEM_Q, ka = base + SMEM_K + s * TILE_BYTES;
        const uint32_t d = tmem + ((i & 1) ? TM_S1 : TM_S0);
#pragma unroll
        for (int j = 0; j < HD / 16; ++j) {  // K-major operands: 32 B per k-block inside the 128 B swizzle row
          const uint32_t off = (j >> 2) * SUB + (j & 3) * 32;
          umma_bf16(d, make_desc(qa + off, 16, 1024), make_desc(ka + off, 16, 1024), IDESC_QK, j > 0);
        }
        umma_commit(bar_s_full + 8 * (i & 1));
      };
      issue_qk(0);
      DBG(3);
      for (int i = 0; i < ntile; ++i) {
        if (i + 1 < ntile) issue_qk(i + 1);  // S is double buffered: next QK^T overlaps this tile's softmax
        const int s = i % NSTAGE;
        mbar_wait(bar_p_full + 8 * (i & 1), (i >> 1) & 1);
        if (i > 0) mbar_wait(bar_o_free, (i - 1) & 1);  // the softmax warps have folded O(i-1) into their registers
        mbar_wait(bar_v_full + 8 * s, (i / NSTAGE) & 1);
        tc_fence_after();
        const uint32_t va = base + SMEM_V + s * TILE_BYTES;
        const uint32_t pa = tmem + ((i & 1) ? TM_P1 : TM_P0);
#pragma unroll
        for (int j = 0; j < BN / 16; ++j) {
          // A = P from TMEM (16 keys = 8 packed columns per k-block); B = V, MN-major: 16 keys = 2 groups of 8 rows
          // (SBO 1024 B), d-halves 16 KB apart (LBO)
          umma_bf16_ts(tmem + TM_O, pa + j * 8, make_desc(va + j * 2048, SUB, 1024), IDESC_PV, j > 0);
        }
        umma_commit(bar_o_full);
        umma_commit(bar_kv_empty + 8 * s);
      }
      DBG(4);
    }
    __syncwarp();
    if (ns > 1) { barrier_a(); cluster_sync_all(); }
  } else if (fused && !warp_active) {
    // ================================================================ idle softmax warps of a 64-row tile, fused mode:
    // they zero the draft tile's key rows 64..127 (never live when the tile holds 64 nodes)
    if (has_draft) {
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        const uint32_t off = half * SUB + row * 128 + ((ch ^ (row & 7)) << 4);
        *reinterpret_cast<uint4 *>(sm + SMEM_K + off) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4 *>(sm + SMEM_V + off) = make_uint4(0, 0, 0, 0);
      }
      fence_async_smem();
      mbar_arrive(bar_draft);
    }
    if (ns > 1) { barrier_a(); cluster_sync_all(); }
  } else if (warp_active) {
    // ================================================================ softmax + accumulate
    // two threads per row: `half` selects 64 of the 128 S columns (keys) and 64 of the 128 O columns (head dim)
    pdl_wait();  // Q (or, fused, the projection output) below is the predecessor's output
    unsigned long long mrow[2] = {0ull, 0ull};
    if (row_live) {
      mrow[0] = p.mask[(row0 + node) * p.mask_words];
      if (p.mask_words > 1) mrow[1] = p.mask[(row0 + node) * p.mask_words + 1];
    }
    if (!fused) {
      uint4 qv[8];  // Q row -> shared memory (UMMA K-major SWIZZLE_128B); each half loads one 64-wide d sub-tile
      const bool have = hs < heads_here && node < n;
      const uint4 *src = reinterpret_cast<const uint4 *>(p.q + ((row0 + node) * p.n_q_heads + hq0 + hs) * HD) + half * 8;
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) qv[ch] = have ? src[ch] : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int ch = 0; ch < 8; ++ch)
        *reinterpret_cast<uint4 *>(sm + SMEM_Q + half * SUB + row * 128 + ((ch ^ (row & 7)) << 4)) = qv[ch];
      fence_async_smem();
      mbar_arrive(bar_q_full);
    } else {
      // RoPE at the node's position = rowsum(mask) - 1 (modeling_llama.py:587): visible prefix + tree depth
      int pos = (P > pad_len ? P - pad_len : 0) + __popcll(mrow[0]) + __popcll(mrow[1]) - 1;
      pos = pos < 0 ? 0 : (pos >= p.max_pos ? p.max_pos - 1 : pos);
      const uint4 *cs = reinterpret_cast<const uint4 *>(p.cos_t + (long long)pos * (HD / 2));
      const uint4 *sn = reinterpret_cast<const uint4 *>(p.sin_t + (long long)pos * (HD / 2));
      const long long row_elems = (long long)(p.n_q_heads + 2 * p.n_kv_heads) * HD;
      const __nv_bfloat16 *xr = p.qkv + (row0 + node) * row_elems;
      const bool have = hs < heads_here && node < n;
      // All global loads of a batch are issued (read-only path: the compiler may not move plain loads across the shared
      // memory stores in between, and eight dependent load rounds of ~0.7 us each would serialise the prologue) before
      // the first value is used; four 16-byte chunks per batch bound the registers.
      {  // Q: rotate this thread's 64-wide half (the other half of the head is the rotation partner)
        const uint4 *qa = reinterpret_cast<const uint4 *>(xr + (long long)(hq0 + hs) * HD) + half * 8;
        const uint4 *qb = reinterpret_cast<const uint4 *>(xr + (long long)(hq0 + hs) * HD) + (half ^ 1) * 8;
#pragma unroll
        for (int b4 = 0; b4 < 2; ++b4) {
          uint4 ra[4], rb[4], rc[4], rs[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int ch = b4 * 4 + j;
            if (have) { ra[j] = __ldg(qa + ch); rb[j] = __ldg(qb + ch); rc[j] = __ldg(cs + ch); rs[j] = __ldg(sn + ch); }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int ch = b4 * 4 + j;
            const uint4 o = have ? rope8(ra[j], rb[j], rc[j], rs[j], half == 0) : make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4 *>(sm + SMEM_Q + half * SUB + row * 128 + ((ch ^ (row & 7)) << 4)) = o;
          }
        }
        fence_async_smem();
        mbar_arrive(bar_q_full);
      }
      if (has_draft) {
        // the draft tile (ring slot 0): key row r = draft node r, K rotated at r's position, V as projected; rows that
        // hold no node are zero.  The threads of the tile's first head (hs == 0: row == node) own the key rows; one CTA
        // per KV head also appends the rows to the cache for the steps to come (pretrained_model.py: the reference's
        // torch.cat of past and new K/V, modeling_llama.py:265-268)
        const bool key_row = hs == 0 && node < n;
        const bool writer = jg == 0;
        const uint4 *ka = reinterpret_cast<const uint4 *>(xr + (long long)(p.n_q_heads + hkv) * HD) + half * 8;
        const uint4 *kb = reinterpret_cast<const uint4 *>(xr + (long long)(p.n_q_heads + hkv) * HD) + (half ^ 1) * 8;
        const uint4 *va = reinterpret_cast<const uint4 *>(xr + (long long)(p.n_q_heads + p.n_kv_heads + hkv) * HD) + half * 8;
        const long long crow = (long long)slot * p.sl.kv_slot_stride + ((long long)hkv * p.max_seq + P + node) * HD + half * 64;
        uint4 *kdst = reinterpret_cast<uint4 *>(p.kc_layer + crow), *vdst = reinterpret_cast<uint4 *>(p.vc_layer + crow);
#pragma unroll
        for (int b4 = 0; b4 < 2; ++b4) {
          uint4 ra[4], rb[4], rc[4], rs[4], rv[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int ch = b4 * 4 + j;
            if (key_row) {
              ra[j] = __ldg(ka + ch); rb[j] = __ldg(kb + ch); rc[j] = __ldg(cs + ch); rs[j] = __ldg(sn + ch);
              rv[j] = __ldg(va + ch);
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int ch = b4 * 4 + j;
            const uint32_t off = half * SUB + row * 128 + ((ch ^ (row & 7)) << 4);
            uint4 ko = make_uint4(0, 0, 0, 0), vo = make_uint4(0, 0, 0, 0);
            if (key_row) { ko = rope8(ra[j], rb[j], rc[j], rs[j], half == 0); vo = rv[j]; }
            *reinterpret_cast<uint4 *>(sm + SMEM_K + off) = ko;
            *reinterpret_cast<uint4 *>(sm + SMEM_V + off) = vo;
            if (key_row && writer) { kdst[ch] = ko; vdst[ch] = vo; }
          }
        }
        fence_async_smem();
        mbar_arrive(bar_draft);
      }
    }
    if (row == 0 && half == 0) DBG(5);
    const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
    const int pair_bar = 1 + (warp & 3);  // named barrier shared by the two warps of this lane quadrant
    float acc[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) acc[j] = 0.f;
    float m_run = -INFINITY, l_run = 0.f, alpha_prev = 0.f;
    uint32_t sv[64];
    for (int i = 0; i < ntile; ++i) {
      const int tl = tile_of(i);
      const bool is_draft = fused && tl == Tp;
      const int key0 = tl * BN + half * 64;
      const uint32_t s_addr = tmem + lane_addr + ((i & 1) ? TM_S1 : TM_S0) + half * 64;
      mbar_wait(bar_s_full + 8 * (i & 1), (i >> 1) & 1);
      tc_fence_after();
      if (row == 0 && half == 0 && i == 0) DBG(6);
      tmem_ld32(s_addr, sv);
      tmem_ld32(s_addr + 32, sv + 32);
      tmem_ld_wait();
      // 32-bit visibility word of keys [kb, kb+32): prefix keys [pad_len, P) are visible to every row, the n draft
      // keys follow the row's ancestor bits (bits beyond the live nodes are never set in the trie's mask rows)
      const bool all_visible = !is_draft && (tl * BN >= pad_len) && (tl * BN + BN <= P);
      auto vis32 = [&](int kb) -> uint32_t {
        if (all_visible) return 0xffffffffu;
        if (is_draft) {  // key kb - Tp * BN is draft node j0: visible iff it is an ancestor (or the node itself)
          const int j0 = kb - Tp * BN;
          if (j0 < 64) {
            unsigned long long x = mrow[0] >> j0;
            if (j0 > 32) x |= mrow[1] << (64 - j0);
            return (uint32_t)x;
          }
          return (uint32_t)(mrow[1] >> (j0 - 64));
        }
        uint32_t m = 0;
        const int lo = kb < pad_len ? pad_len : kb;
        const int hi = kb + 32 < P ? kb + 32 : P;
        if (hi > lo) m = (hi - lo >= 32 ? 0xffffffffu : ((1u << (hi - lo)) - 1u)) << (lo - kb);
        const int j0 = kb - P;
        if (!fused && j0 + 32 > 0 && j0 < n) {
          uint32_t d;
          if (j0 < 0) d = (uint32_t)(mrow[0] << (-j0));
          else if (j0 < 64) {
            unsigned long long x = mrow[0] >> j0;
            if (j0 > 32) x |= mrow[1] << (64 - j0);
            d = (uint32_t)x;
          } else d = (uint32_t)(mrow[1] >> (j0 - 64));
          m |= d;
        }
        return m;
      };
      const uint32_t vm0 = vis32(key0), vm1 = vis32(key0 + 32);
      if ((vm0 & vm1) != 0xffffffffu) {  // tree / padded / ragged tile: hidden keys -> -inf once, then the dense code
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if (!((vm0 >> j) & 1u)) sv[j] = 0xff800000u;
          if (!((vm1 >> j) & 1u)) sv[32 + j] = 0xff800000u;
        }
      }
      // four independent chains (a single 64-long fmaxf / FADD chain is ~250 cycles of pure latency per tile)
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
      for (int j = 0; j < 64; j += 4) {
        mx0 = fmaxf(mx0, __uint_as_float(sv[j])); mx1 = fmaxf(mx1, __uint_as_float(sv[j + 1]));
        mx2 = fmaxf(mx2, __uint_as_float(sv[j + 2])); mx3 = fmaxf(mx3, __uint_as_float(sv[j + 3]));
      }
      const float m_half = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
      // row max across the two halves (double-buffered exchange slot, one named barrier per quadrant pair)
      float *xm = reinterpret_cast<float *>(sm + SMEM_XCH) + (i & 1) * 256;
      xm[half * 128 + row] = m_half;
      asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
      const float m_tile = fmaxf(m_half, xm[(half ^ 1) * 128 + row]);
      const float m_new = fmaxf(m_run, m_tile * p.scale_log2);
      const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
      const float alpha = (m_run == -INFINITY) ? 0.f : ex2(m_run - m_use);
      // p = exp2(s*scale - m) -> bf16 pairs -> TMEM (A operand of the PV MMA: lane = row, one 32-bit column per key
      // pair; this half owns columns [32*half, 32*half+32)), row sum
      float ls[4] = {0.f, 0.f, 0.f, 0.f};
      uint32_t pk[32];
#pragma unroll
      for (int e = 0; e < 32; ++e) {  // ex2(-inf) = 0 for the hidden keys (m_use is finite)
        const float p0 = ex2(__uint_as_float(sv[2 * e]) * p.scale_log2 - m_use);
        const float p1 = ex2(__uint_as_float(sv[2 * e + 1]) * p.scale_log2 - m_use);
        const __nv_bfloat162 b = __floats2bfloat162_rn(p0, p1);
        // the row sum uses the bf16-rounded probabilities, i.e. exactly what the PV MMA consumes
        ls[e & 3] += __bfloat162float(b.x) + __bfloat162float(b.y);
        pk[e] = *reinterpret_cast<const uint32_t *>(&b);
      }
      const float l_tile = (ls[0] + ls[1]) + (ls[2] + ls[3]);
      // P buffer (i & 1) is free: PV(i-2) completed before o_full(i-2), which this thread observed in iteration i-1
      tmem_st32(tmem + lane_addr + ((i & 1) ? TM_P1 : TM_P0) + half * 32, pk);
      tmem_st_wait();
      l_run = l_run * alpha + l_tile;
      m_run = m_new;
      tc_fence_before();    // orders the tcgen05.ld of S and the tcgen05.st of P before the issuer's next MMAs
      mbar_arrive(bar_p_full + 8 * (i & 1));
      if (row == 0 && half == 0 && i == 0) DBG(7);
      // fold the PREVIOUS tile's PV into the register accumulator (this half's 64 head-dim columns) while the tensor
      // core works on PV(i) / QK(i+1): O(i-1) was computed against m_{i-1}, so the older sum is rescaled by
      // alpha_{i-1} = 2^(m_{i-2} - m_{i-1})
      if (i > 0) {
        mbar_wait(bar_o_full, (i - 1) & 1);
        tc_fence_after();
        tmem_ld32(tmem + lane_addr + TM_O + half * 64, sv);
        tmem_ld32(tmem + lane_addr + TM_O + half * 64 + 32, sv + 32);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(bar_o_free);
#pragma unroll
        for (int j = 0; j < 64; ++j) acc[j] = acc[j] * alpha_prev + __uint_as_float(sv[j]);
      }
      alpha_prev = alpha;
    }
    if (ntile > 0) {
      mbar_wait(bar_o_full, (ntile - 1) & 1);
      tc_fence_after();
      if (row == 0 && half == 0) DBG(8);
      tmem_ld32(tmem + lane_addr + TM_O + half * 64, sv);
      tmem_ld32(tmem + lane_addr + TM_O + half * 64 + 32, sv + 32);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 64; ++j) acc[j] = acc[j] * alpha_prev + __uint_as_float(sv[j]);
      tc_fence_before();
    }
    if (row == 0 && half == 0) DBG(9);
    // total row sum = both halves (same running max, so the partial sums just add)
    {
      float *xl = reinterpret_cast<float *>(sm + SMEM_XCH) + 512;
      xl[half * 128 + row] = l_run;
      asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
      l_run += xl[(half ^ 1) * 128 + row];
    }
    if (ns == 1) {
      // single split: normalise and write this half of the final bf16 row
      if (row_live) {
        const float inv = l_run > 0.f ? 1.f / l_run : 0.f;
        uint4 *dst = reinterpret_cast<uint4 *>(p.out + ((row0 + node) * p.n_q_heads + hq0 + hs) * HD + half * 64);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          __nv_bfloat162 b0 = __floats2bfloat162_rn(acc[8 * j] * inv, acc[8 * j + 1] * inv);
          __nv_bfloat162 b1 = __floats2bfloat162_rn(acc[8 * j + 2] * inv, acc[8 * j + 3] * inv);
          __nv_bfloat162 b2 = __floats2bfloat162_rn(acc[8 * j + 4] * inv, acc[8 * j + 5] * inv);
          __nv_bfloat162 b3 = __floats2bfloat162_rn(acc[8 * j + 6] * inv, acc[8 * j + 7] * inv);
          dst[j] = make_uint4(*reinterpret_cast<uint32_t *>(&b0), *reinterpret_cast<uint32_t *>(&b1),
                              *reinterpret_cast<uint32_t *>(&b2), *reinterpret_cast<uint32_t *>(&b3));
        }
      }
    } else {
      // several splits: the ns CTAs of this head group form one thread-block cluster.  After everyone has left its
      // tile loop (barrier A: the Q/P/KV tiles of every CTA are dead) each thread pushes its row half - acc, and the
      // row's (m, l) - straight into the shared memory of the CTA that owns that row's slice (DSMEM), barrier B,
      // and every CTA combines its slice locally: no workspace round trip through L2, no serial last-arriver merge.
      barrier_a();
      if (row == 0 && half == 0) DBG(14);
      const int RS = (rows_used + ns - 1) / ns;       // rows per owner CTA
      const int owner = row / RS, rl = row % RS;
      if (row_live) {
        // partial rows are stored chunk-major ([32 float4 chunks][slot]) so that the lanes of a warp (= consecutive
        // rows) write consecutive 16-byte words of the owner's buffer with every store instruction
        const uint32_t dst = map_to_cta(base + mrg_acc + (uint32_t)((half * 16) * mrg_stride + split * RS + rl) * 16, owner);
#pragma unroll
        for (int j = 0; j < 16; ++j)
          st_cluster_f4(dst + (uint32_t)(j * mrg_stride) * 16, acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
        if (half == 0) st_cluster_f2(map_to_cta(base + mrg_ml + (uint32_t)(split * RS + rl) * 8, owner), m_run, l_run);
      }
      __syncwarp();  // the live-row branch above diverges; the cluster barrier is warp-aligned
      if (row == 0 && half == 0) DBG(15);
      cluster_sync_all();
    }
    if (row == 0 && half == 0) DBG(10);
  } else {
    if (ns > 1) { barrier_a(); cluster_sync_all(); }  // idle softmax warps (rows 64..127 of a one-head tile)
  }
  if (ns > 1) {
    // combine this CTA's row slice: out[r][:] = sum_i acc_i 2^(m_i - M) / sum_i l_i 2^(m_i - M), all operands local
    const int RS = (rows_used + ns - 1) / ns;
    const float4 *macc = reinterpret_cast<const float4 *>(sm + mrg_acc);
    const float2 *mml = reinterpret_cast<const float2 *>(sm + mrg_ml);
    const int items = RS * (HD / 4);
    // RS and np are powers of two in every configuration but ragged ones: shifts instead of four integer divisions per
    // item, and all ns partials of an item are loaded before the first is used (the loop over a runtime ns was a chain
    // of dependent shared-memory round trips: 1.7 us for 512 items on 320 threads)
    const bool pow2 = (RS & (RS - 1)) == 0 && (p.np & (p.np - 1)) == 0;
    const int rs_sh = 31 - __clz(RS), np_sh = 31 - __clz(p.np);
    for (int it = tid; it < items; it += NTHREADS) {
      const int rl = pow2 ? (it & (RS - 1)) : it % RS, c4 = pow2 ? (it >> rs_sh) : it / RS;
      const int r = split * RS + rl;
      if (r >= rows_used) continue;
      const int rh = pow2 ? (r >> np_sh) : r / p.np, rn = pow2 ? (r & (p.np - 1)) : r % p.np;
      if (rn >= n) continue;
      float2 ml[MAX_SPLIT];
      float4 a4[MAX_SPLIT];
#pragma unroll
      for (int i = 0; i < MAX_SPLIT; ++i) {
        if (i < ns) { ml[i] = mml[i * RS + rl]; a4[i] = macc[c4 * mrg_stride + i * RS + rl]; }
        else { ml[i] = make_float2(-INFINITY, 0.f); a4[i] = make_float4(0.f, 0.f, 0.f, 0.f); }
      }
      float M = -INFINITY;
#pragma unroll
      for (int i = 0; i < MAX_SPLIT; ++i) M = fmaxf(M, ml[i].x);
      float den = 0.f;
      float4 o4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < MAX_SPLIT; ++i) {
        const float w = ml[i].x == -INFINITY ? 0.f : ex2(ml[i].x - M);
        den += ml[i].y * w;
        o4.x += a4[i].x * w; o4.y += a4[i].y * w; o4.z += a4[i].z * w; o4.w += a4[i].w * w;
      }
      const float inv = den > 0.f ? 1.f / den : 0.f;
      __nv_bfloat162 b0 = __floats2bfloat162_rn(o4.x * inv, o4.y * inv), b1 = __floats2bfloat162_rn(o4.z * inv, o4.w * inv);
      reinterpret_cast<uint2 *>(p.out + ((row0 + rn) * p.n_q_heads + hq0 + rh) * HD)[c4] =
          make_uint2(*reinterpret_cast<uint32_t *>(&b0), *reinterpret_cast<uint32_t *>(&b1));
    }
  }
  if (tid == 0) DBG(12);
  // every tcgen05 access of this CTA is complete (the softmax warps observed the last o_full): release TMEM
  tc_fence_before();
  __syncthreads();
  if (tid == 0) DBG(13);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS));
  }
  if (tid == 0) DBG(11);
}

}  // namespace attn
}  // namespace pia

// =====================================================================================================
using namespace pia;
using namespace pia::attn;

struct pia_attn_plan {
  pia_attn_config_t cfg;
  CUtensorMap map_k, map_v;
  int heads_per_cta, n_groups, n_split, mask_words, tiles_per_cta;
  unsigned long long *dbg;
  __nv_bfloat16 *k_base, *v_base;  // the caches the TMA maps describe (fused mode appends the draft rows itself)
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int encode_kv_map(CUtensorMap *m, void *base, const pia_attn_config_t &c) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    void *ptr = nullptr;
    PIA_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres));
    PIA_REQUIRE(ptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available in this driver");
    fn = (EncodeTiledFn)ptr;
  }
  // cache viewed as [planes = n_layers * n_kv_heads][max_seq][head_dim] bf16, box = 64 d x 128 keys x 1 plane
  cuuint64_t dims[3] = {(cuuint64_t)c.head_dim, (cuuint64_t)c.max_seq,
                        (cuuint64_t)(c.n_slots > 0 ? c.n_slots : 1) * c.n_layers * c.n_kv_heads};
  cuuint64_t strides[2] = {(cuuint64_t)c.head_dim * 2, (cuuint64_t)c.max_seq * c.head_dim * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)BN, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return PIA_ERR_CUDA; }
  return PIA_OK;
}

extern "C" int pia_attn_plan_create(const pia_attn_config_t *cfg, void *d_k_cache, void *d_v_cache,
                                    pia_attn_plan_t **out) {
  PIA_REQUIRE(cfg && d_k_cache && d_v_cache && out, "null argument");
  if (cfg->head_dim != HD) { set_error("head_dim %d: only 128 is built in this round", cfg->head_dim); return PIA_ERR_UNSUPPORTED; }
  PIA_REQUIRE(cfg->max_nodes == 64 || cfg->max_nodes == 128, "max_nodes must be 64 or 128");
  PIA_REQUIRE(cfg->n_q_heads > 0 && cfg->n_kv_heads > 0 && cfg->n_q_heads % cfg->n_kv_heads == 0, "bad head counts");
  PIA_REQUIRE(cfg->max_seq > 0 && cfg->n_layers > 0, "bad cache shape");
  PIA_REQUIRE((reinterpret_cast<uintptr_t>(d_k_cache) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_v_cache) & 15) == 0, "cache must be 16-byte aligned");
  pia_attn_plan *p = new (std::nothrow) pia_attn_plan();
  PIA_REQUIRE(p, "out of host memory");
  p->cfg = *cfg;
  const int G = cfg->n_q_heads / cfg->n_kv_heads;
  // 64-node drafts under GQA: two query heads of one KV head per CTA; an odd G leaves one single-head group per KV
  // head.  PIA_ATTN_HEAD_PAIRS=0 keeps one head per CTA for odd G (A/B measurement of the two layouts)
  bool pairs = G > 1;
  const char *e = getenv("PIA_ATTN_HEAD_PAIRS");
  if (pairs && G % 2 == 1 && e) pairs = atoi(e) != 0;
  p->heads_per_cta = (cfg->max_nodes == 64 && pairs) ? 2 : 1;
  p->n_groups = cfg->n_kv_heads * ((G + p->heads_per_cta - 1) / p->heads_per_cta);
  p->mask_words = cfg->max_nodes / 64;
  int n_sm = 148, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  const int max_tiles = (cfg->max_seq + BN - 1) / BN;
  // one wave: the split CTAs of a head group are one thread-block cluster, so idle splits still occupy an SM each
  int ns = cfg->kv_split_max > 0 ? cfg->kv_split_max : n_sm / p->n_groups;
  if (ns > max_tiles) ns = max_tiles;
  if (ns < 1) ns = 1;
  if (ns > MAX_SPLIT) ns = MAX_SPLIT;
  p->n_split = ns;
  p->tiles_per_cta = 1;
  if (const char *e = getenv("PIA_ATTN_TILES_PER_CTA")) { int v = atoi(e); if (v >= 1 && v <= 64) p->tiles_per_cta = v; }
  int rc = encode_kv_map(&p->map_k, d_k_cache, *cfg);
  if (rc == PIA_OK) rc = encode_kv_map(&p->map_v, d_v_cache, *cfg);
  if (rc == PIA_OK) {
    cudaError_t e = cudaFuncSetAttribute(k_tree_attn, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TOTAL);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); rc = PIA_ERR_CUDA; }
  }
  p->dbg = nullptr;
  p->k_base = (__nv_bfloat16 *)d_k_cache; p->v_base = (__nv_bfloat16 *)d_v_cache;
  if (rc != PIA_OK) { delete p; return rc; }
  *out = p;
  return PIA_OK;
}

extern "C" int pia_attn_plan_set_debug(pia_attn_plan_t *p, void *d_timestamps) {
  PIA_REQUIRE(p, "null plan");
  p->dbg = (unsigned long long *)d_timestamps;
  return PIA_OK;
}
extern "C" int pia_attn_plan_grid(const pia_attn_plan_t *p, int *n_split, int *n_groups) {
  PIA_REQUIRE(p && n_split && n_groups, "null argument");
  *n_split = p->n_split; *n_groups = p->n_groups;
  return PIA_OK;
}

extern "C" int pia_attn_plan_destroy(pia_attn_plan_t *p) {
  if (p) delete p;
  return PIA_OK;
}

static int attn_launch(pia_attn_plan_t *p, int layer, const void *d_q, const void *d_qkv, const void *d_cos,
                       const void *d_sin, int max_pos, const uint64_t *d_mask, const pia_slots_t *slots, float scale_mul,
                       void *d_out, void *stream) {
  const bool fused = d_qkv != nullptr;
  PIA_REQUIRE(p && (d_q || d_qkv) && d_mask && slots && slots->d_n && slots->d_prefix_len && d_out, "null argument");
  PIA_REQUIRE(layer >= 0 && layer < p->cfg.n_layers, "layer %d outside [0,%d)", layer, p->cfg.n_layers);
  PIA_REQUIRE(slots->batch >= 1 && slots->batch <= 65535 && slots->rows_per_slot >= 1 &&
                  slots->rows_per_slot <= p->cfg.max_nodes, "bad slot table");
  const long long cache_elems = (long long)p->cfg.n_layers * p->cfg.n_kv_heads * p->cfg.max_seq * p->cfg.head_dim;
  const int plan_slots = p->cfg.n_slots > 0 ? p->cfg.n_slots : 1;
  PIA_REQUIRE(slots->kv_first_slot >= 0 && slots->kv_first_slot < plan_slots, "kv_first_slot outside the plan's caches");
  PIA_REQUIRE(slots->kv_slot_stride == 0 || (slots->kv_slot_stride == cache_elems &&
                                              slots->kv_first_slot + slots->batch <= plan_slots),
              "kv_slot_stride must be 0 or one whole cache, and the plan must span `batch` caches");
  // fused mode appends the draft rows of every slot from inside the launch: slots that share one cache (the chain
  // chunks of a prefill pass) would read rows their neighbours are still writing - they take the two-kernel path
  PIA_REQUIRE(!fused || slots->batch == 1 || slots->kv_slot_stride != 0,
              "the fused RoPE / KV-append attention needs one cache per slot");
  PIA_REQUIRE(!fused || (d_cos && d_sin && max_pos > 0), "fused mode needs the RoPE tables");
  Params a;
  a.q = (const __nv_bfloat16 *)d_q;
  a.mask = (const unsigned long long *)d_mask;
  a.sl = *slots;
  a.slot_planes = slots->kv_slot_stride ? p->cfg.n_layers * p->cfg.n_kv_heads : 0;
  a.plane0 = slots->kv_first_slot * p->cfg.n_layers * p->cfg.n_kv_heads;
  a.layer = layer; a.n_q_heads = p->cfg.n_q_heads; a.n_kv_heads = p->cfg.n_kv_heads; a.np = p->cfg.max_nodes;
  a.mask_words = p->mask_words; a.heads_per_cta = p->heads_per_cta; a.max_seq = p->cfg.max_seq;
  a.groups_per_kv = p->n_groups / p->cfg.n_kv_heads;
  // KV splits per (slot, head group): one wave of CTAs over ALL slots - a batch of requests brings its own parallelism,
  // so each cluster shrinks (8 slots x 32 head groups already cover the SMs without any split)
  int ns = p->n_split / slots->batch;
  if (ns < 1) ns = 1;
  a.n_split = ns; a.tiles_per_cta = p->tiles_per_cta;
  a.out = (__nv_bfloat16 *)d_out; a.dbg = p->dbg;
  a.fused = fused ? 1 : 0;
  a.qkv = (const __nv_bfloat16 *)d_qkv; a.cos_t = (const __nv_bfloat16 *)d_cos; a.sin_t = (const __nv_bfloat16 *)d_sin;
  a.max_pos = max_pos;
  const long long layer_off = ((long long)slots->kv_first_slot * p->cfg.n_layers + layer) * p->cfg.n_kv_heads *
                              (long long)p->cfg.max_seq * p->cfg.head_dim;
  a.kc_layer = p->k_base + layer_off; a.vc_layer = p->v_base + layer_off;
  a.scale_log2 = scale_mul * 1.4426950408889634f / sqrtf((float)HD);
  cudaStream_t s = (cudaStream_t)stream;
  PIA_CUDA_CHECK(launch_kernel_cluster(k_tree_attn, dim3(ns, p->n_groups, slots->batch), dim3(NTHREADS), SMEM_TOTAL, s,
                                       (unsigned)ns, p->map_k, p->map_v, a));
  count_launch();
  return PIA_OK;
}

extern "C" int pia_tree_attn_fwd(pia_attn_plan_t *p, int layer, const void *d_q, const uint64_t *d_mask,
                                 const pia_slots_t *slots, float scale_mul, void *d_out, void *stream) {
  PIA_REQUIRE(d_q, "null q");
  return attn_launch(p, layer, d_q, nullptr, nullptr, nullptr, 0, d_mask, slots, scale_mul, d_out, stream);
}

extern "C" int pia_tree_attn_fused_fwd(pia_attn_plan_t *p, int layer, const void *d_qkv, const void *d_cos,
                                       const void *d_sin, int max_pos, const uint64_t *d_mask, const pia_slots_t *slots,
                                       float scale_mul, void *d_out, void *stream) {
  PIA_REQUIRE(d_qkv, "null qkv");
  return attn_launch(p, layer, nullptr, d_qkv, d_cos, d_sin, max_pos, d_mask, slots, scale_mul, d_out, stream);
}
