// Level-3 (C = 256, 16 heads of 16 channels) multi-frame window attention half with the projections on tcgen05.
//
// bde_window_attention_fused for c = 256 with the projection: one CTA per window does window gather + LayerNorm + q / k / v
// projections + softmax(q k^T + relative-position bias) v + output projection + window_reverse + shortcut
// (model/BDE2VID/DTransformer.py:164-207, 254-299).  The q / k / v and output projections -- 70 % of the cycles of the
// earlier all-mma.sync kernel as latency-bound slices -- are tcgen05 MMAs with the operands read once from shared memory and
// the accumulators in TMEM.  They are computed TRANSPOSED so that the weights fill the M = 128 rows of the instruction
// exactly and the window's tokens are the N dimension (160 of 160 columns used, instead of 147 of 256 rows):
//
//   [K^T ; V^T] (128 x XROWS)  = [Wk(hg) ; Wv(hg)] (128 x 256) . Xln^T      per head group hg (64 channels = 4 heads)
//   Q^T (256 x 64)             = Wq (2 tiles of 128 x 256) . Xln_q^T        once (the query frame's tokens come first in Xln)
//   P^T (256 x 64)             = Wproj (2 tiles) . O^T                      after the last head group
//
//   A = weight tiles, streamed by TMA (SWIZZLE_128B) through a 3-stage ring of [128 rows x 64 K] tiles;
//   B = the LayerNorm'ed tokens / the attention output, written by the worker warps straight into the 128B-swizzled
//       K-major layout (one [rows x 64] slab per K block);  D = TMEM: Q^T / P^T 128 columns, K^T|V^T double buffered 2 x 160.
//
// Warps 0-15 (workers): gather + LayerNorm, then per head group: TMEM -> (+bias) -> bf16 / fp16 [token][channel] tiles,
// and the register-resident softmax attention on mma.sync exactly as before (warp = head x 16-row query tile), finally
// the P^T epilogue (thread = output channel: 128-byte coalesced read-modify-write of x per token).
// Warp 16: one elected lane issues every TMA load and every tcgen05.mma; it runs up to two head groups ahead of the
// workers, so the projections of head group hg + 1 overlap the attention of head group hg.
#include <stdlib.h>
#include <string.h>

#include "tc_common.cuh"

namespace bde {
namespace tc {
namespace {

constexpr int kTok = 49, kRel = 169;
constexpr int kWorkers = 512, kThreadsT = kWorkers + 32;
constexpr int kStageBytes = 16384, kStages = 3;

struct TcAttnParams {
  const float* frames[8];
  const int* tok_map;
  const float* bqkv;             // [768] q | k | v (LayerNorm beta / q scale folded in)
  const float* tbl;              // [heads, D * 169]
  const float* bproj;            // [256]
  float* xs;                     // fp32 [P, 256]
  int n_win, D, q_slot;
  long long* dbg;
};

template <int NT>
struct TCfg {
  static constexpr int C = 256, HD = 16, HG = 4, NHG = 4;
  static constexpr int PQ = 72;
  static constexpr int KSTEPS = (NT + 1) / 2;
  static constexpr int XROWS = KSTEPS * 16;       // token rows staged = N of the K^T | V^T MMAs (64 / 112 / 160)
  static constexpr int NKEY = NT * 8;
  static constexpr int DMAX = NT <= 7 ? 1 : (NT <= 13 ? 2 : 3);
  static constexpr int XN_SLAB = XROWS * 128;     // one K block of the LayerNorm'ed tokens (multiple of 1024)
  static constexpr int OFF_XN = 0;
  static constexpr int OFF_RING = OFF_XN + 4 * XN_SLAB;
  static constexpr int OFF_O = OFF_RING + kStages * kStageBytes;        // 4 slabs x [64 rows x 128 B]
  static constexpr int OFF_Q = OFF_O + 4 * 64 * 128;
  static constexpr int PT = XROWS + 8;            // token pitch of the channel-major k / v tiles [64][PT]
  static constexpr int OFF_K = OFF_Q + 64 * PQ * 2;
  static constexpr int OFF_V = OFF_K + 64 * PT * 2;
  static constexpr int OFF_TBL = OFF_V + 64 * PT * 2;
  static constexpr int OFF_COFF = OFF_TBL + HG * DMAX * kRel * 4;
  static constexpr int OFF_ROFF = OFF_COFF + NKEY * 4;
  static constexpr int OFF_PIX = OFF_ROFF + 256;
  static constexpr int OFF_BIAS = OFF_PIX + 256;                      // float [768] q | k | v biases
  static constexpr int OFF_BAR = OFF_BIAS + 768 * 4;
  static constexpr int SMEM = OFF_BAR + 256 + 1024;
  static constexpr int TM_Q = 0, TM_KV = 128, TM_P = 288;         // Q^T 2 x 64 | K^T|V^T 160 (single buffer) | P^T 2 x 64 columns
  static_assert(XN_SLAB % 1024 == 0, "token slabs must keep the swizzle atoms aligned");
  static_assert(OFF_RING % 1024 == 0 && OFF_O % 1024 == 0, "operand regions must be 1024-byte aligned");
  static_assert(SMEM <= 232448, "shared memory budget");
};

__host__ __device__ constexpr uint32_t idesc_mn(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
// Worker-side wait: ONE lane per warp polls (with a short sleep between probes), the rest of the warp parks on __syncwarp.
// 512 threads spinning on mbarrier.try_wait slowed both the TMA loads and the tcgen05 MMAs of the 17th warp several-fold
// (measured with the in-kernel timeline: 1.3-1.7 K cycles per 16 KB stage instead of ~400).
__device__ __forceinline__ void mbar_wait_polite(uint32_t bar, uint32_t parity, int lane) {
  if (lane == 0) {
    uint32_t done = 0;
    while (true) {
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t"
          "}"
          : "=r"(done)
          : "r"(bar), "r"(parity)
          : "memory");
      if (done) break;
      __nanosleep(40);
    }
  }
  __syncwarp();
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void worker_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kWorkers) : "memory"); }

// ---- mma.sync pieces of the attention core (as in attn_fused.cu) -------------------------------------------------------
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma16816_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x2_trans(uint32_t& r0, uint32_t& r1, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ void cpa16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
// one MUFU op each (see attn_fused.cu: the IEEE forms add a Newton step, a range check and a slow-path branch)
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ uint32_t pack2_h(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// v tiles: values beyond the fp16 range saturate at +-65504 instead of becoming inf
__device__ __forceinline__ uint32_t pack2_hs(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ void ldsm_x2(uint32_t& r0, uint32_t& r1, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
// k / v tiles of a head group stay CHANNEL-major, [64 channels][PT tokens] -- the layout the transposed projections leave in
// TMEM (lane = channel, column = token): a thread packs 8 consecutive tokens of its channel into ONE 16-byte store (the
// token-major tiles cost a convert + a 2-byte store per element: 15 % of the kernel's instructions, ncu source view), and the
// B fragments of both products come out of ldmatrix: .trans for q k^T (rows = 16 channels of the head, 8 tokens each), plain
// for P v (rows = 8 channels, 2 x 8 tokens).  Token pitch Cfg::PT = XROWS + 8 (336-byte rows for D = 3): 16-byte aligned and
// conflict-free for 8-row ldmatrix phases.
__device__ __forceinline__ uint32_t ex2_h2(float lo, float hi) {
  float a, b;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(a) : "f"(lo));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(b) : "f"(hi));
  return pack2_h(a, b);
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint2 lds_u64(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}

// Stage schedule of the MMA warp (32 stages of one [128 rows x 64 K] weight tile each):
//   0-3 Q tile 0 | 4-7 K|V hg 0 | 8-11 Q tile 1 | 12-15 K|V hg 1 | 16-17 proj(hg 0) | 18-21 K|V hg 2 | 22-23 proj(hg 1) |
//   24-27 K|V hg 3 | 28-29 proj(hg 2) | 30-31 proj(hg 3)
// kind: 0 = Q tile idx (K block kb), 1 = K|V of head group idx (K block kb), 2 = proj tile kb of K block (= head group) idx
struct StageInfo {
  int kind, idx, kb, first, last;   // first / last stage of its accumulation group
};
__host__ __device__ constexpr StageInfo stage_info(int it) {
  if (it < 4) return {0, 0, it, it == 0, it == 3};
  if (it < 8) return {1, 0, it - 4, it == 4, it == 7};
  if (it < 12) return {0, 1, it - 8, it == 8, it == 11};
  if (it < 16) return {1, 1, it - 12, it == 12, it == 15};
  if (it < 18) return {2, 0, it - 16, 1, 0};
  if (it < 22) return {1, 2, it - 18, it == 18, it == 21};
  if (it < 24) return {2, 1, it - 22, 0, 0};
  if (it < 28) return {1, 3, it - 24, it == 24, it == 27};
  if (it < 30) return {2, 2, it - 28, 0, 0};
  return {2, 3, it - 30, 0, it == 31};
}

// CL = 2 (a 2-CTA cluster per window, used when 2 * n_win CTAs fit one wave): CTA `rank` owns head groups 2 rank, 2 rank + 1
// (16 stages, idx = LOCAL head group / Q tile 0):   0-3 Q | 4-7 K|V l 0 | 8-11 K|V l 1 | 12-13 proj(l 0) | 14-15 proj(l 1)
__host__ __device__ constexpr StageInfo stage_info2(int it) {
  if (it < 4) return {0, 0, it, it == 0, it == 3};
  if (it < 8) return {1, 0, it - 4, it == 4, it == 7};
  if (it < 12) return {1, 1, it - 8, it == 8, it == 11};
  if (it < 14) return {2, 0, it - 12, 1, 0};
  return {2, 1, it - 14, 0, it == 15};
}
__device__ __forceinline__ uint32_t tc_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void tc_cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// 544 threads = 17 warps: one SM sub-partition hosts 5 of them, so its 16 K registers allow 102 -> 96 registers per thread
// (a cap of 112 or 120 makes the launch fail with "too many resources").  The attention core therefore runs its softmax
// over two key halves (online rescaling), which keeps at most 10 score tiles (40 registers) alive instead of 19 (76).
//
// CL = 2: the two CTAs of a cluster share one window and split its four head groups (each streams half of the weights and
// runs half of the attention core; the LayerNorm is done by both).  Their partial output projections meet in x itself, like
// the partial sums of the fused MLP: phase A, CTA r writes shortcut + its partial for the PEER's 128 channels; cluster
// barrier; phase B, it adds its partial + bias to its own 128 channels.  Fixed order -> deterministic.  A first cluster
// barrier after the LayerNorm keeps a fast CTA from overwriting rows its peer has not gathered yet.
template <int NT, int CL>
__global__ void __launch_bounds__(kThreadsT, 1)
attn_win256_tc_kernel(const __grid_constant__ CUtensorMap tmap_wqkv, const __grid_constant__ CUtensorMap tmap_wproj,
                      const TcAttnParams p) {
  using Cfg = TCfg<NT>;
  constexpr int NSTG = CL == 2 ? 16 : 32;         // weight stages of this CTA
  constexpr int NHGL = Cfg::NHG / CL;             // head groups of this CTA
  const int rank = CL == 2 ? (int)tc_cluster_rank() : 0;
  const int hg0 = rank * NHGL;                    // first (global) head group of this CTA
  constexpr int C = Cfg::C, HD = Cfg::HD, HG = Cfg::HG, PQ = Cfg::PQ;
  constexpr int KSTEPS = Cfg::KSTEPS, XROWS = Cfg::XROWS, NKEY = Cfg::NKEY;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sb - smem_u32(smem_raw));
  __nv_bfloat16* qs = reinterpret_cast<__nv_bfloat16*>(sgen + Cfg::OFF_Q);
  __nv_bfloat16* ks = reinterpret_cast<__nv_bfloat16*>(sgen + Cfg::OFF_K);
  __nv_bfloat16* vs = reinterpret_cast<__nv_bfloat16*>(sgen + Cfg::OFF_V);
  int* coff = reinterpret_cast<int*>(sgen + Cfg::OFF_COFF);
  int* roff = reinterpret_cast<int*>(sgen + Cfg::OFF_ROFF);
  int* pix_s = reinterpret_cast<int*>(sgen + Cfg::OFF_PIX);
  float* bias_s = reinterpret_cast<float*>(sgen + Cfg::OFF_BIAS);
  const uint32_t bar0 = sb + Cfg::OFF_BAR;
  const uint32_t bar_full = bar0;               // 3 x 8
  const uint32_t bar_empty = bar0 + 24;         // 3 x 8
  const uint32_t bar_xn = bar0 + 48;            // workers -> MMA: LayerNorm'ed tokens in place
  const uint32_t bar_qfull = bar0 + 56;         // 2 x 8
  // one single-phase barrier per head group (a shared multi-phase barrier could be waited on two phases late)
  const uint32_t bar_kvfull = bar0 + 72;        // 4 x 8  MMA -> workers: K^T|V^T of head group hg complete
  const uint32_t bar_kvempty = bar0 + 104;      // 4 x 8  workers -> MMA: the K^T|V^T accumulator of hg has been read
  const uint32_t bar_oready = bar0 + 136;       // 4 x 8  workers -> MMA: attention output slab hg in place
  const uint32_t bar_pfull = bar0 + 168;
  const uint32_t bar_xn0 = bar0 + 176;          // workers -> MMA: token rows 0 .. 63 (query frame) in place
  const uint32_t tmem_slot = bar0 + 200;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int w = blockIdx.x / CL;
  const int n_kv = p.D * kTok;
  const int tbl_ld = p.D * kRel;
  const bool dbg = p.dbg != nullptr;
  const long long t_begin = dbg ? clock64() : 0;
  long long t_ln = 0, t_wait = 0, t_conv = 0, t_attn = 0;

  pdl_trigger();   // the next kernel of the chain may start its prologue
  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_xn, kWorkers / 32);
    mbar_init(bar_xn0, kWorkers / 32);
    for (int i = 0; i < 2; ++i) mbar_init(bar_qfull + 8 * i, 1);
    for (int i = 0; i < 4; ++i) {
      mbar_init(bar_kvfull + 8 * i, 1);
      mbar_init(bar_kvempty + 8 * i, kWorkers / 32);
      mbar_init(bar_oready + 8 * i, kWorkers / 32);
    }
    mbar_init(bar_pfull, 1);
    fence_barrier_init();
  }
  if (warp == kWorkers / 32) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(sgen + Cfg::OFF_BAR + 200);

  if (warp == kWorkers / 32) {
    // =========================================== TMA + MMA warp ==========================================================
    // stage `it` (0 .. 31) = K block it % 4 of batch it / 4.  The loop is FULLY UNROLLED so that every stage / parity /
    // coordinate / descriptor offset is an immediate: as a rolled loop the single issuing lane spent ~1.5 K cycles per
    // stage in ~300 dependent scalar instructions (batch decoding, % 3, 64-bit descriptor arithmetic) -- 4x the MMA time.
    const uint32_t ring = sb + Cfg::OFF_RING;
    if (CL == 2) tc_cluster_arrive();   // barrier 0 (see the workers); this warp waits for it after its schedule
    auto issue_load = [&](const int it) {
      const StageInfo si = CL == 2 ? stage_info2(it) : stage_info(it);
      const int s = it % kStages;
      const uint32_t dst = ring + s * kStageBytes, bar = bar_full + 8 * s;
      mbar_arrive_expect_tx(bar, kStageBytes);
      // global indices: head group hg0 + idx; Q tile = rank for CL = 2 (the tile that holds this CTA's two head groups)
      const int ghg = hg0 + si.idx, gq = CL == 2 ? rank : si.idx;
      if (si.kind == 2) {         // Wproj rows [128 kb, +128), K block = head group
        tma_load_2d(dst, &tmap_wproj, bar, ghg * BK, 128 * si.kb);
        tma_load_2d(dst + 8192, &tmap_wproj, bar, ghg * BK, 128 * si.kb + 64);
      } else {                    // Q tile: Wq rows [128 gq, +128);  K|V: Wk rows of the head group, then its Wv rows
        const int r0 = si.kind == 1 ? C + 64 * ghg : 128 * gq, r1 = si.kind == 1 ? 2 * C + 64 * ghg : 128 * gq + 64;
        tma_load_2d(dst, &tmap_wqkv, bar, si.kb * BK, r0);
        tma_load_2d(dst + 8192, &tmap_wqkv, bar, si.kb * BK, r1);
      }
    };
    if (elect_one_sync()) {
      prefetch_tmap(&tmap_wqkv);
      prefetch_tmap(&tmap_wproj);
      issue_load(0);
      issue_load(1);
    }
    __syncwarp();
    const uint64_t adesc0 = make_smem_desc(ring);
    const uint64_t bdesc_xn = make_smem_desc(sb + Cfg::OFF_XN), bdesc_o = make_smem_desc(sb + Cfg::OFF_O);
#pragma unroll
    for (int it = 0; it < NSTG; ++it) {
      const StageInfo si = CL == 2 ? stage_info2(it) : stage_info(it);
      const int s = it % kStages;
      if (dbg && lane == 0 && (it & 7) == 0) p.dbg[(size_t)gridDim.x * 8 + (size_t)blockIdx.x * 8 + (it >> 3)] = clock64() - t_begin;
      // operands / accumulator of this group available?
      if (it == 0) mbar_wait(bar_xn0, 0);     // the Q^T tiles read rows 0 .. 63 only
      if (it == 4) mbar_wait(bar_xn, 0);      // first K^T|V^T stage: every token row
      if (si.kind == 1 && si.idx >= 1 && si.first) mbar_wait(bar_kvempty + 8 * (si.idx - 1), 0);   // accumulator read by conversion(idx - 1)
      if (si.kind == 2 && si.kb == 0) mbar_wait(bar_oready + 8 * si.idx, 0);                        // O slab idx written
      mbar_wait(bar_full + 8 * s, (it / kStages) & 1u);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint64_t adesc = adesc0 + (uint64_t)((s * kStageBytes) >> 4);
        // B: the LayerNorm'ed tokens, K block kb (the query frame's tokens are rows 0 .. 48), or attention-output slab idx
        const uint64_t bdesc = si.kind == 2 ? bdesc_o + (uint64_t)((si.idx * 64 * 128) >> 4) : bdesc_xn + (uint64_t)((si.kb * Cfg::XN_SLAB) >> 4);
        const uint32_t d_tmem = tmem_base + (si.kind == 1 ? Cfg::TM_KV : si.kind == 0 ? Cfg::TM_Q + 64 * si.idx : Cfg::TM_P + 64 * si.kb);   // idx is local
        const uint32_t idesc = si.kind == 1 ? idesc_mn(128, XROWS) : idesc_mn(128, 64);
        const bool fresh = si.kind == 2 ? si.idx == 0 : si.kb == 0;      // first K block of its accumulator
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (fresh && k == 0) ? 0u : 1u);
        umma_commit(bar_empty + 8 * s);
        if (si.last) {
          if (si.kind == 0) umma_commit(bar_qfull + 8 * si.idx);
          else if (si.kind == 1) umma_commit(bar_kvfull + 8 * si.idx);
          else umma_commit(bar_pfull);
        }
      }
      __syncwarp();
      // refill AFTER this iteration's MMAs are queued: the wait below is for the MMAs of the PREVIOUS iteration (they
      // free stage (it - 1) % kStages), so the tensor pipe always has the next batch queued behind the running one
      if (it + kStages - 1 < NSTG) {
        const int nx = it + kStages - 1, sn = nx % kStages;
        if (nx >= kStages) mbar_wait(bar_empty + 8 * sn, ((nx / kStages) - 1) & 1u);
        if (elect_one_sync()) issue_load(nx);
        __syncwarp();
      }
    }
    if (dbg && lane == 0) p.dbg[(size_t)gridDim.x * 8 + (size_t)blockIdx.x * 8 + 4] = clock64() - t_begin;
    __syncwarp();
    if (CL == 2) {
      tc_cluster_wait();      // barrier 0
      tc_cluster_arrive();    // barrier 1 (between the two phases of the workers' epilogue)
      tc_cluster_wait();
    }
  } else {
    // =========================================== worker warps ===========================================================
    const int g = lane >> 2, t = lane & 3;
    // ---- index tables.  Token rows are staged with the QUERY frame first: slot s of the staged order is frame
    // d = perm(s) = (s == 0 ? q_slot : (s <= q_slot ? s - 1 : s)); the bias lookup only needs d per key ------------------
    for (int n = tid; n < NKEY; n += kWorkers) {
      int v = 0;
      if (n < n_kv) {
        const int s = n / kTok, r = n - s * kTok, a = r / 7, b = r - a * 7;
        const int d = s == 0 ? p.q_slot : (s <= p.q_slot ? s - 1 : s);
        v = d * kRel + (6 - a) * 13 + (6 - b);
      }
      coff[n] = v * 4;
    }
    if (tid < 64) {
      const int a = tid / 7, b = tid - a * 7;
      roff[tid] = tid < kTok ? (a * 13 + b) * 4 : 0;
      pix_s[tid] = tid < kTok ? __ldg(p.tok_map + (size_t)w * kTok + tid) : -1;
    }
    for (int i = tid; i < 768; i += kWorkers) bias_s[i] = __ldg(p.bqkv + i);
    worker_sync();
    pdl_wait();   // everything above is static data; the frames below were written by the previous kernel of the chain

    // ---- gather + LayerNorm -> 128B-swizzled K-major slabs (8 lanes per token, 64 tokens per pass) ------------------------
    // The loads of pass i + 1 are issued before pass i is reduced (two passes of 32 registers in flight), and the MMA warp
    // is released for the Q^T tiles as soon as pass 0 (rows 0 .. 63: the query frame's tokens) is in place.
    {
      const int j = lane & 7, sub = lane >> 3;
      constexpr int NPASS = (XROWS + 63) / 64;
      auto load_pass = [&](int pass, float (&v)[4][8]) {
        const int n = pass * 64 + warp * 4 + sub;
        const float* src = nullptr;
        if (n < n_kv) {
          const int s = n / kTok, tok = n - s * kTok;
          const int d = s == 0 ? p.q_slot : (s <= p.q_slot ? s - 1 : s);
          const int pix = pix_s[tok];
          const float* fr = p.frames[0];
#pragma unroll
          for (int q = 1; q < 8; ++q) fr = (d == q) ? p.frames[q] : fr;
          if (fr != nullptr && pix >= 0) src = fr + (size_t)pix * C + j * 8;
        }
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) {
          if (src != nullptr) {
            const float4 t0 = *(reinterpret_cast<const float4*>(src + kb * 64));
            const float4 t1 = *(reinterpret_cast<const float4*>(src + kb * 64 + 4));
            v[kb][0] = t0.x; v[kb][1] = t0.y; v[kb][2] = t0.z; v[kb][3] = t0.w;
            v[kb][4] = t1.x; v[kb][5] = t1.y; v[kb][6] = t1.z; v[kb][7] = t1.w;
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[kb][e] = 0.f;
          }
        }
      };
      auto norm_pass = [&](int pass, float (&v)[4][8]) {
        const int n = pass * 64 + warp * 4 + sub;
        if (n >= XROWS) return;
        float sum = 0.f;
#pragma unroll
        for (int kb = 0; kb < 4; ++kb)
#pragma unroll
          for (int e = 0; e < 8; ++e) sum += v[kb][e];
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        sum += __shfl_xor_sync(0xffffffffu, sum, 4);
        const float mean = sum / (float)C;
        float sq = 0.f;
#pragma unroll
        for (int kb = 0; kb < 4; ++kb)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float dlt = v[kb][e] - mean;
            v[kb][e] = dlt;
            sq += dlt * dlt;
          }
        sq += __shfl_xor_sync(0xffffffffu, sq, 1);
        sq += __shfl_xor_sync(0xffffffffu, sq, 2);
        sq += __shfl_xor_sync(0xffffffffu, sq, 4);
        const float rstd = rsqrt_approx(sq / (float)C + 1e-5f);
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) {
#pragma unroll
          for (int e = 0; e < 8; ++e) v[kb][e] *= rstd;
          const uint4 pk = pack8_bf16(v[kb]);
          const uint32_t dst = sb + Cfg::OFF_XN + kb * Cfg::XN_SLAB + (uint32_t)n * 128u + (((uint32_t)j ^ (uint32_t)(n & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk.x), "r"(pk.y), "r"(pk.z), "r"(pk.w) : "memory");
        }
      };
      float va[4][8], vb[4][8];
      load_pass(0, va);
      if (NPASS > 1) load_pass(1, vb);
      norm_pass(0, va);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_xn0);          // rows 0 .. 63 in place: the Q^T tiles can start
      if (NPASS > 2) load_pass(2, va);
      if (NPASS > 1) norm_pass(1, vb);
      if (NPASS > 2) norm_pass(2, va);
      static_assert(NPASS <= 3, "LayerNorm pipeline covers up to 3 passes (XROWS <= 192)");
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_xn);
    if (dbg) t_ln = clock64() - t_begin;
    if (CL == 2) {      // barrier 0: both CTAs have gathered their tokens; from here on the peer may write rows of x
      __syncwarp();
      tc_cluster_arrive();
      tc_cluster_wait();
    }

    const uint32_t ks_u32 = sb + Cfg::OFF_K, vs_u32 = sb + Cfg::OFF_V, tbl_u32 = sb + Cfg::OFF_TBL, coff_u32 = sb + Cfg::OFF_COFF;
    constexpr uint32_t kOnes = 0x3C003C00u;
    constexpr float kLog2e = 1.4426950408889634f;
    const int qd = warp & 3, part = warp >> 2;                   // TMEM lane quarter of this warp, column-chunk phase
    const uint32_t lane_sel = (uint32_t)(qd * 32) << 16;

    for (int l = 0; l < NHGL; ++l) {
      const int hg = hg0 + l;             // global head group (weights, biases, bias table); l indexes barriers / TMEM / O slabs
      const int lq = CL == 2 ? 0 : hg >> 1;
      long long t0 = dbg ? clock64() : 0;
      // bias table of this head group (cp.async, lands while the accumulators are converted)
      {
        const float* src = p.tbl + (size_t)hg * HG * tbl_ld;
        const int n16 = HG * tbl_ld / 4;
        for (int i = tid; i < n16; i += kWorkers) cpa16(sb + Cfg::OFF_TBL + (uint32_t)(i * 16), src + i * 4);
        asm volatile("cp.async.commit_group;" ::: "memory");
      }
      if ((hg & 1) == 0) mbar_wait_polite(bar_qfull + 8 * lq, 0, lane);
      mbar_wait_polite(bar_kvfull + 8 * l, 0, lane);
      tcgen05_fence_after();
      if (dbg) { const long long t1 = clock64(); t_wait += t1 - t0; t0 = t1; }
      // ---- K^T | V^T (TMEM lane = channel: 0..63 k, 64..127 v; column = token) -> [token][channel] tiles -----------------
      {
        const uint32_t tk = tmem_base + Cfg::TM_KV + lane_sel;
        const bool is_k = qd < 2;
        const int ch = (qd & 1) * 32 + lane;
        const float bias = bias_s[(is_k ? C : 2 * C) + hg * 64 + ch];
        __nv_bfloat16* dstm = is_k ? ks : vs;
        constexpr int NCH = (XROWS / 8 + 3) / 4;       // 8-token column chunks per warp (chunk c8 = part + 4 i)
        uint32_t raw[NCH][8];
        const bool has_q = (qd >> 1) == (hg & 1);
#pragma unroll
        for (int i = 0; i < NCH; ++i)
          if (part + 4 * i < XROWS / 8) tmem_ld_x8(tk + (uint32_t)((part + 4 * i) * 8), raw[i]);
        tmem_ld_wait();
        // the accumulators are in registers: hand the TMEM buffer back to the MMA warp before the stores
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_kvempty + 8 * l);
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int c8 = part + 4 * i;
          if (c8 < XROWS / 8) {
            float val[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) val[e] = __uint_as_float(raw[i][e]) + bias;
            // k stays bf16 (q.k^T is a bf16 product); v is fp16 for the fp16 P.V product
            uint4 pk;
            if (is_k) {
              pk.x = pack2(val[0], val[1]); pk.y = pack2(val[2], val[3]); pk.z = pack2(val[4], val[5]); pk.w = pack2(val[6], val[7]);
            } else {
              pk.x = pack2_hs(val[0], val[1]); pk.y = pack2_hs(val[2], val[3]); pk.z = pack2_hs(val[4], val[5]); pk.w = pack2_hs(val[6], val[7]);
            }
            *reinterpret_cast<uint4*>(dstm + ch * Cfg::PT + c8 * 8) = pk;   // tokens [8 c8, 8 c8 + 8) of channel ch
          }
        }
        // Q^T tile hg / 2, lanes (hg & 1) * 64 + channel, columns = the 64 staged query tokens
        if (has_q) {
          const uint32_t tq = tmem_base + Cfg::TM_Q + 64 * lq + lane_sel;
          uint32_t rq[2][8];
          tmem_ld_x8(tq + (uint32_t)(part * 8), rq[0]);
          tmem_ld_x8(tq + (uint32_t)((part + 4) * 8), rq[1]);
          tmem_ld_wait();
          const float bq = bias_s[hg * 64 + ch];
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int e = 0; e < 8; ++e)
              qs[((part + 4 * i) * 8 + e) * PQ + ch] = __float2bfloat16_rn(__uint_as_float(rq[i][e]) + bq);
        }
      }
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      worker_sync();   // q / k / v tiles and the bias table visible to every worker warp
      if (dbg) { const long long t1 = clock64(); t_conv += t1 - t0; t0 = t1; }

      // ---- attention: warp = (head of the group, 16-row query tile); scores stay in registers ----------------------------
      {
        const int hl = warp >> 2, mt = warp & 3;
        const int row0 = mt * 16 + g, row1 = row0 + 8;
        const uint32_t r0a = tbl_u32 + (uint32_t)(hl * tbl_ld * 4 + roff[row0]);
        const uint32_t r1a = tbl_u32 + (uint32_t)(hl * tbl_ld * 4 + roff[row1]);
        uint32_t qa[4];
        {
          const __nv_bfloat16* q0 = qs + row0 * PQ + hl * HD;
          const __nv_bfloat16* q1 = qs + row1 * PQ + hl * HD;
          qa[0] = *reinterpret_cast<const uint32_t*>(q0 + 2 * t);
          qa[1] = *reinterpret_cast<const uint32_t*>(q1 + 2 * t);
          qa[2] = *reinterpret_cast<const uint32_t*>(q0 + 2 * t + 8);
          qa[3] = *reinterpret_cast<const uint32_t*>(q1 + 2 * t + 8);
        }
        float o[2][4], ol[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int v = 0; v < 2; ++v) o[v][0] = o[v][1] = o[v][2] = o[v][3] = 0.f;
        // two key halves of an even number of 8-key tiles (a k16 step of P.V spans two tiles): online softmax
        constexpr int NT1 = ((NT + 1) / 2 + 1) & ~1;      // 19 -> 10, 13 -> 8, 7 -> 4
        float m0s = -INFINITY, m1s = -INFINITY;            // running row maxima, already multiplied by log2(e)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          constexpr int kMaxT = NT1 > NT - NT1 ? NT1 : NT - NT1;
          const int j0 = half == 0 ? 0 : NT1, nj = half == 0 ? NT1 : NT - NT1;
          float s[kMaxT][4];
#pragma unroll
          for (int jj = 0; jj < kMaxT; ++jj) {
            if (jj < nj) {
              const int j = j0 + jj;
              const uint2 cp = lds_u64(coff_u32 + (uint32_t)((j * 8 + 2 * t) * 4));
              s[jj][0] = lds_f32(r0a + cp.x); s[jj][1] = lds_f32(r0a + cp.y);
              s[jj][2] = lds_f32(r1a + cp.x); s[jj][3] = lds_f32(r1a + cp.y);
              if (j == NT - 1) {   // only the last key tile can hold padding keys
                if (j * 8 + 2 * t >= n_kv) s[jj][0] = s[jj][2] = -1e30f;
                if (j * 8 + 2 * t + 1 >= n_kv) s[jj][1] = s[jj][3] = -1e30f;
              }
              uint32_t kb0, kb1;   // (channels 2t, 2t + 1 | 8 + 2t, 9 + 2t of the head; token 8 j + g)
              ldsm_x2_trans(kb0, kb1, ks_u32 + (uint32_t)(((hl * HD + (lane & 15)) * Cfg::PT + j * 8) * 2));
              mma16816(s[jj], qa, kb0, kb1);
            }
          }
          float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
          for (int jj = 0; jj < kMaxT; ++jj) {
            if (jj < nj) {
              mx0 = fmaxf(mx0, fmaxf(s[jj][0], s[jj][1]));
              mx1 = fmaxf(mx1, fmaxf(s[jj][2], s[jj][3]));
            }
          }
          mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
          mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
          mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
          mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
          const float n0s = fmaxf(m0s, mx0 * kLog2e), n1s = fmaxf(m1s, mx1 * kLog2e);
          if (half == 1) {   // rescale what the first half accumulated to the new maxima
            float c0, c1;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(c0) : "f"(m0s - n0s));
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(c1) : "f"(m1s - n1s));
#pragma unroll
            for (int v = 0; v < 2; ++v) { o[v][0] *= c0; o[v][1] *= c0; o[v][2] *= c1; o[v][3] *= c1; }
            ol[0] *= c0; ol[1] *= c0; ol[2] *= c1; ol[3] *= c1;
          }
          m0s = n0s; m1s = n1s;
#pragma unroll
          for (int k2 = 0; k2 < (kMaxT + 1) / 2; ++k2) {
            if (2 * k2 < nj) {
              const int kk = j0 / 2 + k2;
              uint32_t pa[4];
              pa[0] = ex2_h2(fmaf(s[2 * k2][0], kLog2e, -m0s), fmaf(s[2 * k2][1], kLog2e, -m0s));
              pa[1] = ex2_h2(fmaf(s[2 * k2][2], kLog2e, -m1s), fmaf(s[2 * k2][3], kLog2e, -m1s));
              if (2 * k2 + 1 < nj) {
                pa[2] = ex2_h2(fmaf(s[2 * k2 + 1][0], kLog2e, -m0s), fmaf(s[2 * k2 + 1][1], kLog2e, -m0s));
                pa[3] = ex2_h2(fmaf(s[2 * k2 + 1][2], kLog2e, -m1s), fmaf(s[2 * k2 + 1][3], kLog2e, -m1s));
              } else {
                pa[2] = pa[3] = 0u;
              }
#pragma unroll
              for (int v = 0; v < 2; ++v) {
                uint32_t vb0, vb1;
                ldsm_x2(vb0, vb1, vs_u32 + (uint32_t)(((hl * HD + 8 * v + (lane & 7)) * Cfg::PT + kk * 16 + ((lane >> 3) & 1) * 8) * 2));
                mma16816_f16(o[v], pa, vb0, vb1);
              }
              mma16816_f16(ol, pa, kOnes, kOnes);   // row sums
            }
          }
        }
        const float inv0 = rcp_approx(ol[0]), inv1 = rcp_approx(ol[2]);
        // attention output -> slab hg of the swizzled K-major O tile (token row, 64 channels of this head group)
        const uint32_t o_slab = sb + Cfg::OFF_O + l * (64 * 128);
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int col = hl * HD + 8 * v + 2 * t;                     // channel within the head group's 64
          const uint32_t a0 = o_slab + (uint32_t)row0 * 128u + ((((uint32_t)col >> 3) ^ (uint32_t)(row0 & 7)) << 4) + (col & 7) * 2;
          const uint32_t a1 = o_slab + (uint32_t)row1 * 128u + ((((uint32_t)col >> 3) ^ (uint32_t)(row1 & 7)) << 4) + (col & 7) * 2;
          asm volatile("st.shared.b32 [%0], %1;" ::"r"(a0), "r"(pack2(o[v][0] * inv0, o[v][1] * inv0)) : "memory");
          asm volatile("st.shared.b32 [%0], %1;" ::"r"(a1), "r"(pack2(o[v][2] * inv1, o[v][3] * inv1)) : "memory");
        }
      }
      if (dbg) t_attn += clock64() - t0;
      // O slab hg is complete: hand it to the MMA warp, which accumulates P^T += Wproj[:, hg] . O_hg^T while the workers
      // go on with the next head group (only head group 3's share of the projection is left for the end)
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_oready + 8 * l);
      worker_sync();   // every warp is done with this head group's q / k / v tiles and bias table
    }
    // ---- x[pix] = shortcut + proj(o) + b (DTransformer.py:204, 294-299) --------------------------------------------------------
    const long long t_p0 = dbg ? clock64() : 0;
    if (CL == 1) {
      const int pt = part & 1, th = part >> 1;                  // projection tile (128 channels), token half
      const int ch = pt * 128 + qd * 32 + lane;
      const float bp = __ldg(p.bproj + ch);
      // the shortcut rows (independent 128-byte coalesced reads) are in flight while the projection MMAs run.
      // 8-token column chunks: token half 0 takes chunks 0-2 (tokens 0..23), half 1 chunks 3-6 (tokens 24..48)
      const float* shortcut = p.frames[p.q_slot];
      const int c0 = th == 0 ? 0 : 3, nch = th == 0 ? 3 : 4;
      float sc[4][8];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int tok = (c0 + i) * 8 + e;
          const int pix = (i < nch && tok < kTok) ? pix_s[tok] : -1;
          sc[i][e] = pix >= 0 ? *(shortcut + (size_t)pix * C + ch) : 0.f;
        }
      mbar_wait_polite(bar_pfull, 0, lane);
      tcgen05_fence_after();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (i < nch) {
          uint32_t raw[8];
          tmem_ld_x8(tmem_base + Cfg::TM_P + 64 * pt + (uint32_t)((c0 + i) * 8) + lane_sel, raw);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int tok = (c0 + i) * 8 + e;
            const int pix = tok < kTok ? pix_s[tok] : -1;
            if (pix >= 0) p.xs[(size_t)pix * C + ch] = sc[i][e] + __uint_as_float(raw[e]) + bp;
          }
        }
      }
    } else {
      // phase A: the PEER's 128 channels = shortcut + my partial projection.  All 16 warps work on one projection tile:
      // lane quarter -> 32 channels, part -> token chunks 2 part, 2 part + 1 (7 chunks of 8 tokens)
      const float* shortcut = p.frames[p.q_slot];
      {
        const int pt = 1 - rank;
        const int ch = pt * 128 + qd * 32 + lane;
        float sc[2][8];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int tok = (2 * part + i) * 8 + e;
            const int pix = tok < kTok ? pix_s[tok] : -1;
            sc[i][e] = pix >= 0 ? *(shortcut + (size_t)pix * C + ch) : 0.f;
          }
        mbar_wait_polite(bar_pfull, 0, lane);
        tcgen05_fence_after();
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          if ((2 * part + i) * 8 < kTok) {
            uint32_t raw[8];
            tmem_ld_x8(tmem_base + Cfg::TM_P + 64 * pt + (uint32_t)((2 * part + i) * 8) + lane_sel, raw);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int tok = (2 * part + i) * 8 + e;
              const int pix = tok < kTok ? pix_s[tok] : -1;
              if (pix >= 0) p.xs[(size_t)pix * C + ch] = sc[i][e] + __uint_as_float(raw[e]);
            }
          }
        }
      }
      __syncwarp();
      tc_cluster_arrive();    // barrier 1: the peer's phase-A rows of my channels are in x (release / acquire at cluster scope)
      tc_cluster_wait();
      // phase B: my own 128 channels += my partial + bias (read through L2: the peer wrote them)
      {
        const int pt = rank;
        const int ch = pt * 128 + qd * 32 + lane;
        const float bp = __ldg(p.bproj + ch);
        float cur[2][8];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int tok = (2 * part + i) * 8 + e;
            const int pix = tok < kTok ? pix_s[tok] : -1;
            cur[i][e] = pix >= 0 ? __ldcg(p.xs + (size_t)pix * C + ch) : 0.f;
          }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          if ((2 * part + i) * 8 < kTok) {
            uint32_t raw[8];
            tmem_ld_x8(tmem_base + Cfg::TM_P + 64 * pt + (uint32_t)((2 * part + i) * 8) + lane_sel, raw);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int tok = (2 * part + i) * 8 + e;
              const int pix = tok < kTok ? pix_s[tok] : -1;
              if (pix >= 0) p.xs[(size_t)pix * C + ch] = cur[i][e] + __uint_as_float(raw[e]) + bp;
            }
          }
        }
      }
    }
    tcgen05_fence_before();
    if (dbg && tid == 0) {
      long long* o = p.dbg + (size_t)blockIdx.x * 8;
      const long long t_end = clock64();
      o[0] = t_end - t_begin; o[1] = t_ln; o[2] = t_wait; o[3] = t_conv; o[4] = 0; o[5] = t_attn; o[6] = t_end - t_p0;
    }
  }
  __syncthreads();
  if (warp == kWorkers / 32) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int NT, int CL>
int launch_tc256(const CUtensorMap& tq, const CUtensorMap& tp, const TcAttnParams& p, cudaStream_t s) {
  using Cfg = TCfg<NT>;
  auto kern = attn_win256_tc_kernel<NT, CL>;
  if (first_use_on_device((const void*)kern)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    BDE_REQUIRE(e == cudaSuccess, "bde_window_attention_fused: smem attribute (%d bytes): %s", Cfg::SMEM, cudaGetErrorString(e));
  }
  TcAttnParams q = p;
  q.dbg = (g_dbg != nullptr && (size_t)2 * CL * p.n_win <= g_dbg_ctas) ? g_dbg : nullptr;   // rows [n_ctas, 2 n_ctas): MMA-warp timeline
  const cudaError_t le = launch_pdl(kern, (unsigned)(p.n_win * CL), (unsigned)kThreadsT, (size_t)Cfg::SMEM, s, CL, tq, tp, q);
  BDE_REQUIRE(le == cudaSuccess, "bde_window_attention_fused: launch: %s", cudaGetErrorString(le));
  return check_launch("attn_win256_tc_kernel");
}

}  // namespace

// C = 256 whole-window attention half with tcgen05 projections; called by bde_window_attention_fused (attn_fused.cu)
int attn_win256_tc_launch(const float* const* frames, int D, int q_slot, const int* tok_map, int n_win, const void* wqkv,
                          const float* bqkv, const float* bias_tbl, const void* wproj, const float* bproj, float* xs,
                          cudaStream_t s) {
  BDE_REQUIRE((((uintptr_t)wqkv) & 127) == 0 && (((uintptr_t)wproj) & 127) == 0,
              "bde_window_attention_fused: weights must be 128-byte aligned for the TMA path");
  CUtensorMap tq, tp;
  int rc = get_weight_tmap(wqkv, 768, 256, 64, &tq);
  if (rc != 0) return rc;
  rc = get_weight_tmap(wproj, 256, 256, 64, &tp);
  if (rc != 0) return rc;
  TcAttnParams p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < 8; ++i) p.frames[i] = i < D ? frames[i] : nullptr;
  p.tok_map = tok_map;
  p.bqkv = bqkv;
  p.tbl = bias_tbl;
  p.bproj = bproj;
  p.xs = xs;
  p.n_win = n_win; p.D = D; p.q_slot = q_slot;
  // a 2-CTA cluster per window while both CTAs of every window still fit one wave (one sequence: 35 windows -> 70 CTAs)
  int cl = 2 * n_win <= device_sm_count() ? 2 : 1;
  if (const char* e = getenv("BDE2VID_ATTN_TC256_CLUSTER")) {
    const int f = atoi(e);
    if (f == 1 || f == 2) cl = f;
  }
  if (cl == 2) {
    switch (D) {
      case 1: return launch_tc256<7, 2>(tq, tp, p, s);
      case 2: return launch_tc256<13, 2>(tq, tp, p, s);
      default: return launch_tc256<19, 2>(tq, tp, p, s);
    }
  }
  switch (D) {
    case 1: return launch_tc256<7, 1>(tq, tp, p, s);
    case 2: return launch_tc256<13, 1>(tq, tp, p, s);
    default: return launch_tc256<19, 1>(tq, tp, p, s);
  }
}

}  // namespace tc
}  // namespace bde
