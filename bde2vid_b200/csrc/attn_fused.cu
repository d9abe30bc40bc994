// Fused multi-frame window attention for one SwinTransformerBlock3D attention half
// (model/BDE2VID/DTransformer.py:254-299, WindowAttention3D :164-207):
//
//   window gather (plain or dilated, via a token map) -> LayerNorm (norm_q / norm_kv, affine folded
//   into the projections) -> q, k, v projections -> softmax(q k^T + relative-position bias) v
//   -> [C == 64: output projection + window_reverse + crop + shortcut, scatter-added into x]
//      [C == 256: bf16 attention output, the projection runs as a tcgen05 GEMM with a scatter epilogue]
//
// One CTA = one window x one group of 64 projection columns (= 64 / head_dim heads), so q, k and v never
// leave shared memory: the unfused path wrote a [tokens, 3C] bf16 buffer to HBM and read it back.
// The GEMMs here are small (<= 160 x 64 x C per CTA) and the softmax needs the scores in registers,
// so the kernel uses warp-level mma.sync (bf16, fp32 accumulate) fed by ldmatrix from padded smem rows.
// The relative-position bias is rebuilt from the compact per-head table (D x 13 x 13 entries) instead
// of the expanded [heads, 49, D*49] tensor, which would not fit in shared memory next to the operands.
#include "common.cuh"

#include <cuda_fp16.h>
// Ablation builds for tools/attn64_probe.sh (timing only, results are wrong): bit 0 = no bias-table loads, bit 1 = no MUFU.EX2
// in the probabilities, 4 = skip the level-1 attention core altogether, 8 = no global gather (LayerNorm of zeros), 16 = no q/k/v
// projection MMAs, 32 = no output projection + scatter.  0 in every shipped build.
#ifndef BDE_ATTN_PROBE
#define BDE_ATTN_PROBE 0
#endif
namespace bde {
namespace tc {
extern long long* g_dbg;   // bring-up cycle-counter buffer owned by gemm_tc.cu (bde_tc_debug_enable)
extern size_t g_dbg_ctas;
int attn_win256_tc_launch(const float* const* frames, int D, int q_slot, const int* tok_map, int n_win, const void* wqkv,
                          const float* bqkv, const float* bias_tbl, const void* wproj, const float* bproj, float* xs,
                          cudaStream_t s);
}  // namespace tc
namespace {

constexpr int kTok = 49;       // 7 x 7 window
constexpr int kRel = 169;      // 13 x 13 relative offsets per frame pair
constexpr int kThreadsF = 256;

struct FusedAttnParams {
  const float* frames[8];        // D fp32 [P, C] frame maps (query slot = the running x), NULL = all-zero frame
  const int* tok_map;            // int32 [n_win * 49]: source / destination pixel row or -1
  const __nv_bfloat16* wqkv;     // [3C, C] rows q | k | v, LayerNorm gamma and the q scale folded in
  const float* bqkv;             // [3C]
  const float* tbl;              // [heads, D * 169] bias table rows of the query slot
  const __nv_bfloat16* wproj;    // [C, C]   (C == 64)
  const float* bproj;            // [C]      (C == 64)
  float* xs;                     // fp32 [P, C] += proj(attn)      (C == 64)
  __nv_bfloat16* o_out;          // bf16 [n_win * 49, C]           (C == 256)
  int n_win, D, q_slot, heads;
  long long* dbg;   // optional per-CTA phase cycle counters (8 slots per CTA), bring-up profiling
};

__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// K = 8 form: head_dim 4 fills half of it (lanes t >= 2 hold zeros); the K = 16 form needed two more zero registers per
// operand, materialised with MOV / CS2R in front of every score tile (2.9 % of the level-1 kernel's instructions)
__device__ __forceinline__ void mma1688(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(b0));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_trans(uint32_t& r0, uint32_t& r1, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ void cpa16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cpa_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cpa_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
template <int OFF>
__device__ __forceinline__ float lds_f32_off(uint32_t addr) {   // [register + immediate]: no address add
  float v;
  asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(addr), "n"(OFF));
  return v;
}
__device__ __forceinline__ uint2 lds_u64(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}
// P.V runs in fp16 (fp32 accumulate): fp16 carries 3 more mantissa bits than bf16 for the probabilities;
// p <= 1 and |v| is O(10), far inside the fp16 range.
__device__ __forceinline__ void mma16816_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// 1 / x and 1 / sqrt(x) as ONE MUFU op each (<= 1-2 ulp; the results are rounded to bf16 right after).  The IEEE forms cost a
// MUFU + Newton step + range check + slow-path branch each: 3.4 % + 1.8 % of the level-1 kernel's stall samples (ncu source view)
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
// V tiles: values beyond the fp16 range saturate at +-65504 instead of becoming inf (inf * p = nan for p = 0); with the
// LayerNorm'ed inputs of this model |v| is O(10), the clamp only matters for pathological checkpoints
__device__ __forceinline__ uint32_t pack2_hs(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// (2^lo, 2^hi) as an fp16 pair.  Two fp32 MUFU.EX2 + one packing convert: ex2.approx.f16x2 is NOT a single MUFU op on
// sm_100a (ptxas expands it to unpack + 2 x MUFU.EX2 + pack: measured +30 % instructions in this kernel).
__device__ __forceinline__ uint32_t ex2_h2(float lo, float hi) {
#if BDE_ATTN_PROBE & 2
  return pack2_h(lo, hi);
#endif
  float a, b;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(a) : "f"(lo));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(b) : "f"(hi));
  return pack2_h(a, b);
}

template <int C, int HD, int NT>
struct FusedCfg {
  static constexpr int HG = 64 / HD;              // heads per CTA
  static constexpr int PX = C + 8;                // pitch (bf16 elements) of the LayerNorm'ed tokens and weight slices
  static constexpr int PQ = 72;                   // pitch of q / k / v / o tiles
  static constexpr int KSTEPS = (NT + 1) / 2;     // k16 steps of P.V
  static constexpr int XROWS = KSTEPS * 16;       // token rows staged (zero beyond n_kv)
  static constexpr int NKEY = NT * 8;
  static constexpr int DMAX = NT <= 7 ? 1 : (NT <= 13 ? 2 : 3);
  static constexpr int NW = C == 64 ? 3 : 2;      // weight-slice buffers
  static constexpr int XN_BYTES = XROWS * PX * 2;
  static constexpr int W_BYTES = NW * 64 * PX * 2;
  static constexpr int TBL_BYTES = HG * DMAX * kRel * 4;
  static constexpr int OS_BYTES = 64 * PQ * 2;
  static constexpr int WP_BYTES = C == 64 ? 64 * PX * 2 : 0;
  // C == 64, one window per CTA: the bias table, the attention-output tile and the projection weights reuse the token /
  // weight region once the q, k, v projections are done (keeps the CTA under half an SM's shared memory)
  static constexpr int A_BYTES = C == 64 ? (XN_BYTES + W_BYTES > TBL_BYTES + OS_BYTES + WP_BYTES ? XN_BYTES + W_BYTES
                                                                                               : TBL_BYTES + OS_BYTES + WP_BYTES)
                                         : XN_BYTES + W_BYTES + TBL_BYTES;
  static constexpr int OFF_XN = 0;
  static constexpr int OFF_W = XN_BYTES;
  static constexpr int OFF_TBL = C == 64 ? 0 : XN_BYTES + W_BYTES;
  static constexpr int OFF_OS = TBL_BYTES;                  // C == 64 only
  static constexpr int OFF_WP = TBL_BYTES + OS_BYTES;       // C == 64 only
  static constexpr int OFF_Q = A_BYTES;
  static constexpr int OFF_K = OFF_Q + 64 * PQ * 2;
  static constexpr int OFF_V = OFF_K + NKEY * PQ * 2;
  static constexpr int OFF_COFF = OFF_V + XROWS * PQ * 2;   // int32 [NKEY]  byte offsets into a bias-table row block
  static constexpr int OFF_ROFF = OFF_COFF + NKEY * 4;      // int32 [64]
  static constexpr int OFF_PIX = OFF_ROFF + 256;            // int32 [64]
  static constexpr int SMEM = OFF_PIX + 256;
};

// acc[mt][nt][4] += A[rows, C] (smem, pitch PX) * Wslice[64, C]^T (smem, pitch PX) for this warp's
// (m-tile list, n-tile pair).  a_row(mt, r) gives the smem row of tile row r.
// The accumulators start at (init0, init1): the bias of this lane's two column pairs (n-tile 0 / 1), or zero.
template <int C, int PX, int MT, typename RowFn>
__device__ __forceinline__ void warp_gemm(float (&acc)[MT][2][4], int n_mt, uint32_t a_base, RowFn a_row, uint32_t w_base,
                                          int npair, int lane, float2 init0 = make_float2(0.f, 0.f),
                                          float2 init1 = make_float2(0.f, 0.f)) {
#pragma unroll
  for (int i = 0; i < MT; ++i) {
    acc[i][0][0] = acc[i][0][2] = init0.x; acc[i][0][1] = acc[i][0][3] = init0.y;
    acc[i][1][0] = acc[i][1][2] = init1.x; acc[i][1][1] = acc[i][1][3] = init1.y;
  }
  // B: matrices (n 0-7, k 0-7) (n 0-7, k 8-15) (n 8-15, k 0-7) (n 8-15, k 8-15)
  const int bm = lane >> 3;
  const uint32_t b_addr0 = w_base + (uint32_t)(((npair * 16 + (bm >> 1) * 8 + (lane & 7)) * PX + (bm & 1) * 8) * 2);
#pragma unroll 4
  for (int kk = 0; kk < C / 16; ++kk) {
    uint32_t b[4];
    ldsm_x4(b, b_addr0 + (uint32_t)(kk * 32));
#pragma unroll
    for (int i = 0; i < MT; ++i) {
      if (i < n_mt) {
        uint32_t a[4];
        ldsm_x4(a, a_base + (uint32_t)((a_row(i, lane & 15) * PX + kk * 16 + (lane >> 4) * 8) * 2));
        mma16816(acc[i][0], a, b[0], b[1]);
        mma16816(acc[i][1], a, b[2], b[3]);
      }
    }
  }
}

template <int C, int HD, int NT>
__global__ void __launch_bounds__(kThreadsF, C == 64 ? 2 : 1) attn_fused_kernel(const FusedAttnParams p) {
  using Cfg = FusedCfg<C, HD, NT>;
  constexpr int PX = Cfg::PX, PQ = Cfg::PQ, HG = Cfg::HG, KSTEPS = Cfg::KSTEPS, XROWS = Cfg::XROWS, NKEY = Cfg::NKEY;
  constexpr int NW = Cfg::NW;
  extern __shared__ __align__(16) uint8_t smem[];
  const uint32_t sb = (uint32_t)__cvta_generic_to_shared(smem);
  __nv_bfloat16* xn = reinterpret_cast<__nv_bfloat16*>(smem + Cfg::OFF_XN);
  float* tbl_s = reinterpret_cast<float*>(smem + Cfg::OFF_TBL);
  __nv_bfloat16* qs = reinterpret_cast<__nv_bfloat16*>(smem + Cfg::OFF_Q);
  __nv_bfloat16* ks = reinterpret_cast<__nv_bfloat16*>(smem + Cfg::OFF_K);
  __nv_bfloat16* vs = reinterpret_cast<__nv_bfloat16*>(smem + Cfg::OFF_V);
  int* coff = reinterpret_cast<int*>(smem + Cfg::OFF_COFF);
  int* roff = reinterpret_cast<int*>(smem + Cfg::OFF_ROFF);
  int* pix_s = reinterpret_cast<int*>(smem + Cfg::OFF_PIX);

  const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const bool dbg = p.dbg != nullptr;
  const long long t_begin = dbg ? clock64() : 0;
  long long t_mark = t_begin, t_ln = 0, t_qkv = 0, t_tbl = 0, t_attn = 0;
  constexpr int NHG = C / 64;
  const int hg = (int)(blockIdx.x % NHG);
  const int w = (int)(blockIdx.x / NHG);
  const int n_kv = p.D * kTok;
  const int tbl_ld = p.D * kRel;

  pdl_trigger();   // the next kernel of the chain may start its prologue
  // ---- weight slices (q, k, v rows of this head group) -> smem, asynchronously ----------------------
  auto load_w_slice = [&](int which, int buf) {  // which: 0 = q, 1 = k, 2 = v
    const __nv_bfloat16* src = p.wqkv + (size_t)(which * C + hg * 64) * C;
    const uint32_t dst = sb + Cfg::OFF_W + (uint32_t)(buf * 64 * PX * 2);
    for (int i = tid; i < 64 * (C / 8); i += kThreadsF) {
      const int r = i / (C / 8), ch = i - r * (C / 8);
      cpa16(dst + (uint32_t)((r * PX + ch * 8) * 2), src + (size_t)r * C + ch * 8);
    }
    cpa_commit();
  };
#pragma unroll
  for (int i = 0; i < NW; ++i) load_w_slice(i, i);

  // ---- index tables -----------------------------------------------------------------------------------
  for (int n = tid; n < NKEY; n += kThreadsF) {
    int v = 0;  // padding keys read entry 0 and are masked in the last key tile
    if (n < n_kv) {
      const int d = n / kTok, r = n - d * kTok, a = r / 7, b = r - a * 7;
      v = d * kRel + (6 - a) * 13 + (6 - b);
    }
    coff[n] = v * 4;
  }
  if (tid < 64) {
    const int a = tid / 7, b = tid - a * 7;
    roff[tid] = tid < kTok ? (a * 13 + b) * 4 : 0;
  }
  if (tid < 64) pix_s[tid] = tid < kTok ? __ldg(p.tok_map + (size_t)w * kTok + tid) : -1;
  __syncthreads();
  pdl_wait();   // everything above is static data; the frames below were written by the previous kernel of the chain

  // ---- gather + LayerNorm: 8 lanes per token, 4 tokens per warp pass ----------------------------------
  // The loads of NB passes are issued together (independent global reads in flight) before any of them is reduced.
  {
    constexpr int NCH = C / 64;
    constexpr int NPASS = XROWS / 32;             // passes per warp (XROWS = 64, 112 or 160 -> 2, 3.5, 5)
    constexpr int NB = C == 64 ? 5 : 2;           // passes batched (register budget: NB * NCH * 8 floats)
    const int j = lane & 7, sub = lane >> 3;
    for (int pb = 0; pb * 32 * NB < XROWS; ++pb) {
      float v[NB][NCH][8];
      int nn[NB];
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const int n = (pb * NB + b) * 32 + warp * 4 + sub;
        nn[b] = n;
        const float* src = nullptr;
        if (n < n_kv) {
          const int d = n / kTok, tok = n - d * kTok;
          const int pix = pix_s[tok];
          const float* fr = p.frames[0];
#pragma unroll
          for (int q = 1; q < 8; ++q) fr = (d == q) ? p.frames[q] : fr;
          if (fr != nullptr && pix >= 0) src = fr + (size_t)pix * C + j * 8;
        }
#if BDE_ATTN_PROBE & 8
        src = nullptr;
#endif
#pragma unroll
        for (int kb = 0; kb < NCH; ++kb) {
          if (src != nullptr) {
            const float4 t0 = *(reinterpret_cast<const float4*>(src + kb * 64));
            const float4 t1 = *(reinterpret_cast<const float4*>(src + kb * 64 + 4));
            v[b][kb][0] = t0.x; v[b][kb][1] = t0.y; v[b][kb][2] = t0.z; v[b][kb][3] = t0.w;
            v[b][kb][4] = t1.x; v[b][kb][5] = t1.y; v[b][kb][6] = t1.z; v[b][kb][7] = t1.w;
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[b][kb][e] = 0.f;
          }
        }
      }
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        if (nn[b] >= XROWS) continue;   // warp-uniform up to the 4-token granularity of XROWS (a multiple of 16)
        float sum = 0.f;
#pragma unroll
        for (int kb = 0; kb < NCH; ++kb)
#pragma unroll
          for (int e = 0; e < 8; ++e) sum += v[b][kb][e];
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        sum += __shfl_xor_sync(0xffffffffu, sum, 4);
        const float mean = sum / (float)C;
        float sq = 0.f;
#pragma unroll
        for (int kb = 0; kb < NCH; ++kb)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float dlt = v[b][kb][e] - mean;
            v[b][kb][e] = dlt;
            sq += dlt * dlt;
          }
        sq += __shfl_xor_sync(0xffffffffu, sq, 1);
        sq += __shfl_xor_sync(0xffffffffu, sq, 2);
        sq += __shfl_xor_sync(0xffffffffu, sq, 4);
        const float rstd = rsqrt_approx(sq / (float)C + 1e-5f);
#pragma unroll
        for (int kb = 0; kb < NCH; ++kb) {
          uint4 pk;
          pk.x = pack2(v[b][kb][0] * rstd, v[b][kb][1] * rstd);
          pk.y = pack2(v[b][kb][2] * rstd, v[b][kb][3] * rstd);
          pk.z = pack2(v[b][kb][4] * rstd, v[b][kb][5] * rstd);
          pk.w = pack2(v[b][kb][6] * rstd, v[b][kb][7] * rstd);
          *reinterpret_cast<uint4*>(xn + (size_t)nn[b] * PX + kb * 64 + j * 8) = pk;
        }
      }
    }
    (void)NPASS;
  }

  if (dbg) { const long long c = clock64(); t_ln = c - t_mark; t_mark = c; }
  // ---- q, k, v projections (mma.sync): warp = (n-tile pair, m half) --------------------------------------
  const int npair = warp & 3, mh = warp >> 2;
  const uint32_t xn_u32 = sb + Cfg::OFF_XN;
  constexpr int MTK = (KSTEPS + 1) / 2;  // k / v m-tiles per warp
  if (NW == 3) {  // all three weight slices were loaded up front: one barrier covers them and the LayerNorm'ed tokens
    cpa_wait<0>();
    __syncthreads();
  }
  for (int which = 0; which < ((BDE_ATTN_PROBE & 16) ? 0 : 3); ++which) {
    if (NW != 3) {
      // slices were committed in order: wait until slice `which` has landed
      if (which == 2) cpa_wait<0>(); else cpa_wait<1>();
      __syncthreads();  // slice + (first pass) the LayerNorm'ed tokens visible to every warp
    }
    const uint32_t w_base = sb + Cfg::OFF_W + (uint32_t)((which % NW) * 64 * PX * 2);
    const float* bsrc = p.bqkv + which * C + hg * 64 + npair * 16 + 2 * t;
    const float2 bia0 = __ldg(reinterpret_cast<const float2*>(bsrc));
    const float2 bia1 = __ldg(reinterpret_cast<const float2*>(bsrc + 8));
    if (which == 0) {
      // q: the 49 tokens of the query slot (4 m-tiles, 2 per warp); rows past the staged block are clamped
      float acc[2][2][4];
      const int qrow0 = p.q_slot * kTok;
      warp_gemm<C, PX, 2>(acc, 2, xn_u32, [&](int i, int r) { return min(qrow0 + (mh * 2 + i) * 16 + r, XROWS - 1); }, w_base,
                          npair, lane, bia0, bia1);   // accumulators start at the bias
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int r0 = (mh * 2 + i) * 16 + g;
#pragma unroll
        for (int n = 0; n < 2; ++n) {
          const int col = npair * 16 + n * 8 + 2 * t;
          *reinterpret_cast<uint32_t*>(qs + r0 * PQ + col) = pack2(acc[i][n][0], acc[i][n][1]);
          *reinterpret_cast<uint32_t*>(qs + (r0 + 8) * PQ + col) = pack2(acc[i][n][2], acc[i][n][3]);
        }
      }
    } else {
      float acc[MTK][2][4];
      const int mt0 = mh * MTK;
      const int n_mt = min(MTK, KSTEPS - mt0);
      warp_gemm<C, PX, MTK>(acc, n_mt, xn_u32, [&](int i, int r) { return (mt0 + i) * 16 + r; }, w_base, npair, lane, bia0, bia1);
      __nv_bfloat16* dstm = which == 1 ? ks : vs;
      const int row_lim = which == 1 ? NKEY : XROWS;
#pragma unroll
      for (int i = 0; i < MTK; ++i) {
        if (i < n_mt) {
          const int r0 = (mt0 + i) * 16 + g;
#pragma unroll
          for (int n = 0; n < 2; ++n) {
            const int col = npair * 16 + n * 8 + 2 * t;
            // k stays bf16 (q.k^T is a bf16 product); v is stored as fp16 for the fp16 P.V product
            const float v00 = acc[i][n][0], v01 = acc[i][n][1], v10 = acc[i][n][2], v11 = acc[i][n][3];
            if (r0 < row_lim) *reinterpret_cast<uint32_t*>(dstm + r0 * PQ + col) = which == 1 ? pack2(v00, v01) : pack2_hs(v00, v01);
            if (r0 + 8 < row_lim)
              *reinterpret_cast<uint32_t*>(dstm + (r0 + 8) * PQ + col) = which == 1 ? pack2(v10, v11) : pack2_hs(v10, v11);
          }
        }
      }
    }
    if (which + NW < 3) {
      __syncthreads();  // every warp is done reading buffer which % NW
      load_w_slice(which + NW, which % NW);
    }
  }
  __syncthreads();  // q, k, v complete; the token / weight region is free
  if (dbg) { const long long c = clock64(); t_qkv = c - t_mark; t_mark = c; }

  // ---- bias table (+ projection weights) -> smem ------------------------------------------------------------
  {
    const float* src = p.tbl + (size_t)hg * HG * tbl_ld;
    const int n16 = HG * tbl_ld / 4;  // 16-byte chunks (HG * D * 169 floats; multiple of 4 because HG is)
    for (int i = tid; i < n16; i += kThreadsF) cpa16(sb + Cfg::OFF_TBL + (uint32_t)(i * 16), src + i * 4);
    if (C == 64) {
      for (int i = tid; i < 64 * (C / 8); i += kThreadsF) {
        const int r = i / (C / 8), ch = i - r * (C / 8);
        cpa16(sb + Cfg::OFF_WP + (uint32_t)((r * PX + ch * 8) * 2), p.wproj + (size_t)r * C + ch * 8);
      }
    }
    cpa_commit();
    cpa_wait<0>();
    __syncthreads();
  }

  if (dbg) { const long long c = clock64(); t_tbl = c - t_mark; t_mark = c; }
  // ---- attention: unit = (head of the group, 16-row query tile); scores stay in registers ----------------------
  // head_dim 4: the 49th query row would cost a whole tile per head, so the normal units cover rows 0..47 and one
  // "special" unit packs row 48 of all 16 heads into a single tile (tile row = head; the query fragment carries only
  // that head's 4 channels, the key fragment all 64, so each row still sees its own head's dot product).
  const uint32_t vs_u32 = sb + Cfg::OFF_V;
  const uint32_t tbl_u32 = sb + Cfg::OFF_TBL;
  const uint32_t coff_u32 = sb + Cfg::OFF_COFF;
  __nv_bfloat16* os = reinterpret_cast<__nv_bfloat16*>(smem + Cfg::OFF_OS);  // C == 64 only
  constexpr int MTN = HD == 4 ? 3 : 4;                 // query tiles per head handled by normal units
  constexpr int NUNITS = HG * MTN;
  constexpr uint32_t kOnes = 0x3C003C00u;              // fp16x2 (1, 1)
  constexpr float kLog2e = 1.4426950408889634f;
  if (HD == 4) {
    // ---- head_dim 4, normal units: TWO units per warp in flight, softmax over three key segments ------------------------
    // The unit is a long dependent chain (bias + QK^T -> row max -> exp -> P.V) and only 16 warps fit on an SM, so the
    // kernel was issue-latency bound (warps active 24 %, no pipe above 60 %).  Interleaving two independent units doubles
    // the instruction-level parallelism per warp; the online softmax over three key segments (6 / 6 / 7 tiles for D = 3)
    // keeps 2 x 7 score tiles alive instead of 2 x 19, so both fit the 128-register budget of two CTAs per SM.
    // The two units of a warp are the SAME query tile of heads h and h + 8: bias row / column offsets, the ones-lane pattern
    // and every shared-memory base address are then shared, and the second head's operands sit at compile-time byte
    // offsets (bias table +8 rows of D * 169 floats, q / k / v columns +32 channels) -> half the address arithmetic.
    constexpr int NPAIRS = HG * MTN / 2;                          // 24 pairs: (head pair, 16-row query tile)
    constexpr int TLD = Cfg::DMAX * kRel;                         // == tbl_ld: launch_fused picks NT from D
    constexpr int kTblOff = 8 * TLD * 4;                          // bias table: head h -> h + 8
    constexpr int kChOff = 8 * HD * 2;                            // q / k / v tiles: head h -> h + 8 (bf16 / fp16 columns)
    constexpr int SEG = ((NT + 2) / 3) & ~1;                      // even segment size: 19 -> 6, 13 -> 4, 7 -> 2
    constexpr int LAST = NT - 2 * SEG;                            // 7 / 5 / 3
    constexpr int kMaxT = LAST > SEG ? LAST : SEG;
    for (int pi = warp; pi < ((BDE_ATTN_PROBE & 4) ? 0 : NPAIRS); pi += kThreadsF / 32) {
      const int hp = pi / MTN, mt = pi - hp * MTN;                // heads hp and hp + 8
      const int row0 = mt * 16 + g, row1 = row0 + 8;
      const uint32_t r0a = tbl_u32 + (uint32_t)(hp * TLD * 4 + roff[row0]);
      const uint32_t r1a = tbl_u32 + (uint32_t)(hp * TLD * 4 + roff[row1]);
      uint32_t qa0[2] = {0u, 0u}, qa1[2] = {0u, 0u};
      if (2 * t < HD) {
        const __nv_bfloat16* q0 = qs + row0 * PQ + hp * HD + 2 * t;
        const __nv_bfloat16* q1 = qs + row1 * PQ + hp * HD + 2 * t;
        qa0[0] = *reinterpret_cast<const uint32_t*>(q0); qa0[1] = *reinterpret_cast<const uint32_t*>(q0 + 8 * HD);
        qa1[0] = *reinterpret_cast<const uint32_t*>(q1); qa1[1] = *reinterpret_cast<const uint32_t*>(q1 + 8 * HD);
      }
      // one 8-channel V tile holds a head pair (2 hp', 2 hp' + 1); the other head's columns are replaced by ones -> row sums
      const bool ones_lane = (g >> 2) != (hp & 1);
      const uint32_t vaddr = vs_u32 + (uint32_t)(((lane & 15) * PQ + (hp >> 1) * 8) * 2);
      const __nv_bfloat16* kp = ks + g * PQ + hp * HD + 2 * t;
      float oa[2][4], ob[2][4], m0s[2], m1s[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        oa[u][0] = oa[u][1] = oa[u][2] = oa[u][3] = 0.f;
        ob[u][0] = ob[u][1] = ob[u][2] = ob[u][3] = 0.f;
        m0s[u] = m1s[u] = -INFINITY;                              // running row maxima times log2(e)
      }
#pragma unroll
      for (int seg = 0; seg < 3; ++seg) {
        const int j0 = seg * SEG, nj = seg < 2 ? SEG : LAST;
        float s[2][kMaxT][4];
#pragma unroll
        for (int jj = 0; jj < kMaxT; ++jj) {
          if (jj < nj) {
            const int j = j0 + jj;
#if BDE_ATTN_PROBE & 1
            s[0][jj][0] = s[0][jj][1] = s[0][jj][2] = s[0][jj][3] = 0.f;
            s[1][jj][0] = s[1][jj][1] = s[1][jj][2] = s[1][jj][3] = 0.f;
#else
            const uint2 cp = lds_u64(coff_u32 + (uint32_t)((j * 8 + 2 * t) * 4));
            const uint32_t a00 = r0a + cp.x, a01 = r0a + cp.y, a10 = r1a + cp.x, a11 = r1a + cp.y;
            s[0][jj][0] = lds_f32_off<0>(a00); s[0][jj][1] = lds_f32_off<0>(a01);
            s[0][jj][2] = lds_f32_off<0>(a10); s[0][jj][3] = lds_f32_off<0>(a11);
            s[1][jj][0] = lds_f32_off<kTblOff>(a00); s[1][jj][1] = lds_f32_off<kTblOff>(a01);
            s[1][jj][2] = lds_f32_off<kTblOff>(a10); s[1][jj][3] = lds_f32_off<kTblOff>(a11);
#endif
            uint32_t kb[2] = {0u, 0u};
            if (2 * t < HD) {
              kb[0] = *reinterpret_cast<const uint32_t*>(kp + j * 8 * PQ);
              kb[1] = *reinterpret_cast<const uint32_t*>(kp + j * 8 * PQ + 8 * HD);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              if (j == NT - 1) {  // only the last key tile can hold padding keys
                if (j * 8 + 2 * t >= n_kv) s[u][jj][0] = s[u][jj][2] = -1e30f;
                if (j * 8 + 2 * t + 1 >= n_kv) s[u][jj][1] = s[u][jj][3] = -1e30f;
              }
              mma1688(s[u][jj], qa0[u], qa1[u], kb[u]);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
          for (int jj = 0; jj < kMaxT; ++jj) {
            if (jj < nj) {
              mx0 = fmaxf(mx0, fmaxf(s[u][jj][0], s[u][jj][1]));
              mx1 = fmaxf(mx1, fmaxf(s[u][jj][2], s[u][jj][3]));
            }
          }
          mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
          mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
          mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
          mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
          const float n0s = fmaxf(m0s[u], mx0 * kLog2e), n1s = fmaxf(m1s[u], mx1 * kLog2e);
          if (seg > 0) {   // rescale what the earlier segments accumulated (values and ones-column row sums alike)
            float c0, c1;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(c0) : "f"(m0s[u] - n0s));
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(c1) : "f"(m1s[u] - n1s));
            oa[u][0] = (oa[u][0] + ob[u][0]) * c0; oa[u][1] = (oa[u][1] + ob[u][1]) * c0;
            oa[u][2] = (oa[u][2] + ob[u][2]) * c1; oa[u][3] = (oa[u][3] + ob[u][3]) * c1;
            ob[u][0] = ob[u][1] = ob[u][2] = ob[u][3] = 0.f;
          }
          m0s[u] = n0s; m1s[u] = n1s;
        }
#pragma unroll
        for (int k2 = 0; k2 < (kMaxT + 1) / 2; ++k2) {
          if (2 * k2 < nj) {
            const int kk = j0 / 2 + k2;
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              uint32_t pa[4];
              pa[0] = ex2_h2(fmaf(s[u][2 * k2][0], kLog2e, -m0s[u]), fmaf(s[u][2 * k2][1], kLog2e, -m0s[u]));
              pa[1] = ex2_h2(fmaf(s[u][2 * k2][2], kLog2e, -m1s[u]), fmaf(s[u][2 * k2][3], kLog2e, -m1s[u]));
              if (2 * k2 + 1 < nj) {
                pa[2] = ex2_h2(fmaf(s[u][2 * k2 + 1][0], kLog2e, -m0s[u]), fmaf(s[u][2 * k2 + 1][1], kLog2e, -m0s[u]));
                pa[3] = ex2_h2(fmaf(s[u][2 * k2 + 1][2], kLog2e, -m1s[u]), fmaf(s[u][2 * k2 + 1][3], kLog2e, -m1s[u]));
              } else {
                pa[2] = pa[3] = 0u;
              }
              uint32_t vb0, vb1;
              ldsm_x2_trans(vb0, vb1, vaddr + (uint32_t)(kk * 16 * PQ * 2 + u * kChOff));
              if (ones_lane) { vb0 = kOnes; vb1 = kOnes; }
              if (k2 & 1) mma16816_f16(ob[u], pa, vb0, vb1); else mma16816_f16(oa[u], pa, vb0, vb1);
            }
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
#pragma unroll
        for (int e = 0; e < 4; ++e) oa[u][e] += ob[u][e];
        const float l0 = __shfl_xor_sync(0xffffffffu, oa[u][0], 2), l1 = __shfl_xor_sync(0xffffffffu, oa[u][2], 2);
        if ((t >> 1) == (hp & 1)) {
          const float inv0 = rcp_approx(l0), inv1 = rcp_approx(l1);
          const int col = ((hp + 8 * u) >> 1) * 8 + 2 * t;
          *reinterpret_cast<uint32_t*>(os + row0 * PQ + col) = pack2(oa[u][0] * inv0, oa[u][1] * inv0);
          *reinterpret_cast<uint32_t*>(os + row1 * PQ + col) = pack2(oa[u][2] * inv1, oa[u][3] * inv1);
        }
      }
    }
  }
  if (HD == 4) {
    // ---- query token 48 of all 16 heads on the CUDA cores: warp = two heads, 16 lanes per head, keys strided over lanes ----
    // (As a 49th tensor-core unit this row cost one warp ~1000 instructions while the other seven waited at the barrier
    // below: 10 % of the kernel's warp-time in the round-2 profile.  Spread over every lane it is ~300 per warp.)
    const int h = warp * 2 + (lane >> 4), sl = lane & 15;
    float qf[4];
    {
      const uint2 qr = *reinterpret_cast<const uint2*>(qs + 48 * PQ + h * 4);
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qr.x));
      const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qr.y));
      qf[0] = a.x; qf[1] = a.y; qf[2] = b.x; qf[3] = b.y;
    }
    const uint32_t ra = tbl_u32 + (uint32_t)(h * tbl_ld * 4 + roff[48]);
    constexpr int NI = (NKEY + 15) / 16;
    float sv[NI];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int n = sl + 16 * i;
      sv[i] = -INFINITY;
      if (n < n_kv) {
        const uint2 kr = *reinterpret_cast<const uint2*>(ks + n * PQ + h * 4);
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&kr.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&kr.y));
        float acc = lds_f32(ra + (uint32_t)coff[n]);
        acc = fmaf(qf[0], a.x, acc); acc = fmaf(qf[1], a.y, acc); acc = fmaf(qf[2], b.x, acc); acc = fmaf(qf[3], b.y, acc);
        sv[i] = acc;
      }
      mx = fmaxf(mx, sv[i]);
    }
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float ms = mx * kLog2e;   // every lane owns at least three real keys (n_kv >= 49), so mx is finite
    float l = 0.f, o4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int n = sl + 16 * i;
      if (n < n_kv) {
        float pr;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(pr) : "f"(fmaf(sv[i], kLog2e, -ms)));
        const uint2 vr = *reinterpret_cast<const uint2*>(vs + n * PQ + h * 4);   // fp16 x 4
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&vr.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&vr.y));
        l += pr;
        o4[0] = fmaf(pr, a.x, o4[0]); o4[1] = fmaf(pr, a.y, o4[1]); o4[2] = fmaf(pr, b.x, o4[2]); o4[3] = fmaf(pr, b.y, o4[3]);
      }
    }
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
      l += __shfl_xor_sync(0xffffffffu, l, o);
#pragma unroll
      for (int e = 0; e < 4; ++e) o4[e] += __shfl_xor_sync(0xffffffffu, o4[e], o);
    }
    if (sl == 0) {
      const float inv = rcp_approx(l);
      uint2 pk;
      pk.x = pack2(o4[0] * inv, o4[1] * inv);
      pk.y = pack2(o4[2] * inv, o4[3] * inv);
      *reinterpret_cast<uint2*>(os + 48 * PQ + h * 4) = pk;
    }
  }
  for (int unit = HD == 4 ? NUNITS : warp; unit < NUNITS; unit += kThreadsF / 32) {   // head_dim >= 8 (C == 256) only
    const int hl = unit / MTN, mt = unit - hl * MTN;
    const int row0 = mt * 16 + g, row1 = row0 + 8;
    float s[NT][4];
    {
      const uint32_t r0a = tbl_u32 + (uint32_t)(hl * tbl_ld * 4 + roff[row0]);
      const uint32_t r1a = tbl_u32 + (uint32_t)(hl * tbl_ld * 4 + roff[row1]);
      uint32_t qa[4] = {0u, 0u, 0u, 0u};
      {
        const __nv_bfloat16* q0 = qs + row0 * PQ + hl * HD;
        const __nv_bfloat16* q1 = qs + row1 * PQ + hl * HD;
        if (2 * t < HD) {
          qa[0] = *reinterpret_cast<const uint32_t*>(q0 + 2 * t);
          qa[1] = *reinterpret_cast<const uint32_t*>(q1 + 2 * t);
        }
        if (2 * t + 8 < HD) {
          qa[2] = *reinterpret_cast<const uint32_t*>(q0 + 2 * t + 8);
          qa[3] = *reinterpret_cast<const uint32_t*>(q1 + 2 * t + 8);
        }
      }
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        const uint2 cp = lds_u64(coff_u32 + (uint32_t)((j * 8 + 2 * t) * 4));
        s[j][0] = lds_f32(r0a + cp.x); s[j][1] = lds_f32(r0a + cp.y);
        s[j][2] = lds_f32(r1a + cp.x); s[j][3] = lds_f32(r1a + cp.y);
        if (j == NT - 1) {  // only the last key tile can hold padding keys
          if (j * 8 + 2 * t >= n_kv) s[j][0] = s[j][2] = -1e30f;
          if (j * 8 + 2 * t + 1 >= n_kv) s[j][1] = s[j][3] = -1e30f;
        }
        const __nv_bfloat16* kr = ks + (j * 8 + g) * PQ + hl * HD;
        uint32_t kb0 = 0u, kb1 = 0u;
        if (2 * t < HD) kb0 = *reinterpret_cast<const uint32_t*>(kr + 2 * t);
        if (2 * t + 8 < HD) kb1 = *reinterpret_cast<const uint32_t*>(kr + 2 * t + 8);
        mma16816(s[j], qa, kb0, kb1);
      }
    }
    // ---- softmax numerators (the row sums come out of the P.V product through a column of ones) -------------------
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
      mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float m0s = mx0 * kLog2e, m1s = mx1 * kLog2e;
    uint32_t pp[NT][2];   // P as fp16 pairs: [j][0] = row0 (cols 2t, 2t+1), [j][1] = row1
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      pp[j][0] = ex2_h2(fmaf(s[j][0], kLog2e, -m0s), fmaf(s[j][1], kLog2e, -m0s));
      pp[j][1] = ex2_h2(fmaf(s[j][2], kLog2e, -m1s), fmaf(s[j][3], kLog2e, -m1s));
    }
    constexpr int NV = HD >= 8 ? HD / 8 : 1;
    float o[NV][4], ol[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int v = 0; v < NV; ++v) o[v][0] = o[v][1] = o[v][2] = o[v][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < KSTEPS; ++kk) {
      uint32_t pa[4];
      pa[0] = pp[2 * kk][0];
      pa[1] = pp[2 * kk][1];
      pa[2] = 2 * kk + 1 < NT ? pp[2 * kk + 1][0] : 0u;
      pa[3] = 2 * kk + 1 < NT ? pp[2 * kk + 1][1] : 0u;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        uint32_t vb0, vb1;
        ldsm_x2_trans(vb0, vb1, vs_u32 + (uint32_t)(((kk * 16 + (lane & 15)) * PQ + hl * HD + 8 * v) * 2));
        mma16816_f16(o[v], pa, vb0, vb1);
      }
      mma16816_f16(ol, pa, kOnes, kOnes);   // row sums
    }
    const float inv0 = 1.0f / ol[0], inv1 = 1.0f / ol[2];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int col = hl * HD + 8 * v + 2 * t;
      const uint32_t v0 = pack2(o[v][0] * inv0, o[v][1] * inv0), v1 = pack2(o[v][2] * inv1, o[v][3] * inv1);
      if (C == 64) {
        *reinterpret_cast<uint32_t*>(os + row0 * PQ + col) = v0;
        *reinterpret_cast<uint32_t*>(os + row1 * PQ + col) = v1;
      } else {
        __nv_bfloat16* og = p.o_out + (size_t)w * kTok * C + hg * 64 + col;
        if (row0 < kTok) *reinterpret_cast<uint32_t*>(og + (size_t)row0 * C) = v0;
        if (row1 < kTok) *reinterpret_cast<uint32_t*>(og + (size_t)row1 * C) = v1;
      }
    }
  }

  if (dbg) { const long long c = clock64(); t_attn = c - t_mark; t_mark = c; }
  if (C == 64 && !(BDE_ATTN_PROBE & 32)) {
    // ---- output projection + window_reverse + shortcut: x[pix] += proj(o) + b (DTransformer.py:204,294-299) ----
    // shortcut = the query frame (DTransformer.py:294-299; xs itself when the block runs in place): this thread's eight
    // float2 values are fetched BEFORE the projection GEMM -- inside the store loop every load waited behind the previous
    // store (xs and the frame may alias), eight global round trips in a row
    const float* shortcut = p.frames[p.q_slot];
    float2 sc[2][2][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int r = (mh * 2 + i) * 16 + g + hrow * 8;
        const int pix = r < kTok ? pix_s[r] : -1;
#pragma unroll
        for (int n = 0; n < 2; ++n)
          sc[i][hrow][n] = pix >= 0 ? *(reinterpret_cast<const float2*>(shortcut + (size_t)pix * C + npair * 16 + n * 8 + 2 * t))
                                    : make_float2(0.f, 0.f);
      }
    __syncthreads();
    float acc[2][2][4];
    warp_gemm<C, PQ, 2>(acc, 2, sb + Cfg::OFF_OS, [&](int i, int r) { return (mh * 2 + i) * 16 + r; }, sb + Cfg::OFF_WP, npair, lane);
    // note: os has pitch PQ == PX for C == 64, so the same routine serves both operands
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        const int r = (mh * 2 + i) * 16 + g + hrow * 8;
        const int pix = r < kTok ? pix_s[r] : -1;
        if (pix >= 0) {
#pragma unroll
          for (int n = 0; n < 2; ++n) {
            const int col = npair * 16 + n * 8 + 2 * t;
            const float2 bb = __ldg(reinterpret_cast<const float2*>(p.bproj + col));
            float2 cur = sc[i][hrow][n];
            cur.x += acc[i][n][hrow * 2 + 0] + bb.x;
            cur.y += acc[i][n][hrow * 2 + 1] + bb.y;
            *reinterpret_cast<float2*>(p.xs + (size_t)pix * C + col) = cur;
          }
        }
      }
    }
  }
  if (dbg && tid == 0) {
    long long* o = p.dbg + (size_t)blockIdx.x * 8;
    const long long c = clock64();
    o[0] = c - t_begin; o[1] = t_ln; o[2] = 0; o[3] = t_qkv; o[4] = t_tbl; o[5] = t_attn; o[6] = c - t_mark;
  }
}

template <int C, int HD, int NT>
int launch_fused(const FusedAttnParams& p, cudaStream_t s) {
  using Cfg = FusedCfg<C, HD, NT>;
  static_assert(C != 64 || Cfg::PQ == Cfg::PX, "C == 64 shares one pitch between token and q/k/v tiles");
  auto kern = attn_fused_kernel<C, HD, NT>;
  if (first_use_on_device((const void*)kern)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    BDE_REQUIRE(e == cudaSuccess, "bde_window_attention_fused: smem attribute (%d bytes): %s", Cfg::SMEM, cudaGetErrorString(e));
  }
  FusedAttnParams q = p;
  q.dbg = (tc::g_dbg != nullptr && (size_t)p.n_win * (C / 64) <= tc::g_dbg_ctas) ? tc::g_dbg : nullptr;
  const cudaError_t le = launch_pdl(kern, (unsigned)(p.n_win * (C / 64)), (unsigned)kThreadsF, (size_t)Cfg::SMEM, s, 1, q);
  BDE_REQUIRE(le == cudaSuccess, "bde_window_attention_fused: launch: %s", cudaGetErrorString(le));
  return check_launch("attn_fused_kernel");
}

}  // namespace
}  // namespace bde

using namespace bde;

extern "C" int bde_window_attention_fused_supported(int c, int heads, int n_tok, int D) {
  if (n_tok != kTok || D < 1 || D > 3 || heads <= 0 || c % heads != 0) return 0;
  const int hd = c / heads;
  return ((c == 64 && hd == 4) || (c == 256 && hd == 16)) ? 1 : 0;
}

extern "C" int bde_window_attention_fused(const float* const* frames_host, int D, int q_slot, const int* tok_map, int n_win,
                                          int c, int heads, const void* wqkv, const float* bqkv, const float* bias_tbl,
                                          const void* wproj, const float* bproj, float* xs, void* o_out, void* stream) {
  if (n_win == 0) return 0;
  BDE_REQUIRE(bde_window_attention_fused_supported(c, heads, kTok, D) == 1,
              "bde_window_attention_fused: unsupported shape (c=%d heads=%d D=%d)", c, heads, D);
  BDE_REQUIRE(q_slot >= 0 && q_slot < D && frames_host != nullptr && tok_map != nullptr && wqkv != nullptr && bqkv != nullptr &&
                  bias_tbl != nullptr,
              "bde_window_attention_fused: bad arguments");
  const bool with_proj = wproj != nullptr && bproj != nullptr && xs != nullptr;
  BDE_REQUIRE(!with_proj || frames_host[q_slot] != nullptr, "bde_window_attention_fused: the query frame (shortcut source) must not be NULL");
  BDE_REQUIRE(c == 64 ? with_proj : (with_proj || o_out != nullptr), "bde_window_attention_fused: missing output operands");
  BDE_REQUIRE((((uintptr_t)wqkv) & 15) == 0 && (((uintptr_t)bias_tbl) & 15) == 0 && (((uintptr_t)wproj) & 15) == 0,
              "bde_window_attention_fused: operands must be 16-byte aligned");
  FusedAttnParams p;
  for (int i = 0; i < 8; ++i) p.frames[i] = i < D ? frames_host[i] : nullptr;
  p.tok_map = tok_map;
  p.wqkv = (const __nv_bfloat16*)wqkv;
  p.bqkv = bqkv;
  p.tbl = bias_tbl;
  p.wproj = (const __nv_bfloat16*)wproj;
  p.bproj = bproj;
  p.xs = xs;
  p.o_out = (__nv_bfloat16*)o_out;
  p.n_win = n_win; p.D = D; p.q_slot = q_slot; p.heads = heads;
  p.dbg = nullptr;
  cudaStream_t s = (cudaStream_t)stream;
#define BDE_FUSED(C_, HD_)                                       \
  switch (D) {                                                   \
    case 1: return launch_fused<C_, HD_, 7>(p, s);               \
    case 2: return launch_fused<C_, HD_, 13>(p, s);              \
    default: return launch_fused<C_, HD_, 19>(p, s);             \
  }
  if (c == 64) BDE_FUSED(64, 4)
  // c == 256 with the projection fused: whole-window kernel, projections on tcgen05 (attn_tc256.cu; it refuses weights
  // that are not 128-byte aligned)
  if (with_proj)
    return tc::attn_win256_tc_launch(frames_host, D, q_slot, tok_map, n_win, wqkv, bqkv, bias_tbl, wproj, bproj, xs, s);
  BDE_FUSED(256, 16)
#undef BDE_FUSED
}
