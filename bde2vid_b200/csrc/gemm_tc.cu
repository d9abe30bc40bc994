// tcgen05 implicit-GEMM engine (bf16 operands, fp32 accumulation in TMEM) for sm_100a.
//
//   C[m, n] = sum_k A[m, k] * W[n, k]      m = (img, oy, ox),  k = (tap, channel)
//
// One CTA computes a 128 x BN output tile.  Warp roles (320 threads):
//   warps 0-7  A producers.  8 consecutive lanes fetch the 8 16-byte chunks of one 128-byte im2col
//              row (cp.async, zero fill for padding / K tail / M tail) into the 128B-swizzled
//              K-major layout UMMA expects, so a warp-wide copy touches 4 full cache lines.
//              Everything that depends only on the output pixel (base index, per-tap validity
//              mask) is computed once; the per-K-block work is a handful of integer ops per row.
//              After the main loop the same warps run the epilogue (warp w <-> TMEM lanes
//              32*(w&3).., column half w>>2).
//   warp 8     B producer: one thread issues a TMA 2D tiled load (SWIZZLE_128B) of the
//              [BN x 64] weight tile per K block.  (kBTma=false: cp.async gather, for bring-up.)
//   warp 9     MMA issuer: one thread issues 4 x tcgen05.mma (M128 x BN x K16) per K block and
//              commits to the stage's "empty" barrier; owns the TMEM allocation.
// Pipelines: smem full/empty mbarriers per stage, one "accumulator ready" mbarrier.
// Epilogues are fused: bias + activation (+ fp32 residual), ConvLSTM gate math, window scatter.
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <tuple>

#include "tc_common.cuh"

namespace bde {
namespace tc {

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
// two CTAs per SM wherever the tile's shared memory allows it (the register allocation must then fit 640 threads)
template <int BN, bool kDeep, int kLn>
constexpr int kMinCtas = TileCfg<BN, kDeep, kLn>::kSmemBytes <= 113 * 1024 ? 2 : 1;

template <int BN, bool kBTma, bool kDeep, int kLn>
__global__ void __launch_bounds__(kThreads, kMinCtas<BN, kDeep, kLn>) gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_b, const TcParams p) {
  using Cfg = TileCfg<BN, kDeep, kLn>;
  constexpr int S = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment is required by SWIZZLE_128B tiles
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;                       // S x [128 x 128B]
  const uint32_t smem_b = smem_base + S * Cfg::kABytes;    // S x [BN x 128B]
  const uint32_t bar_base = smem_base + Cfg::kOperandBytes;   // after the stages and the epilogue's staging
  const uint32_t bar_full = bar_base;                      // S x 8B
  const uint32_t bar_empty = bar_base + 8 * S;             // S x 8B
  const uint32_t bar_acc = bar_base + 16 * S;              // 8B
  const uint32_t tmem_slot = bar_base + 16 * S + 8;        // 4B
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));  // generic pointer to smem_base
  float* bias_s = reinterpret_cast<float*>(smem_gen + Cfg::kOperandBytes + 256);  // BN floats

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x, n0 = blockIdx.y * BN;
  const int num_kb = p.num_kb;

  if (threadIdx.x == 0) BDE_DBG(0);
  // bias slice -> smem once (the epilogue then never waits on global memory for it)
  if ((int)threadIdx.x < BN) bias_s[threadIdx.x] = p.bias != nullptr ? __ldg(p.bias + blockIdx.y * BN + threadIdx.x) : 0.0f;
  if (threadIdx.x == 0) {
    const uint32_t full_count = kNumProducerThreads + (kBTma ? 1 : 32);
    for (int s = 0; s < S; ++s) {
      mbar_init(bar_full + 8 * s, full_count);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_acc, 1);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));
  if (threadIdx.x == 0) BDE_DBG(1);
  TileGeom geom;
  geom.init(p, m_tile);

  if (warp < kNumProducerWarps) {
    // =============================== A producers ========================================
    // lane l owns 16-byte chunk j = l & 7 of rows warp*16 + 4*i + (l >> 3), i = 0..3
    const int j = lane & 7;
    const int rsub = lane >> 3;
    const int ntaps = p.ksize * p.ksize;
    if (kLn > 0) {
      // ---- LayerNorm-gather producer: fp32 rows -> normalised bf16 operand tile, all K blocks at once ----
      constexpr int nchunk = kLn > 0 ? kLn : 1;  // K blocks = pipeline stages (C = 64 * nchunk)
      constexpr int C = 64 * nchunk;
      // rows are independent: unroll so that several rows' loads are in flight (all 4 for C <= 128)
#pragma unroll(kLn <= 2 ? 4 : 2)
      for (int i = 0; i < kRowsPerThread; ++i) {
        const int row = warp * (4 * kRowsPerThread) + i * 4 + rsub;
        const uint32_t dst = (uint32_t)row * 128u + (((uint32_t)j ^ (uint32_t)(row & 7)) << 4);
        const int mm = geom.m0 + row;
        const float* src = nullptr;
        if (mm < p.M) {
          int pix = mm, d = 0;
          if (p.ln_map != nullptr) {
            const int tok = mm % p.ln_ntok;
            const int r2 = mm / p.ln_ntok;
            d = r2 % p.ln_D;
            pix = __ldg(p.ln_map + (r2 / p.ln_D) * p.ln_ntok + tok);
          }
          const float* fr = p.ln_f[0];
#pragma unroll
          for (int t = 1; t < 8; ++t) fr = (d == t) ? p.ln_f[t] : fr;
          if (fr != nullptr && pix >= 0) src = fr + (size_t)pix * C + j * 8;
        }
        float v[nchunk][8];
        float sum = 0.f;
#pragma unroll
        for (int kb = 0; kb < nchunk; ++kb) {
          if (src != nullptr) {
            const float4 t0 = *reinterpret_cast<const float4*>(src + kb * 64), t1 = *reinterpret_cast<const float4*>(src + kb * 64 + 4);
            v[kb][0] = t0.x; v[kb][1] = t0.y; v[kb][2] = t0.z; v[kb][3] = t0.w;
            v[kb][4] = t1.x; v[kb][5] = t1.y; v[kb][6] = t1.z; v[kb][7] = t1.w;
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[kb][e] = 0.f;
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) sum += v[kb][e];
        }
        // the 8 lanes of a row group (same rsub) reduce with xor 1, 2, 4
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        sum += __shfl_xor_sync(0xffffffffu, sum, 4);
        const float mean = sum / (float)C;
        float sq = 0.f;
#pragma unroll
        for (int kb = 0; kb < nchunk; ++kb)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float dlt = v[kb][e] - mean;
            v[kb][e] = dlt;
            sq += dlt * dlt;
          }
        sq += __shfl_xor_sync(0xffffffffu, sq, 1);
        sq += __shfl_xor_sync(0xffffffffu, sq, 2);
        sq += __shfl_xor_sync(0xffffffffu, sq, 4);
        const float rstd = 1.0f / sqrtf(sq / (float)C + 1e-5f);
#pragma unroll
        for (int kb = 0; kb < nchunk; ++kb) {
          {
            float o[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = v[kb][e] * rstd;
            const uint4 pk = pack8_bf16(o);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(smem_a + kb * Cfg::kABytes + dst), "r"(pk.x), "r"(pk.y),
                         "r"(pk.z), "r"(pk.w)
                         : "memory");
          }
        }
      }
      // generic-proxy stores -> visible to the tensor core's async proxy, then one arrival per K block
      fence_proxy_async_smem();
      for (int kb = 0; kb < nchunk; ++kb) mbar_arrive(bar_full + 8 * kb);
    } else {
    int pix0[kRowsPerThread];        // linear input pixel index of tap (0,0) (may lie outside the image)
    uint32_t vmask[kRowsPerThread];  // bit t set <=> tap t of this output pixel is inside the image
    uint32_t dsto[kRowsPerThread];   // swizzled byte offset of this lane's chunk inside a stage
    {
#pragma unroll
      for (int i = 0; i < kRowsPerThread; ++i) {
        const int row = warp * (4 * kRowsPerThread) + i * 4 + rsub;
        dsto[i] = (uint32_t)row * 128u + (((uint32_t)j ^ (uint32_t)(row & 7)) << 4);
        pix0[i] = 0;
        vmask[i] = 0u;
        int img, oy, ox, mm;
        if (!geom.row_pixel(p, row, img, oy, ox, mm)) continue;
        if (p.dense) {
          pix0[i] = mm;
          vmask[i] = 1u;
        } else {
          const int iy0 = oy * p.stride - p.pad, ix0 = ox * p.stride - p.pad;
          pix0[i] = (img * p.h_in + iy0) * p.w_in + ix0;
          // valid taps form a rectangle [ky_lo, ky_hi) x [kx_lo, kx_hi): x bits times the pattern of valid rows
          const int kx_lo = max(0, -ix0), kx_hi = min(p.ksize, p.w_in - ix0);
          const int ky_lo = max(0, -iy0), ky_hi = min(p.ksize, p.h_in - iy0);
          uint32_t msk = 0u;
          if (kx_hi > kx_lo && ky_hi > ky_lo) {
            const uint32_t xm = ((1u << (kx_hi - kx_lo)) - 1u) << kx_lo;
            const uint32_t rows = ((1u << (ky_hi * p.ksize)) - 1u) & ~((1u << (ky_lo * p.ksize)) - 1u);
            msk = xm * (p.ypat_all & rows);
          }
          vmask[i] = msk;
        }
      }
    }
    if (threadIdx.x == 0) BDE_DBG(2);
    // running (tap, channel) position of this lane's chunk: k = kb*64 + j*8
    int tap, c;
    if (p.k_order == 1) {  // chunk-major: every lane is on the same tap; channel = chunk*64 + j*8
      tap = 0;
      c = j * 8;
    } else {
      tap = (j * 8) / p.ctot;
      c = (j * 8) - tap * p.ctot;
    }
    int ky = tap / p.ksize, kx = tap - ky * p.ksize;
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % S;
      const uint32_t ph = (uint32_t)(kb / S) & 1u;
      const bool from0 = c < p.c0;
      const __nv_bfloat16* sbase = from0 ? p.a0 + c : p.a1 + (c - p.c0);
      const int cs = from0 ? p.c0 : p.c1;
      const int tapoff = ky * p.w_in + kx;
      const uint32_t tapbit = (tap < ntaps && c < p.ctot) ? (1u << tap) : 0u;  // K tail -> zero fill
      mbar_wait(bar_empty + 8 * s, ph ^ 1u);
      const uint32_t stage_a = smem_a + s * Cfg::kABytes;
#pragma unroll
      for (int i = 0; i < kRowsPerThread; ++i) {
        const bool ok = (vmask[i] & tapbit) != 0u;
        const __nv_bfloat16* src = ok ? sbase + (size_t)(pix0[i] + tapoff) * cs : p.a0;
        cp_async_16(stage_a + dsto[i], src, ok ? 16u : 0u);
      }
      // asynchronous arrive: fires when this thread's copies for the stage have landed, so the
      // thread runs ahead by up to S stages without ever blocking on its own loads
      cp_async_mbar_arrive_noinc(bar_full + 8 * s);
      // advance to the next K block
      if (p.k_order == 1) {
        ++tap;
        if (++kx == p.ksize) {
          kx = 0;
          if (++ky == p.ksize) {  // all taps of this 64-channel chunk done -> next chunk
            ky = 0;
            tap = 0;
            c += BK;
          }
        }
      } else {
        c += BK;
        while (c >= p.ctot) {
          c -= p.ctot;
          ++tap;
          if (++kx == p.ksize) {
            kx = 0;
            ++ky;
          }
        }
      }
    }

    }  // !kLn

    // =============================== epilogue ===========================================
    // thread <-> tile row (TMEM lane) 32*(warp & 3) + lane; the two warps sharing a lane quarter
    // split the columns in alternating 32-wide chunks
    const int q = warp & 3, half = warp >> 2;
    if (threadIdx.x == 0) BDE_DBG(3);
    // TMEM hands every thread one accumulator ROW (32 columns per load).  Writing rows straight to
    // global memory would make every warp-wide store touch 32 different lines, so each warp first
    // transposes its 32 x 32 chunk through shared memory (the pipeline stages are free once the
    // accumulator is complete) and then works on quads: lane -> (row 4*it + lane/8, columns 4*(lane%8)..+3),
    // i.e. 8 lanes cover 128 contiguous bytes of one output row.
    constexpr int kPitch = 36;  // floats; 16-byte aligned rows, conflict-free for both access patterns
    static_assert(kNumProducerWarps * 32 * kPitch * 4 <= Cfg::kEpiBytes, "epilogue staging outgrows TileCfg::kEpiBytes");
    float* stg = reinterpret_cast<float*>(smem_gen) + warp * (32 * kPitch);
    const int rq = lane >> 3, cq = (lane & 7) * 4;
    int m_it[8];            // output row index of (4*it + rq), -1 if outside the problem
    int dst_it[8];          // SCATTER destination
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      int im, oy, ox, mm;
      const bool ok = geom.row_pixel(p, q * 32 + it * 4 + rq, im, oy, ox, mm);
      m_it[it] = ok ? mm : -1;
      dst_it[it] = (ok && p.epi == BDE_EPI_SCATTER) ? __ldg(p.row_map + mm) : -1;
    }
    // operands the epilogue READS from global memory (c_prev / residual / scatter destination) for the first column
    // chunk: in flight while the accumulator is still being computed
    const bool need_aux = p.epi != BDE_EPI_STORE || p.residual != nullptr;
    float4 aux[8];
#pragma unroll
    for (int it = 0; it < 8; ++it)
      aux[it] = (need_aux && m_it[it] >= 0) ? aux_load(p, m_it[it], n0 + half * 32 + cq, dst_it[it]) : make_float4(0.f, 0.f, 0.f, 0.f);
    mbar_wait(bar_acc, 0);
    tcgen05_fence_after();
    if (threadIdx.x == 0) BDE_DBG(5);
    const uint32_t lane_taddr = tmem_acc + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
    for (int cb = half * 32; cb < BN; cb += 64) {
      uint32_t raw[32];
      tmem_ld_32x32b_x32(lane_taddr + (uint32_t)cb, raw);
      tmem_ld_wait();
      __syncwarp();  // previous chunk fully read back before it is overwritten
#pragma unroll
      for (int jq = 0; jq < 32; jq += 4)
        *reinterpret_cast<float4*>(stg + lane * kPitch + jq) =
            make_float4(__uint_as_float(raw[jq]), __uint_as_float(raw[jq + 1]), __uint_as_float(raw[jq + 2]),
                        __uint_as_float(raw[jq + 3]));
      __syncwarp();
      float4 accv[8];
#pragma unroll
      for (int it = 0; it < 8; ++it) accv[it] = *reinterpret_cast<const float4*>(stg + (it * 4 + rq) * kPitch + cq);
      const float4 bq = *reinterpret_cast<const float4*>(bias_s + cb + cq);
#pragma unroll
      for (int it = 0; it < 8; ++it)
        if (m_it[it] >= 0) epilogue_quad_aux(p, m_it[it], n0 + cb + cq, accv[it], bq, dst_it[it], aux[it]);
      // next chunk's reads: issued together, after this chunk's stores
      if (need_aux && cb + 64 < BN) {
#pragma unroll
        for (int it = 0; it < 8; ++it)
          if (m_it[it] >= 0) aux[it] = aux_load(p, m_it[it], n0 + cb + 64 + cq, dst_it[it]);
      }
    }
    tcgen05_fence_before();
    if (threadIdx.x == 0) BDE_DBG(6);
  } else if (warp == kTmaWarp) {
    // =============================== B producer =========================================
    if (kBTma) {
      if (lane == 0) {
        for (int kb = 0; kb < num_kb; ++kb) {
          const int s = kb % S;
          const uint32_t ph = (uint32_t)(kb / S) & 1u;
          mbar_wait(bar_empty + 8 * s, ph ^ 1u);
          mbar_arrive_expect_tx(bar_full + 8 * s, Cfg::kBBytes);
          tma_load_2d(smem_b + s * Cfg::kBBytes, &tmap_b, bar_full + 8 * s, kb * BK, n0);
        }
      }
    } else {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % S;
        const uint32_t ph = (uint32_t)(kb / S) & 1u;
        mbar_wait(bar_empty + 8 * s, ph ^ 1u);
        for (int row = lane >> 3; row < BN; row += 4) {
          const int jj = lane & 7;
          const __nv_bfloat16* src = p.w + (size_t)(n0 + row) * p.w_ld + kb * BK + jj * 8;
          cp_async_16(smem_b + s * Cfg::kBBytes + (uint32_t)row * 128u + (((uint32_t)jj ^ (uint32_t)(row & 7)) << 4), src, 16u);
        }
        cp_async_mbar_arrive_noinc(bar_full + 8 * s);
      }
    }
  } else {
    // =============================== MMA issuer =========================================
    // all lanes walk the loop, one elected lane issues (see elect_one_sync in tc_common.cuh)
    {
      constexpr uint32_t idesc = make_idesc(BN);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % S;
        const uint32_t ph = (uint32_t)(kb / S) & 1u;
        mbar_wait(bar_full + 8 * s, ph);
        if (kb == 0 && lane == 0) BDE_DBG(4);
        // operands were written through the generic proxy (cp.async): order them before the
        // tensor core's async-proxy reads
        fence_proxy_async_smem();
        tcgen05_fence_after();
        if (elect_one_sync()) {
          const uint64_t adesc = make_smem_desc(smem_a + s * Cfg::kABytes);
          const uint64_t bdesc = make_smem_desc(smem_b + s * Cfg::kBBytes);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 bf16 = 32 bytes inside the swizzle row: +2 in the (addr >> 4) field
            umma_bf16(tmem_acc, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(bar_empty + 8 * s);  // frees the smem stage once these MMAs have read it
          if (kb == num_kb - 1) umma_commit(bar_acc);  // accumulator complete
        }
        __syncwarp();
      }
    }
  }

  __syncthreads();
  if (warp == kMmaWarp) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_acc, Cfg::kTmemCols);
    if (lane == 0) BDE_DBG(7);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  });
  return fn;
}

// weight tensor maps are immutable per (pointer, shape, tile): cache them
int get_weight_tmap(const void* w, int n, int w_ld, int bn, CUtensorMap* out) {
  static std::mutex mu;
  static std::map<std::tuple<const void*, int, int, int>, CUtensorMap> cache;
  std::lock_guard<std::mutex> lock(mu);
  auto key = std::make_tuple(w, n, w_ld, bn);
  auto it = cache.find(key);
  if (it != cache.end()) {
    *out = it->second;
    return 0;
  }
  auto encode = get_encode_fn();
  BDE_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled entry point not available");
  CUtensorMap m;
  cuuint64_t gdim[2] = {(cuuint64_t)w_ld, (cuuint64_t)n};
  cuuint64_t gstride[1] = {(cuuint64_t)w_ld * sizeof(__nv_bfloat16)};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)bn};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BDE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  if (cache.size() > 4096) cache.clear();
  cache[key] = m;
  *out = m;
  return 0;
}

template <int BN, bool kBTma, bool kDeep, int kLn = 0>
int launch(const CUtensorMap& tmap, const TcParams& p, cudaStream_t s) {
  using Cfg = TileCfg<BN, kDeep, kLn>;
  auto kern = gemm_tc_kernel<BN, kBTma, kDeep, kLn>;
  if (first_use_on_device((const void*)kern)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    BDE_REQUIRE(e == cudaSuccess, "bde_gemm(tcgen05): smem attribute: %s", cudaGetErrorString(e));
  }
  const size_t m_tiles = p.tiles_x > 0 ? (size_t)p.n_img * p.tiles_x * p.tiles_y : ceil_div(p.M, BM);
  dim3 grid((unsigned)m_tiles, (unsigned)(p.N / BN));
  kern<<<grid, kThreads, Cfg::kSmemBytes, s>>>(tmap, p);
  return check_launch("gemm_tc_kernel");
}

// bring-up profiling: bde_tc_debug_enable(n) allocates 8 timestamps per CTA for the next launches
long long* g_dbg = nullptr;
size_t g_dbg_ctas = 0;

// tuning switches (read per call; used by tools/tc_phase_probe.py to compare configurations)
bool env_flag(const char* name, bool dflt) {
  const char* e = getenv(name);
  if (e == nullptr || e[0] == 0) return dflt;
  return e[0] == '1';
}

// BDE2VID_TC_B_CPASYNC=1 loads the weight tile with cp.async instead of TMA (bring-up / bisecting)
bool b_via_tma() {
  const char* e = getenv("BDE2VID_TC_B_CPASYNC");
  return !(e != nullptr && e[0] == '1');
}

int fill_params(const bde_gemm_desc* d, TcParams& p, bool& ln) {
  BDE_REQUIRE(d->dtype == BDE_BF16, "bde_gemm(tcgen05): operands must be bf16");
  p.a0 = (const __nv_bfloat16*)d->a0;
  p.a1 = (const __nv_bfloat16*)d->a1;
  p.w = (const __nv_bfloat16*)d->w;
  p.bias = d->bias;
  p.c0 = d->c0; p.c1 = d->c1; p.ctot = d->c0 + d->c1;
  p.n_img = d->n_img;
  p.h_in = d->h_in; p.w_in = d->w_in; p.h_out = d->h_out; p.w_out = d->w_out;
  p.ksize = d->ksize; p.stride = d->stride; p.pad = d->pad;
  p.M = d->n_img * d->h_out * d->w_out;
  p.N = d->n;
  p.K = d->ksize * d->ksize * p.ctot;
  p.w_ld = d->w_ld > 0 ? d->w_ld : p.K;
  p.num_kb = (p.K + BK - 1) / BK;
  p.epi = d->epi; p.act = d->act; p.out_f32 = d->out_f32;
  p.out = d->out; p.out2 = d->out2; p.residual = d->residual; p.res_mode = d->res_mode; p.c_prev = d->c_prev; p.c_out = d->c_out;
  p.row_map = d->row_map;
  p.dbg = nullptr;
  ln = d->ln_mode != 0;
  for (int i = 0; i < 8; ++i) p.ln_f[i] = ln && i < d->ln_D ? d->ln_frames[i] : nullptr;
  p.ln_map = d->ln_tok_map;
  p.ln_D = ln ? d->ln_D : 1;
  p.ln_ntok = ln ? (d->ln_n_tok > 0 ? d->ln_n_tok : 1) : 1;
  if (ln) {
    BDE_REQUIRE(d->ksize == 1 && d->stride == 1 && d->pad == 0 && d->c1 == 0, "bde_gemm(tcgen05): ln_mode needs a 1x1 / dense GEMM");
    BDE_REQUIRE(d->c0 == 64 || d->c0 == 128 || d->c0 == 256, "bde_gemm(tcgen05): ln_mode supports C in {64, 128, 256}");
    BDE_REQUIRE(d->ln_D >= 1 && d->ln_D <= 8, "bde_gemm(tcgen05): ln_D must be in [1, 8]");
  }
  BDE_REQUIRE(p.c0 % 8 == 0 && p.c1 % 8 == 0, "bde_gemm(tcgen05): channel counts must be multiples of 8");
  BDE_REQUIRE(p.ksize * p.ksize <= 32, "bde_gemm(tcgen05): kernel size up to 5x5");
  BDE_REQUIRE(p.w_ld % BK == 0 && p.w_ld >= p.num_kb * BK, "bde_gemm(tcgen05): w_ld must be a zero-padded multiple of 64");
  BDE_REQUIRE(p.N % 32 == 0, "bde_gemm(tcgen05): N must be a multiple of 32");
  BDE_REQUIRE((size_t)d->n_img * d->h_in * d->w_in < ((size_t)1 << 31), "bde_gemm(tcgen05): input pixel count overflows int32");
  BDE_REQUIRE(ln || d->a0 != nullptr, "bde_gemm(tcgen05): null A operand");
  BDE_REQUIRE((((uintptr_t)d->a0) & 15) == 0 && (((uintptr_t)d->a1) & 15) == 0 && (((uintptr_t)d->w) & 127) == 0,
              "bde_gemm(tcgen05): operands must be 16-byte (weights 128-byte) aligned");
  p.k_order = d->k_order;
  p.dense = (p.ksize == 1 && p.stride == 1 && p.pad == 0) ? 1 : 0;
  p.ypat_all = 0u;
  for (int ky = 0; ky < p.ksize; ++ky) p.ypat_all |= 1u << (ky * p.ksize);
  BDE_REQUIRE(p.k_order == 0 || (p.k_order == 1 && p.c0 % BK == 0 && p.c1 % BK == 0),
              "bde_gemm(tcgen05): chunk-major K order needs channel counts that are multiples of 64");
  // convolutions with a real footprint use 2-D pixel tiles + the deep one-CTA-per-SM configuration
  const bool conv = p.ksize > 1 && p.h_out >= kTileH && p.w_out >= kTileW;
  const bool tile2d = conv && env_flag("BDE2VID_TC_TILE2D", true);
  p.tiles_x = tile2d ? (int)ceil_div(p.w_out, kTileW) : 0;
  p.tiles_y = tile2d ? (int)ceil_div(p.h_out, kTileH) : 0;
  return 0;
}

}  // namespace tc

namespace tc {
bool conv_tma_eligible(const TcParams& p, bool ln);
int conv_tma_launch(const bde_gemm_desc* d, const TcParams& p, cudaStream_t s);
}  // namespace tc

int gemm_tcgen05(const bde_gemm_desc* d, cudaStream_t s) {
  using namespace tc;
  TcParams p;
  bool ln = false;
  int rc0 = fill_params(d, p, ln);
  if (rc0 != 0) return rc0;
  if (p.M == 0) return 0;
  // convolutions over 64-channel slabs: persistent kernel with both operands fed by the TMA (gemm_tc_conv.cu)
  if (conv_tma_eligible(p, ln)) return conv_tma_launch(d, p, s);
  BDE_REQUIRE((d->a0_ld == 0 || d->a0_ld == d->c0) && (d->c1 == 0 || d->a1_ld == 0 || d->a1_ld == d->c1),
              "bde_gemm(tcgen05): pitched A operands are only supported by the TMA convolution kernel");
  // tile width: widest tile that still gives most SMs work (measured on the LSTM / encoder shapes: a 256-wide tile
  // gathers the A operand half as often and wins as soon as it yields >= ~100 CTAs; tools/tc_phase_probe.py bn)
  int bn = 32;
  if (p.N % 128 == 0) bn = 128;
  else if (p.N % 64 == 0) bn = 64;
  const size_t m_tiles = p.tiles_x > 0 ? (size_t)p.n_img * p.tiles_x * p.tiles_y : ceil_div(p.M, BM);
  if (p.N % 256 == 0 && p.K >= 512 && m_tiles * (p.N / 256) >= 100) bn = 256;
  {
    // tuning override (tools/tc_phase_probe.py): force the N tile where it divides N
    const char* e = getenv("BDE2VID_TC_BN");
    const int f = (e != nullptr && e[0] != 0) ? atoi(e) : 0;
    if ((f == 32 || f == 64 || f == 128 || f == 256) && p.N % f == 0) bn = f;
  }
  if (ln) {
    // the LayerNorm is recomputed by every N tile of a row block: prefer the widest tile
    bn = (p.N % 256 == 0) ? 256 : (p.N % 192 == 0) ? 192 : (p.N % 128 == 0) ? 128 : (p.N % 64 == 0) ? 64 : 32;
  }
  // grids of at most one CTA per SM cannot overlap two CTAs' phases: give the single CTA a deeper pipeline instead
  const bool small_grid = !ln && m_tiles * (size_t)(p.N / bn) <= (size_t)device_sm_count() && p.num_kb >= 8;
  const bool deep = (p.tiles_x > 0 && env_flag("BDE2VID_TC_DEEP", false)) || (small_grid && env_flag("BDE2VID_TC_DEEP_SMALL", true));
  if (g_dbg != nullptr) {
    const size_t mt = p.tiles_x > 0 ? (size_t)p.n_img * p.tiles_x * p.tiles_y : ceil_div(p.M, BM);
    if (mt * (p.N / bn) <= g_dbg_ctas) p.dbg = g_dbg;
  }
  const bool tma = b_via_tma();
  CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  if (tma) {
    int rc = get_weight_tmap(d->w, p.N, p.w_ld, bn, &tmap);
    if (rc != 0) return rc;
  }
  if (ln) {
    const int chunks = p.c0 / 64;
#define BDE_TC_LN(BN_, CH_) \
  return tma ? launch<BN_, true, false, CH_>(tmap, p, s) : launch<BN_, false, false, CH_>(tmap, p, s)
#define BDE_TC_LN_BN(CH_)                 \
  switch (bn) {                           \
    case 32: BDE_TC_LN(32, CH_);          \
    case 64: BDE_TC_LN(64, CH_);          \
    case 128: BDE_TC_LN(128, CH_);        \
    case 192: BDE_TC_LN(192, CH_);        \
    default: BDE_TC_LN(256, CH_);         \
  }
    if (chunks == 1) { BDE_TC_LN_BN(1) }
    if (chunks == 2) { BDE_TC_LN_BN(2) }
    BDE_TC_LN_BN(4)
#undef BDE_TC_LN_BN
#undef BDE_TC_LN
  }
#define BDE_TC_LAUNCH(BN_)                                                                                   \
  case BN_:                                                                                                  \
    if (deep) return tma ? launch<BN_, true, true>(tmap, p, s) : launch<BN_, false, true>(tmap, p, s);       \
    return tma ? launch<BN_, true, false>(tmap, p, s) : launch<BN_, false, false>(tmap, p, s);
  switch (bn) {
    BDE_TC_LAUNCH(32)
    BDE_TC_LAUNCH(64)
    BDE_TC_LAUNCH(128)
    BDE_TC_LAUNCH(256)
  }
#undef BDE_TC_LAUNCH
  BDE_REQUIRE(false, "bde_gemm(tcgen05): no tile config");
}

}  // namespace bde

extern "C" int bde_tc_debug_enable(size_t max_ctas) {
  using namespace bde::tc;
  if (g_dbg != nullptr) cudaFree(g_dbg);
  g_dbg = nullptr;
  g_dbg_ctas = 0;
  if (max_ctas == 0) return 0;
  if (cudaMalloc(&g_dbg, max_ctas * 8 * sizeof(long long)) != cudaSuccess) return -1;
  cudaMemset(g_dbg, 0, max_ctas * 8 * sizeof(long long));
  g_dbg_ctas = max_ctas;
  return 0;
}

extern "C" int bde_tc_debug_read(long long* host_out, size_t n_ctas) {
  using namespace bde::tc;
  if (g_dbg == nullptr || n_ctas > g_dbg_ctas) return -1;
  return cudaMemcpy(host_out, g_dbg, n_ctas * 8 * sizeof(long long), cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -2;
}
