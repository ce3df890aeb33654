// avc_chain.cu -- the SDF value chain (models/fields.py:72-88: embed -> [Linear -> Softplus] x L -> sdf head) of a tile
// of 128 points as ONE kernel: the layer's activations never leave the SM.
//
// Used by the sample-placement passes of NeuSRenderer.render (renderer.py:336-352: coarse SDF + the up-sampling rounds,
// under no_grad) and by SDFNetwork.sdf queries (extract_fields / validate_mesh) -- everywhere the chain runs without a
// stash for the backward.  Per CTA (persistent, one per SM, tiles of 128 points):
//
//   shared memory   A: the current layer's input as a two-term bf16 split, K-major SWIZZLE_128B, 4 k-blocks x (hi, lo)
//                      x 16 KB = 128 KB -- written in place by the epilogue of the previous layer (layer 0: by TMA);
//                   W: 3-stage ring of 32 KB slabs ([<=256 rows][64 k] of W_l hi or lo), streamed by TMA from L2
//                      (the whole 1.6-3.2 MB model is L2 resident), running ahead across layers and tiles
//   tensor memory   one 128 x 256 fp32 accumulator (256 columns)
//   warp 0          TMA producer;  warp 1: tcgen05.mma issuer (hi*hi + lo*hi on the W_hi slab, hi*lo on the W_lo slab);
//   warps 2-17      epilogue: tcgen05.ld 16 columns at a time, bias + softplus_100 (SFU) + 1/sqrt(2) skip scaling,
//                   bf16 (hi, lo) split, 16-byte st.shared into the swizzled A tile of the NEXT layer; the last hidden
//                   layer instead folds its 64 columns into the sdf head (fp32 dot with row 0 of the last linear)
//
// HBM traffic per point: 160 B in (the encoded pair) + 4 B out, against 2 x 1 KB per layer and direction for the
// unfused launches (8 launches per pass); L2 -> SM: 256 KB of weights per layer and 128-point tile.
// Synchronisation: wfull/wempty (W ring), a0full (TMA tile input), afull (epilogue -> MMA: next A complete AND
// accumulator drained, one arrival per epilogue warp), accfull (tcgen05.commit: accumulator complete, A reads done),
// afree (tcgen05.commit with the last layer's final slab, once per tile: the A tile may take the next tile's input).
#include <cuda.h>

#include <cstdlib>

#include "avc_chain.h"
#include "avc_gemm_tc.cuh"

namespace avc {
namespace chain {

using namespace avc::tc;

constexpr int kCM = 128;
constexpr int kASlab = kCM * 128;                 // [128 rows][64 bf16]: 16 KB
constexpr int kAKB = 4;                           // K <= 256
constexpr int kABytes = kAKB * 2 * kASlab;        // 131072
constexpr int kWSlab = 256 * 128;                 // [256 rows][64 bf16]: 32 KB
constexpr int kWStages = 3;
constexpr int kEW = 16;                           // epilogue warps: 4 TMEM lane quarters x 4 column groups of 64
constexpr int kThreads = 64 + 32 * kEW;
constexpr int kTmemCols = 256;
constexpr int kBarBytes = 256;
constexpr int kSmemBytes = 1024 + kABytes + kWStages * kWSlab + kBarBytes + kCM * 4 + 16;
static_assert(kSmemBytes <= 232448, "exceeds the 227 KB of shared memory per CTA");

struct DevLayer {
  int N, K, nkb, n_mma;
  const float* bias;
  float oscale;
  int next_skip_cols;
};
struct DevArgs {
  int L;
  DevLayer lay[kMaxHidden];
  const __nv_bfloat16* skip_hi;
  const __nv_bfloat16* skip_lo;
  int skip_ld, skip_col0;
  const float* w_sdf;
  const float* b_sdf;
  int head_skip_cols, head_hidden;   // head_hidden = columns of the head input produced by the last hidden layer
  float inv_scale;
  float* sdf_out;
  int nz, pitch;
  long long P;
  int tiles;
  long long* dbg;     // profiling aid (AVC_CHAIN_DEBUG=1): cycle counters of block 0, see launch()
};
struct Maps {
  CUtensorMap a0hi, a0lo;
  CUtensorMap whi[kMaxHidden], wlo[kMaxHidden];
};

__device__ __forceinline__ void named_bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void st_shared_b16(uint32_t addr, uint16_t v) {
  asm volatile("st.shared.b16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
}

__global__ void __launch_bounds__(kThreads, 1)
k_sdf_chain(const __grid_constant__ Maps maps, const __grid_constant__ DevArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t sA = smem_u32(smem);
  const uint32_t sW = sA + kABytes;
  uint64_t* bars = (uint64_t*)(smem + kABytes + kWStages * kWSlab);
  float* sdf_acc = (float*)(smem + kABytes + kWStages * kWSlab + kBarBytes);
  uint32_t* tmem_slot = (uint32_t*)(sdf_acc + kCM);
  const uint32_t wfull0 = smem_u32(bars), wempty0 = wfull0 + 8 * kWStages, a0full = wempty0 + 8 * kWStages,
                 afull = a0full + 8, accfull = afull + 8, afree = accfull + 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = a.L;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.a0hi); tma_prefetch_desc(&maps.a0lo);
    for (int s = 0; s < kWStages; ++s) { mbar_init(wfull0 + 8 * s, 1); mbar_init(wempty0 + 8 * s, 1); }
    mbar_init(a0full, 1);
    mbar_init(afull, kEW);
    mbar_init(accfull, 1);
    mbar_init(afree, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), kTmemCols);
  for (int i = threadIdx.x; i < kCM; i += blockDim.x) sdf_acc[i] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int it = 0, lt = 0;
      pdl_wait();            // the encoded points are the predecessor kernel's output (launched with launch_pdl: this
      pdl_trigger();         // CTA's set-up ran while that kernel was still draining)
      for (int tile = blockIdx.x; tile < a.tiles; tile += gridDim.x, ++lt) {
        // the A buffer is free for the next tile's input once the last layer's MMAs of the previous tile completed.
        // afree completes once per tile and its next phase needs this tile's input, so the producer is never more than
        // one phase behind and the parity wait cannot be satisfied by an older phase.  (Waiting on accfull, which
        // completes once per LAYER, could be: with a last layer of one k-block the 3-stage weight ring lets the producer
        // get here before layer L-2 has committed, and the TMA load would overwrite the A tile that layer's epilogue
        // is still writing.)
        if (lt > 0) mbar_wait(afree, (uint32_t)((lt - 1) & 1));
        mbar_expect_tx(a0full, 2 * kASlab);
        tma_load_2d(sA, &maps.a0hi, 0, tile * kCM, a0full);
        tma_load_2d(sA + kASlab, &maps.a0lo, 0, tile * kCM, a0full);
        for (int l = 0; l < L; ++l) {
          const uint32_t bytes = (uint32_t)a.lay[l].n_mma * 128u;
          for (int kb = 0; kb < a.lay[l].nkb; ++kb)
            for (int h = 0; h < 2; ++h, ++it) {
              const int s = it % kWStages;
              mbar_wait(wempty0 + 8 * s, ((it / kWStages) & 1) ^ 1);
              mbar_expect_tx(wfull0 + 8 * s, bytes);
              tma_load_2d(sW + s * kWSlab, h == 0 ? &maps.whi[l] : &maps.wlo[l], kb * 64, 0, wfull0 + 8 * s);
            }
        }
      }
      if (lt > 0) mbar_wait(afree, (uint32_t)((lt - 1) & 1));   // the last tile's arrival lands before the CTA exits
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    int it = 0, lt = 0;
    const bool prof = a.dbg != nullptr && blockIdx.x == 0 && lane == 0;
    long long t_wa = 0, t_ww = 0, t_all0 = prof ? clock64() : 0;
    for (int tile = blockIdx.x; tile < a.tiles; tile += gridDim.x, ++lt) {
      for (int l = 0; l < L; ++l) {
        long long t0 = prof ? clock64() : 0;
        if (l == 0) mbar_wait(a0full, (uint32_t)(lt & 1));
        const int need = lt * L + l - 1;        // epilogue completion that frees the accumulator / publishes A(l)
        if (need >= 0) mbar_wait(afull, (uint32_t)(need & 1));
        if (prof) t_wa += clock64() - t0;
        tc_fence_after();
        const uint32_t idesc = make_idesc_bf16(kCM, a.lay[l].n_mma, 0, 0);
        const int nkb = a.lay[l].nkb;
        for (int kb = 0; kb < nkb; ++kb)
          for (int h = 0; h < 2; ++h, ++it) {
            const int s = it % kWStages;
            long long t1 = prof ? clock64() : 0;
            mbar_wait(wfull0 + 8 * s, (uint32_t)((it / kWStages) & 1));
            if (prof) t_ww += clock64() - t1;
            tc_fence_after();
            if (elect_one_sync()) {
              const uint64_t da_hi = make_smem_desc(sA + (uint32_t)(kb * 2) * kASlab, 0, 1024);
              const uint64_t da_lo = make_smem_desc(sA + (uint32_t)(kb * 2 + 1) * kASlab, 0, 1024);
              const uint64_t db = make_smem_desc(sW + s * kWSlab, 0, 1024);
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) {
                if (h == 0) {
                  umma_f16(tmem_base, da_hi + 2 * k4, db + 2 * k4, idesc, (kb | k4) ? 1u : 0u);
                  umma_f16(tmem_base, da_lo + 2 * k4, db + 2 * k4, idesc, 1u);
                } else {
                  umma_f16(tmem_base, da_hi + 2 * k4, db + 2 * k4, idesc, 1u);
                }
              }
              umma_commit(wempty0 + 8 * s);
              if (kb == nkb - 1 && h == 1) {
                umma_commit(accfull);
                if (l == L - 1) umma_commit(afree);
              }
            }
            __syncwarp();
          }
      }
    }
    if (prof) { a.dbg[0] = t_wa; a.dbg[1] = t_ww; a.dbg[2] = clock64() - t_all0; a.dbg[3] = (long long)lt * L; }
  } else {
    // ------------------------------------------------------------------------------------------ epilogue
    pdl_wait();                             // skip-concat columns in, sdf out: predecessor kernels' buffers
    const int q = warp & 3;                 // TMEM lane quarter
    const int cw = (warp - 2) >> 2;         // column group: columns [64 cw, 64 cw + 64) = k-block cw of the next A
    const int row = q * 32 + lane;          // row of the tile this thread owns
    const int et = threadIdx.x - 64;        // 0 .. 511
    const uint32_t a_row = (uint32_t)((row >> 3) * 1024 + (row & 7) * 128);
    const uint32_t sw = (uint32_t)(row & 7);
    int lt = 0;
    const bool eprof = a.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == 64;
    long long e_wait = 0, e_work = 0;
    for (int tile = blockIdx.x; tile < a.tiles; tile += gridDim.x, ++lt) {
      const long long p = (long long)tile * kCM + row;
      for (int l = 0; l < L; ++l) {
        const DevLayer& ly = a.lay[l];
        const bool last = (l == L - 1);
        // the biases (sdf-row weights for the last layer come later) of the first 16 columns are fetched before the wait
        // for the accumulator, every further group's one group ahead: their L1 / L2 latency hides under the SFU work
        auto load_bias = [&](float4 (&dst)[4], int c0) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            dst[i] = (c0 + 4 * i < ly.N) ? __ldg(reinterpret_cast<const float4*>(ly.bias + c0) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        float4 bq[4];
        load_bias(bq, 64 * cw);
        long long e0 = eprof ? clock64() : 0;
        mbar_wait(accfull, (uint32_t)((lt * L + l) & 1));
        long long e1 = eprof ? clock64() : 0;
        if (eprof) e_wait += e1 - e0;
        tc_fence_after();
        float dot = 0.f;
        const uint32_t dst_hi = sA + (uint32_t)(cw * 2) * kASlab + a_row;
        const uint32_t dst_lo = dst_hi + kASlab;
        // columns this warp must provide to the next layer: k-block cw exists there iff 64 cw < K_next
        const int k_next = last ? a.head_hidden : a.lay[l + 1].K;
        if (64 * cw < k_next || (last && 64 * cw < ly.N)) {
#pragma unroll 1
          for (int g = 0; g < 4; ++g) {
            const int c0 = 64 * cw + 16 * g;
            uint32_t r[16];
            if (c0 < ly.n_mma) {
              tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) r[i] = 0u;
            }
            // branch-free and batched: the 16 biases arrive as four 16-byte loads issued together, then 16 independent
            // SFU chains (ex2 -> lg2); columns >= N are zeroed by a select.  (A per-element `if (c < N) { load; softplus }`
            // serialised load and SFU latencies: 21.5 k cycles per tile-layer measured, against 6.1 k of tensor work.)
            float bb[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) { bb[4 * i] = bq[i].x; bb[4 * i + 1] = bq[i].y; bb[4 * i + 2] = bq[i].z; bb[4 * i + 3] = bq[i].w; }
            if (g < 3) load_bias(bq, c0 + 16);
            float hv[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float z = __uint_as_float(r[i]) + bb[i];
              const float bz = z * kBeta;
              const float sp = __logf(1.0f + __expf(bz)) * (1.0f / kBeta);
              const float h = (bz > kThresh ? z : sp) * ly.oscale;
              hv[i] = (c0 + i < ly.N) ? h : 0.f;
            }
            if (last) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);      // hv is already zero for columns >= N
                if (c0 + 4 * i < ly.N) t = __ldg(reinterpret_cast<const float4*>(a.w_sdf + c0) + i);
                dot = fmaf(hv[4 * i], t.x, fmaf(hv[4 * i + 1], t.y, fmaf(hv[4 * i + 2], t.z, fmaf(hv[4 * i + 3], t.w, dot))));
              }
            } else {
#pragma unroll
              for (int ch = 0; ch < 2; ++ch) {
                const float* v = hv + 8 * ch;
                const uint32_t h01 = bf16x2_bits(v[0], v[1]), h23 = bf16x2_bits(v[2], v[3]);
                const uint32_t h45 = bf16x2_bits(v[4], v[5]), h67 = bf16x2_bits(v[6], v[7]);
                const uint32_t l01 = bf16x2_bits(v[0] - __uint_as_float(h01 << 16), v[1] - __uint_as_float(h01 & 0xffff0000u));
                const uint32_t l23 = bf16x2_bits(v[2] - __uint_as_float(h23 << 16), v[3] - __uint_as_float(h23 & 0xffff0000u));
                const uint32_t l45 = bf16x2_bits(v[4] - __uint_as_float(h45 << 16), v[5] - __uint_as_float(h45 & 0xffff0000u));
                const uint32_t l67 = bf16x2_bits(v[6] - __uint_as_float(h67 << 16), v[7] - __uint_as_float(h67 & 0xffff0000u));
                const uint32_t off = (((uint32_t)(2 * g + ch)) ^ sw) << 4;
                st_shared_v4(dst_hi + off, h01, h23, h45, h67);
                st_shared_v4(dst_lo + off, l01, l23, l45, l67);
              }
            }
          }
        }
        if (!last) {
          if (ly.next_skip_cols > 0) {
            // cat([h, enc]) / sqrt(2): the enc / sqrt(2) columns come from the pair k_encode_* wrote for this layer.
            // Every epilogue warp has passed accfull, but the writers of the overlapping 16-byte chunks (columns
            // < N of the same chunk, zeros above) must be done first: sync the 16 epilogue warps.
            named_bar_sync(1, 32 * kEW);
            const int E = ly.next_skip_cols;
            for (int e = et; e < kCM * E; e += 32 * kEW) {
              const int rr = e / E, c = ly.N + (e - rr * E);
              const long long pp = (long long)tile * kCM + rr;
              uint16_t vh = 0, vl = 0;
              if (pp < a.P) {
                const size_t o = (size_t)pp * a.skip_ld + a.skip_col0 + (c - ly.N);
                vh = reinterpret_cast<const uint16_t*>(a.skip_hi)[o];
                vl = reinterpret_cast<const uint16_t*>(a.skip_lo)[o];
              }
              const uint32_t base = sA + (uint32_t)((c >> 6) * 2) * kASlab + (uint32_t)((rr >> 3) * 1024 + (rr & 7) * 128) +
                                    (((uint32_t)((c & 63) >> 3) ^ (uint32_t)(rr & 7)) << 4) + (uint32_t)(c & 7) * 2u;
              st_shared_b16(base, vh);
              st_shared_b16(base + kASlab, vl);
            }
          }
          fence_proxy_async();            // generic-proxy smem writes -> visible to the tensor core (async proxy)
        } else {
          // sdf head: the partial dots of the 4 column groups are added in a FIXED order (group 0, 1, 2, 3), so the
          // result does not depend on warp scheduling (sample placement is discontinuous in the sdf: bit-stable runs)
#pragma unroll 1
          for (int k = 0; k < 4; ++k) {
            if (cw == k && 64 * cw < ly.N) sdf_acc[row] += dot;
            named_bar_sync(1, 32 * kEW);
          }
          if (cw == 0) {
            float s = sdf_acc[row];
            sdf_acc[row] = 0.f;
            if (p < a.P) {
              for (int c = 0; c < a.head_skip_cols; ++c) {      // head takes the skip concat itself (skip_in has n_layers)
                const size_t o = (size_t)p * a.skip_ld + a.skip_col0 + c;
                s = fmaf(__bfloat162float(a.skip_hi[o]) + __bfloat162float(a.skip_lo[o]), __ldg(a.w_sdf + ly.N + c), s);
              }
              const long long o = a.nz > 0 ? (p / a.nz) * a.pitch + (p % a.nz) : p;
              a.sdf_out[o] = (s + __ldg(a.b_sdf)) * a.inv_scale;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(afull);
        if (eprof) e_work += clock64() - e1;
      }
    }
    if (eprof) { a.dbg[4] = e_wait; a.dbg[5] = e_work; }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

static long long* g_dbg = nullptr;

bool supported(const Args& a) {
  if (a.L < 1 || a.L > kMaxHidden) return false;
  for (int l = 0; l < a.L; ++l) {
    const Layer& y = a.lay[l];
    if (y.N < 1 || y.N > 256 || y.K < 1 || y.K > 256 || (y.ldw % 8) != 0) return false;
    if (l + 1 < a.L && y.N + y.next_skip_cols != a.lay[l + 1].K) return false;
  }
  if (a.lay[a.L - 1].N + a.head_skip_cols != a.K_head) return false;
  if (a.ld0 % 8) return false;
  return true;
}

int launch(const Args& a, cudaStream_t st) {
  if (a.P <= 0) return 0;
  if (!supported(a)) return AVC_E_BADCFG;
  Maps m;
  DevArgs d;
  d.L = a.L;
  AVC_TRY(make_map_bf16_cached(&m.a0hi, a.a0_hi, (uint64_t)a.P, (uint64_t)a.lay[0].K, (uint64_t)a.ld0, 64, kCM));
  AVC_TRY(make_map_bf16_cached(&m.a0lo, a.a0_lo, (uint64_t)a.P, (uint64_t)a.lay[0].K, (uint64_t)a.ld0, 64, kCM));
  for (int l = 0; l < a.L; ++l) {
    const Layer& y = a.lay[l];
    DevLayer& o = d.lay[l];
    o.N = y.N; o.K = y.K; o.nkb = (y.K + 63) / 64; o.n_mma = ((y.N + 15) / 16) * 16;
    o.bias = y.bias; o.oscale = y.oscale; o.next_skip_cols = y.next_skip_cols;
    AVC_TRY(make_map_bf16_cached(&m.whi[l], y.w_hi, (uint64_t)y.N, (uint64_t)y.K, (uint64_t)y.ldw, 64, (uint32_t)o.n_mma));
    AVC_TRY(make_map_bf16_cached(&m.wlo[l], y.w_lo, (uint64_t)y.N, (uint64_t)y.K, (uint64_t)y.ldw, 64, (uint32_t)o.n_mma));
  }
  for (int l = a.L; l < kMaxHidden; ++l) { m.whi[l] = m.whi[0]; m.wlo[l] = m.wlo[0]; d.lay[l] = d.lay[0]; }
  d.skip_hi = a.skip_hi; d.skip_lo = a.skip_lo; d.skip_ld = a.skip_ld; d.skip_col0 = a.skip_col0;
  d.w_sdf = a.w_sdf; d.b_sdf = a.b_sdf; d.head_skip_cols = a.head_skip_cols; d.head_hidden = a.lay[a.L - 1].N;
  d.inv_scale = a.inv_scale; d.sdf_out = a.sdf_out; d.nz = a.nz; d.pitch = a.pitch; d.P = a.P;
  d.tiles = (int)((a.P + kCM - 1) / kCM);
  static thread_local bool attr_set = false;
  if (!attr_set) {
    AVC_CUDA_TRY(cudaFuncSetAttribute(k_sdf_chain, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  static thread_local int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    AVC_CUDA_TRY(cudaGetDevice(&dev));
    AVC_CUDA_TRY(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int grid = d.tiles < num_sms ? d.tiles : num_sms;
  d.dbg = nullptr;
  static long long* dbg_buf = nullptr;
  const char* dbg_env = getenv("AVC_CHAIN_DEBUG");      // profiling aid: cycle counters of block 0 -> avc_chain_debug_read
  if (dbg_env && atoi(dbg_env) == 1) {
    if (!dbg_buf) AVC_CUDA_TRY(cudaMalloc(&dbg_buf, 16 * sizeof(long long)));
    AVC_CUDA_TRY(cudaMemsetAsync(dbg_buf, 0, 16 * sizeof(long long), st));
    d.dbg = dbg_buf;
    g_dbg = dbg_buf;
  }
  AVC_CUDA_TRY(launch_pdl(k_sdf_chain, dim3(grid), dim3(kThreads), (size_t)kSmemBytes, st, m, d));
  AVC_LAUNCH_TRY();
  return 0;
}

// [0] MMA warp waiting for its A operand (a0full / afull), [1] waiting for weight slabs (wfull), [2] MMA warp total,
// [3] tile-layers processed, [4] epilogue thread waiting for the accumulator, [5] epilogue work (accfull -> arrive)
int debug_read(long long out[8]) {
  if (!g_dbg) return AVC_E_NULL;
  AVC_CUDA_TRY(cudaDeviceSynchronize());
  AVC_CUDA_TRY(cudaMemcpy(out, g_dbg, 8 * sizeof(long long), cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace chain
}  // namespace avc

extern "C" int avc_chain_debug_read(long long* out8) { return avc::chain::debug_read(out8); }
