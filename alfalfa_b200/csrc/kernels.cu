// kernels.cu -- sm_100a kernels of the VP8 pixel pipeline.
//
// Three kernels per frame batch, all "one warp per macroblock (row)":
//   k_inter        every inter-coded macroblock is independent (the reference frame is frozen):
//                  one warp per macroblock, six-tap motion compensation + token expansion +
//                  dequant + IWHT + IDCT + add, fully parallel.         (macroblock.cc:553-601)
//   k_intra        intra macroblocks read unfiltered pixels of their left / above / above-right
//                  neighbours in the same frame: one warp per macroblock ROW sweeping left to
//                  right, rows chained by progress counters in HBM (2-macroblock lag).
//                                                                       (macroblock.cc:523-551)
//   k_loopfilter   same wavefront shape for the in-loop deblocking filter: lanes 0-15 filter
//                  the 16 luma positions of an edge, lanes 16-23 / 24-31 the 8 U / 8 V ones.
//                                                    (loopfilter.cc:133-154, frame.cc:139-182)
// Arithmetic lives in vp8_math.cuh (shared with the CPU unit tests); this file is data movement.
//
// Memory-model notes for the wavefront kernels: pixels written by another warp are read with
// ld.global.cg (L2, never a stale L1 line); a finished macroblock is published with
// __syncwarp() (orders every lane's stores before lane 0) and one st.release.gpu by lane 0; the
// consumer polls with ld.acquire.gpu on lane 0 and __syncwarp()s before the other lanes read.
#include <cuda_runtime.h>
#include <stdint.h>

#include "enc_costs.h"
#include "engine.h"
#include "vp8_math.cuh"

namespace vp8 {
namespace {

#define VP8_LUT_QUALIFIER __device__ const
#include "bpred_lut.inc"

// sixtap_filters (prediction.cc:645-653)
__constant__ int16_t c_sixtap[8][6] = {{0, 0, 128, 0, 0, 0},     {0, -6, 123, 12, -1, 0}, {2, -11, 108, 36, -8, 1},
                                      {0, -9, 93, 50, -6, 0},   {3, -16, 77, 77, -16, 3}, {0, -6, 50, 93, -9, 0},
                                      {1, -8, 36, 108, -11, 2}, {0, -1, 12, 123, -6, 0}};

// Optional phase profiling of the wavefront kernels (build with -DVP8_PROFILE, tools/phase_profile.py):
// lane 0 of every warp accumulates clock64() deltas per phase and adds them to g_prof at exit.
#ifdef VP8_PROFILE
__device__ unsigned long long g_prof[32];
#define PROF_DECL unsigned long long prof_t = clock64(), prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; unsigned prof_n = 0
#define PROF(i)                                  \
  do {                                           \
    const unsigned long long now_ = clock64();   \
    prof_acc[i] += now_ - prof_t;                \
    prof_t = now_;                               \
  } while (0)
#define PROF_COUNT() (prof_n++)
#define PROF_FLUSH(base)                                                           \
  do {                                                                             \
    if (lane == 0) {                                                               \
      for (int i_ = 0; i_ < 8; i_++) atomicAdd(&g_prof[(base) + i_], prof_acc[i_]); \
      atomicAdd(&g_prof[(base) + 8], (unsigned long long)prof_n);                  \
    }                                                                              \
  } while (0)
#else
#define PROF_DECL
#define PROF(i)
#define PROF_COUNT()
#define PROF_FLUSH(base)
#endif

constexpr int CS = 20;          // int16 stride of one 4x4 coefficient block in shared memory: 40 bytes, so a block
                                // row is one aligned 8-byte access and 16 lanes x 8 bytes hit 32 distinct banks
constexpr int COEF_I16 = 25 * CS + 4;    // 504 int16 = 63 16-byte vectors (zeroed as vectors)

struct MbFields {
  uint32_t tok_off, tok_cnt;
  int y_mode, uv_mode, ref, segment, lf_level, flags;
  int mv_x, mv_y;
  uint32_t split_idx;
  uint32_t bm_lo, bm_hi;
};

__device__ __forceinline__ MbFields load_mb(const vp8gpu_mb* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  const uint4 a = __ldg(q), b = __ldg(q + 1);
  MbFields f;
  f.tok_off = a.x;
  f.tok_cnt = a.y & 0xFFFF;
  f.y_mode = (a.y >> 16) & 0xFF;
  f.uv_mode = a.y >> 24;
  f.ref = a.z & 0xFF;
  f.segment = (a.z >> 8) & 0xFF;
  f.lf_level = (a.z >> 16) & 0xFF;
  f.flags = a.z >> 24;
  f.mv_x = (int16_t)(a.w & 0xFFFF);
  f.mv_y = (int16_t)(a.w >> 16);
  f.split_idx = b.x;
  f.bm_lo = b.z;
  f.bm_hi = b.w;
  return f;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// MotionVector::luma_to_chroma (macroblock.cc:289-299) on the int16 sum of four luma components
__device__ __forceinline__ int chroma_component(int sum) {
  const int s = (int16_t)sum;
  return s >= 0 ? (s + 4) >> 3 : -((-s + 4) >> 3);
}

// ------------------------------------------------------------------------------------------------
// Motion compensation of one N x N block by the whole warp (prediction.cc:655-674, 919-971).
// (x0, y0) = block origin in the plane, mv in 1/8 pel.
//  * the source window ((N+5)^2, or N^2 for whole-pel vectors) is staged in shared memory; when it
//    lies inside the plane it is fetched as aligned 32-bit words, otherwise pixel by pixel with
//    clamped coordinates (EdgeExtendedRaster::at, vp8_raster.hh:327-338) -- no padded planes needed;
//  * each lane filters strips of 4 outputs from a 9-pixel run (9 loads, 24 MACs);
//  * a pass whose fraction is 0 is skipped: its taps are {0,0,128,0,0,0}, (128 p + 64) >> 7 = p.
// ------------------------------------------------------------------------------------------------
template <int N>
struct Mc {
  static constexpr int NW = (N + 11) / 4;  // words per staged row: covers 3 + N + 5 bytes
  static constexpr int TS = 4 * NW;        // staged row stride in bytes (24 / 16 / 12)
};

// returns the byte offset of window column 0 inside a staged row
template <int N>
__device__ __forceinline__ int load_window(const uint8_t* __restrict__ ref, int pitch, int PW, int PH, int wx, int wy,
                                           int wcols, int wrows, uint8_t* tile, int lane) {
  constexpr int NW = Mc<N>::NW, TS = Mc<N>::TS;
  if (wx >= 0 && wy >= 0 && wx + wcols <= PW && wy + wrows <= PH) {
    const int o = wx & 3;
    const uint8_t* base = ref + (size_t)wy * pitch + (wx - o);
    uint32_t* tw = reinterpret_cast<uint32_t*>(tile);
    for (int i = lane; i < wrows * NW; i += 32) {
      const int r = i / NW, w = i - r * NW;
      tw[i] = __ldg(reinterpret_cast<const uint32_t*>(base + (size_t)r * pitch) + w);
    }
    return o;
  }
  for (int i = lane; i < wrows * wcols; i += 32) {
    const int r = i / wcols, c = i - r * wcols;
    tile[r * TS + c] = __ldg(ref + (size_t)clampi(wy + r, 0, PH - 1) * pitch + clampi(wx + c, 0, PW - 1));
  }
  return 0;
}

// horizontal 6-tap over `nrows` staged rows: out[r][c] from win[r][c .. c+5]; 4 outputs per item
template <int N>
__device__ __forceinline__ void hpass(const uint8_t* win, int nrows, const int16_t* hf, uint8_t* out, int ostride,
                                      int lane) {
  constexpr int G = N / 4, TS = Mc<N>::TS;
  for (int i = lane; i < nrows * G; i += 32) {
    const int r = i / G, g = i - r * G;
    const uint8_t* t = win + r * TS + 4 * g;
    int p[9];
#pragma unroll
    for (int k = 0; k < 9; k++) p[k] = t[k];
    uint32_t o = 0;
#pragma unroll
    for (int j = 0; j < 4; j++)
      o |= (uint32_t)vp8m::sixtap(p[j], p[j + 1], p[j + 2], p[j + 3], p[j + 4], p[j + 5], hf) << (8 * j);
    *reinterpret_cast<uint32_t*>(out + r * ostride + 4 * g) = o;
  }
}
// vertical 6-tap: dst[r][c] from src[r .. r+5][c]; each item = one column, 4 rows
template <int N>
__device__ __forceinline__ void vpass(const uint8_t* src, int sstride, const int16_t* vf, uint8_t* dst, int dstride,
                                      int lane) {
  constexpr int G = N / 4;
  for (int i = lane; i < N * G; i += 32) {
    const int g = i / N, c = i - g * N;
    const uint8_t* m = src + (4 * g) * sstride + c;
    int p[9];
#pragma unroll
    for (int k = 0; k < 9; k++) p[k] = m[k * sstride];
#pragma unroll
    for (int j = 0; j < 4; j++)
      dst[(4 * g + j) * dstride + c] = (uint8_t)vp8m::sixtap(p[j], p[j + 1], p[j + 2], p[j + 3], p[j + 4], p[j + 5], vf);
  }
}

// A planned block prediction: where its source window is, and (when the window lies inside the
// plane) the window itself, already requested into registers so that the loads of several planes
// are in flight together.
template <int N>
struct McPlan {
  static constexpr int K = (Mc<N>::NW * (N + 5) + 31) / 32;  // words per lane: 4 / 2 / 1
  int wx, wy, wsize, mx, my, o;
  bool fast;
  uint32_t regs[K];
};

template <int N>
__device__ __forceinline__ void mc_plan(McPlan<N>& p, const uint8_t* __restrict__ ref, int pitch, int PW, int PH,
                                        int x0, int y0, int mvx, int mvy, int lane) {
  constexpr int NW = Mc<N>::NW;
  p.mx = mvx & 7;
  p.my = mvy & 7;
  const bool whole = (p.mx | p.my) == 0;
  p.wx = x0 + (mvx >> 3) - (whole ? 0 : 2);
  p.wy = y0 + (mvy >> 3) - (whole ? 0 : 2);
  p.wsize = whole ? N : N + 5;
  p.fast = p.wx >= 0 && p.wy >= 0 && p.wx + p.wsize <= PW && p.wy + p.wsize <= PH;
  p.o = p.fast ? (p.wx & 3) : 0;
  if (p.fast) {
    const uint8_t* base = ref + (size_t)p.wy * pitch + (p.wx - p.o);
#pragma unroll
    for (int k = 0; k < McPlan<N>::K; k++) {
      const int i = lane + 32 * k;
      const int r = i / NW, w = i - r * NW;
      p.regs[k] = i < p.wsize * NW ? __ldg(reinterpret_cast<const uint32_t*>(base + (size_t)r * pitch) + w) : 0u;
    }
  }
}

template <int N>
__device__ __forceinline__ void mc_finish(const McPlan<N>& p, const uint8_t* __restrict__ ref, int pitch, int PW, int PH,
                                          uint8_t* dst, int dstride, uint8_t* tile, uint8_t* mid, int lane) {
  constexpr int TS = Mc<N>::TS, NW = Mc<N>::NW, G = N / 4;
  if (p.fast) {
    uint32_t* tw = reinterpret_cast<uint32_t*>(tile);
#pragma unroll
    for (int k = 0; k < McPlan<N>::K; k++) {
      const int i = lane + 32 * k;
      if (i < p.wsize * NW) tw[i] = p.regs[k];
    }
  } else {
    for (int i = lane; i < p.wsize * p.wsize; i += 32) {
      const int r = i / p.wsize, c = i - r * p.wsize;
      tile[r * TS + c] = __ldg(ref + (size_t)clampi(p.wy + r, 0, PH - 1) * pitch + clampi(p.wx + c, 0, PW - 1));
    }
  }
  __syncwarp();
  const uint8_t* win = tile + p.o;
  if ((p.mx | p.my) == 0) {
    for (int i = lane; i < N * G; i += 32) {
      const int r = i / G, g = i - r * G;
      const uint8_t* t = win + r * TS + 4 * g;
      *reinterpret_cast<uint32_t*>(dst + r * dstride + 4 * g) =
          (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16) | ((uint32_t)t[3] << 24);
    }
  } else if (p.mx && p.my) {
    hpass<N>(win, N + 5, c_sixtap[p.mx], mid, N, lane);
    __syncwarp();
    vpass<N>(mid, N, c_sixtap[p.my], dst, dstride, lane);
  } else if (p.mx) {
    hpass<N>(win + 2 * TS, N, c_sixtap[p.mx], dst, dstride, lane);
  } else {
    vpass<N>(win + 2, TS, c_sixtap[p.my], dst, dstride, lane);
  }
  __syncwarp();
}

template <int N>
__device__ __forceinline__ void mc_block(const uint8_t* __restrict__ ref, int pitch, int PW, int PH, int x0, int y0,
                                         int mvx, int mvy, uint8_t* dst, int dstride, uint8_t* tile, uint8_t* mid,
                                         int lane) {
  McPlan<N> p;
  mc_plan<N>(p, ref, pitch, PW, PH, x0, y0, mvx, mvy, lane);
  mc_finish<N>(p, ref, pitch, PW, PH, dst, dstride, tile, mid, lane);
}

// ------------------------------------------------------------------------------------------------
// GPU back end of the entropy decoder: expand the macroblock's token list into dequantised
// coefficient blocks (quantization.cc:95-126, int16 wrap), run the inverse WHT (transform.cc:47-88)
// and the inverse DCT (transform.cc:100-137).  On return coef[blk*CS + y*4 + x] holds the
// RESIDUAL of pixel (x, y) of block blk (0-15 Y, 16-19 U, 20-23 V).
// ------------------------------------------------------------------------------------------------
// second half, shared with the encoder's reconstruction: coef holds DEQUANTISED coefficients.
// Returns the mask of blocks (bit b, b < 24) whose residual is not all zero.
__device__ __forceinline__ uint32_t inverse_transforms(int16_t* coef, bool has_y2, int lane);

__device__ __forceinline__ uint32_t build_residuals(const DevJob& J, const MbFields& f, int16_t* coef, int lane) {
  uint4* z = reinterpret_cast<uint4*>(coef);
  for (int i = lane; i < COEF_I16 / 8; i += 32) z[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncwarp();
  const vp8gpu_quant q = J.quant[f.segment];
  const vp8gpu_token* tok = J.tokens + f.tok_off;
  for (uint32_t t = lane; t < f.tok_cnt; t += 32) {
    const uint32_t v = __ldg(tok + t);
    const int blk = (v >> 20) & 31, pos = (v >> 16) & 15;
    const int val = (int16_t)(v & 0xFFFF);
    int factor;
    if (blk < 16) factor = pos ? q.y_ac : q.y_dc;
    else if (blk < 24) factor = pos ? q.uv_ac : q.uv_dc;
    else factor = pos ? q.y2_ac : q.y2_dc;
    coef[blk * CS + pos] = (int16_t)(val * factor);
  }
  __syncwarp();
  return inverse_transforms(coef, (f.flags & VP8GPU_MB_HAS_Y2) != 0, lane);
}

__device__ __forceinline__ uint32_t inverse_transforms(int16_t* coef, bool has_y2, int lane) {
  if (has_y2) {
    // inverse WHT on 16 lanes (transform.cc:47-88): lane i first produces intermediate m[i]
    // (column i & 3, butterfly output i >> 2), the row pass exchanges m through shuffles.
    const int16_t* y2 = coef + 24 * CS;
    int m = 0;
    if (lane < 16) {
      const int c = lane & 3;
      const int v0 = y2[c], v1 = y2[c + 4], v2 = y2[c + 8], v3 = y2[c + 12];
      const int a1 = v0 + v3, b1 = v1 + v2, c1 = v1 - v2, d1 = v0 - v3;
      const int k = lane >> 2;
      m = vp8m::wrap16(k == 0 ? a1 + b1 : (k == 1 ? c1 + d1 : (k == 2 ? a1 - b1 : d1 - c1)));
    }
    const int o4 = lane & 12;
    const int m0 = __shfl_sync(0xffffffffu, m, o4), m1 = __shfl_sync(0xffffffffu, m, o4 + 1);
    const int m2 = __shfl_sync(0xffffffffu, m, o4 + 2), m3 = __shfl_sync(0xffffffffu, m, o4 + 3);
    if (lane < 16) {
      const int a1 = m0 + m3, b1 = m1 + m2, c1 = m1 - m2, d1 = m0 - m3;
      const int p = lane & 3;
      const int x = p == 0 ? a1 + b1 : (p == 1 ? c1 + d1 : (p == 2 ? a1 - b1 : d1 - c1));
      coef[lane * CS] = (int16_t)((x + 3) >> 3);  // DC of luma sub-block `lane`
    }
    __syncwarp();
  }
  bool nonzero = false;
  if (lane < 24) {
    uint2* cv = reinterpret_cast<uint2*>(coef + lane * CS);  // four 8-byte rows
    uint2 v[4];
#pragma unroll
    for (int k = 0; k < 4; k++) v[k] = cv[k];
    const uint32_t ac = (v[0].x & 0xFFFF0000u) | v[0].y | v[1].x | v[1].y | v[2].x | v[2].y | v[3].x | v[3].y;
    if (ac) {
      int16_t in[16], r[16];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        in[4 * k] = (int16_t)(v[k].x & 0xFFFF), in[4 * k + 1] = (int16_t)(v[k].x >> 16);
        in[4 * k + 2] = (int16_t)(v[k].y & 0xFFFF), in[4 * k + 3] = (int16_t)(v[k].y >> 16);
      }
      vp8m::idct16(in, r);
#pragma unroll
      for (int k = 0; k < 4; k++)
        cv[k] = make_uint2((uint32_t)(uint16_t)r[4 * k] | ((uint32_t)(uint16_t)r[4 * k + 1] << 16),
                           (uint32_t)(uint16_t)r[4 * k + 2] | ((uint32_t)(uint16_t)r[4 * k + 3] << 16));
      nonzero = true;
    } else if (v[0].x) {
      // DC only: both passes of idct_add reduce to (dc + 4) >> 3 for every pixel
      const uint32_t r = (uint32_t)(uint16_t)(((int)(int16_t)(v[0].x & 0xFFFF) + 4) >> 3);
      const uint32_t rr = r | (r << 16);
#pragma unroll
      for (int k = 0; k < 4; k++) cv[k] = make_uint2(rr, rr);
      nonzero = r != 0;
    }
  }
  const uint32_t nz = __ballot_sync(0xffffffffu, nonzero);
  __syncwarp();
  return nz;
}

// macroblock buffer -> frame: 16-byte luma rows by lanes 0-15, 8-byte chroma rows by 16-31
__device__ __forceinline__ void store_mb(const uint8_t* pix, uint8_t* frame, const Geom& g, int col, int row,
                                         int lane) {
  if (lane < 16) {
    const uint4 v = *reinterpret_cast<const uint4*>(pix + lane * 16);
    *reinterpret_cast<uint4*>(frame + (size_t)(16 * row + lane) * g.y_pitch + 16 * col) = v;
  } else {
    const int plane = (lane - 16) >> 3, y = (lane - 16) & 7;
    const uint2 v = *reinterpret_cast<const uint2*>(pix + 256 + plane * 64 + y * 8);
    uint8_t* base = frame + (plane ? g.v_off : g.u_off);
    *reinterpret_cast<uint2*>(base + (size_t)(8 * row + y) * g.c_pitch + 8 * col) = v;
  }
}

// ================================================================================================
// k_inter: one warp per inter-coded macroblock (macroblock.cc:553-601).
//
//  * The three source windows (luma 21 x 21 inside a 48 x 21 box, chroma 13 x 13 inside 32 x 13 boxes) are
//    fetched by TMA (cp.async.bulk.tensor.2d, one tensor map per plane of every raster, engine.cu) into
//    the warp's shared-memory tile and signalled on the warp's mbarrier; lane 0 issues the three copies,
//    nobody computes an address per pixel.  TMA wants the box to start on a 16-byte boundary of the row
//    (tools/probe/tma_probe.cu), so the box starts at the window's x rounded down to 16 and the window
//    sits at byte offset x & 15 of every tile row; the row filter re-aligns with one funnel shift per
//    word.  A window that leaves the plane takes the clamped path (EdgeExtendedRaster::at,
//    vp8_raster.hh:327-338): TMA fills out-of-range pixels with zeros, the reference replicates the edge.
//  * While the tiles are in flight the warp expands the macroblock's tokens into residuals (dequant,
//    IWHT, IDCT).
//  * Six-tap filter on packed pixels (vp8_math.cuh): rows as two 4-byte dot products per output (dp4a),
//    columns as 32-bit multiply-adds on pixel pairs; clamp + pack with cvt.pack.sat.  A pass whose
//    fraction is 0 is skipped ((128 p + 64) >> 7 = p), a whole-pel vector is a copy.
//  * SPLITMV: the 24 4x4 blocks (16 Y, 4 U, 4 V) are staged and filtered lane-parallel, (block, row)
//    and (block, column pair) items spread over the warp.
// ================================================================================================
constexpr int INTER_WARPS = 4;
constexpr int TSY = 48, TSC = 32;  // tile row strides = box widths
constexpr uint32_t TILE_Y_BYTES = 21 * TSY, TILE_C_BYTES = 13 * TSC;  // TMA boxes (engine.cu make_tensor_maps)

__constant__ uint32_t c_taps03[8] = {0x00800000u, 0x0c7bfa00u, 0x246cf502u, 0x325df700u, 0x4d4df003u, 0x5d32fa00u, 0x6c24f801u, 0x7b0cff00u};
__constant__ uint32_t c_taps45[8] = {0x0000u, 0x00ffu, 0x01f8u, 0x00fau, 0x03f0u, 0x00f7u, 0x02f5u, 0x00fau};

struct __align__(128) InterSmem {  // per warp
  union {
    struct {
      uint8_t y[1024];     // 21 rows x 48 B (TMA destination, 128-byte aligned)
      uint8_t u[512];      // 13 rows x 32 B
      uint8_t v[512];
      uint8_t mid_y[21 * 16];
      uint8_t mid_c[2][13 * 8];
    } n;
    struct {
      uint8_t win[24][9][12];  // SPLITMV: 9 x 9 window of every 4x4 block, window column 0 at byte 0
      uint8_t mid[24][9][4];
    } s;
  };
  uint8_t pix[384];            // Y 16x16 at 0, U 8x8 at 256, V 8x8 at 320
  int16_t coef[COEF_I16];
  unsigned long long bar;      // mbarrier
  uint8_t nzlist[24];
};

#ifndef VP8GPU_SIMT_EMUL
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, int x, int y, unsigned long long* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(dst)),
               "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
               : "memory");
}
// A tensor map in global memory that is MODIFIED while kernels can see it must be acquired (tensormap
// proxy) by the thread that uses it.  Ours are written once into never-reused arena slots before any
// kernel gets their address (engine.cu tmap_arena_alloc), so the fence is compiled out; building with
// -DVP8_TMAP_FENCE puts it back (9x slower k_inter, same results).
__device__ __forceinline__ void tmap_acquire(const void* tmap) {
#ifdef VP8_TMAP_FENCE
  asm volatile("fence.proxy.tensormap::generic.acquire.sys [%0], 128;" ::"l"(tmap) : "memory");
#else
  (void)tmap;
#endif
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
#else
// tests/simt: the copy is done at issue time, the barrier word counts the bytes still expected and flips bit 63
// when they have arrived (the kernel initialises the barrier for every macroblock and waits for phase 0 only)
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int) { *bar = 0; }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) { *bar = bytes; }
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, int x, int y, unsigned long long* bar) {
  *bar -= simt::tma_copy_2d(dst, tmap, x, y);
  if (*bar == 0) *bar = 1ull << 63;
}
__device__ __forceinline__ void tmap_acquire(const void*) {}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t) {
  while (!(*bar >> 63)) simt::yield();
}
#endif

// window that leaves the plane: pixel by pixel with clamped coordinates into the same tile layout
template <int TS>
__device__ __forceinline__ void stage_clamped(uint8_t* tile, const uint8_t* __restrict__ ref, int pitch, int PW, int PH, int wx,
                                              int wy, int wcols, int wrows, int lane) {
  for (int i = lane; i < wrows * wcols; i += 32) {
    const int r = i / wcols, c = i - r * wcols;
    tile[r * TS + c] = __ldg(ref + (size_t)clampi(wy + r, 0, PH - 1) * pitch + clampi(wx + c, 0, PW - 1));
  }
}

// rows: out[r][4g .. 4g+3] from tile[r][o + 4g .. o + 4g + 8]; o = byte offset of the window in a tile row
template <int N, int TS, int OS>
__device__ __forceinline__ void hpass2(const uint8_t* tile, int o, int nrows, int mx, uint8_t* out, int lane) {
  constexpr int G = N / 4;
  const uint32_t t03 = c_taps03[mx], t45 = c_taps45[mx];
  const int sh = 8 * (o & 3);
  for (int i = lane; i < nrows * G; i += 32) {
    const int r = i / G, g = i - r * G;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(tile + r * TS) + (o >> 2) + g;
    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
    *reinterpret_cast<uint32_t*>(out + r * OS + 4 * g) =
        vp8m::sixtap_h4(vp8m::bytes_at(w0, w1, sh), vp8m::bytes_at(w1, w2, sh), vp8m::bytes_at(w2, w3, sh), t03, t45);
  }
}
// the same walk without a filter (fraction 0): re-aligned copy of N pixels per row
template <int N, int TS, int OS>
__device__ __forceinline__ void hcopy(const uint8_t* tile, int o, int nrows, uint8_t* out, int lane) {
  constexpr int G = N / 4;
  const int sh = 8 * (o & 3);
  for (int i = lane; i < nrows * G; i += 32) {
    const int r = i / G, g = i - r * G;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(tile + r * TS) + (o >> 2) + g;
    *reinterpret_cast<uint32_t*>(out + r * OS + 4 * g) = vp8m::bytes_at(w[0], w[1], sh);
  }
}
// columns: R output rows of one pixel pair; s = &src[first input row][column], d = &dst[first output row][column]
template <int R>
__device__ __forceinline__ void vitem(const uint8_t* s, int ss, const int16_t* t, uint8_t* d, int ds) {
  uint32_t p[R + 5];
#pragma unroll
  for (int k = 0; k < R + 5; k++) p[k] = vp8m::pair_of(*reinterpret_cast<const uint16_t*>(s + k * ss));
#pragma unroll
  for (int j = 0; j < R; j++)
    *reinterpret_cast<uint16_t*>(d + j * ds) = (uint16_t)vp8m::sixtap_v2(p[j], p[j + 1], p[j + 2], p[j + 3], p[j + 4], p[j + 5], t);
}

// pixel = clamp255(prediction + residual) on the blocks of mask nz only; pix layout as in InterSmem
__device__ __forceinline__ void add_residuals(uint8_t* pix, const int16_t* coef, uint32_t nz, uint8_t* nzlist, int lane) {
  if ((nz >> lane) & 1) nzlist[__popc(nz & ((1u << lane) - 1))] = (uint8_t)lane;
  __syncwarp();
  const int n = 4 * __popc(nz);
  for (int i = lane; i < n; i += 32) {
    const int blk = nzlist[i >> 2], ry = i & 3;
    int off;
    if (blk < 16) off = ((blk >> 2) * 4 + ry) * 16 + (blk & 3) * 4;
    else off = 256 + ((blk - 16) >> 2) * 64 + (((blk >> 1) & 1) * 4 + ry) * 8 + (blk & 1) * 4;
    const uint2 r = *reinterpret_cast<const uint2*>(coef + blk * CS + ry * 4);
    uint32_t* p = reinterpret_cast<uint32_t*>(pix + off);
    *p = vp8m::add_residual4(*p, r.x, r.y);
  }
  __syncwarp();
}

__global__ void __launch_bounds__(INTER_WARPS * 32, 10) k_inter(const DevJob* __restrict__ jobs, Geom g) {
  __shared__ InterSmem s_all[INTER_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const DevJob& J = jobs[blockIdx.y];
  const int mbi = blockIdx.x * INTER_WARPS + warp;
  if (mbi >= g.mb_cols * g.mb_rows) return;
  const MbFields f = load_mb(J.mbs + mbi);
  if (f.ref == VP8GPU_REF_CURRENT) return;  // intra macroblocks belong to k_intra
  const int row = mbi / g.mb_cols, col = mbi - row * g.mb_cols;
  InterSmem& S = s_all[warp];
  uint8_t* const pix = S.pix;
  const uint8_t* ref = J.ref[f.ref - 1];
  const uint8_t* refU = ref + g.u_off;
  const uint8_t* refV = ref + g.v_off;
  const int CW = g.W >> 1, CH = g.H >> 1;
  uint32_t nz = 0;

  if (f.y_mode != VP8GPU_SPLITMV) {
    // ---- where the windows are: first pixel the filter needs, and how much of the tile it reads ----
    const int mx = f.mv_x & 7, my = f.mv_y & 7;
    const int X = 16 * col + (f.mv_x >> 3) - (mx ? 2 : 0), Y = 16 * row + (f.mv_y >> 3) - (my ? 2 : 0);
    const int ncols = 16 + (mx ? 5 : 0), nrows = 16 + (my ? 5 : 0);
    const bool fastY = X >= 0 && Y >= 0 && X + ncols <= g.W && Y + nrows <= g.H;
    const int cmvx = chroma_component(4 * f.mv_x), cmvy = chroma_component(4 * f.mv_y);
    const int cmx = cmvx & 7, cmy = cmvy & 7;
    const int CX = 8 * col + (cmvx >> 3) - (cmx ? 2 : 0), CY = 8 * row + (cmvy >> 3) - (cmy ? 2 : 0);
    const int cncols = 8 + (cmx ? 5 : 0), cnrows = 8 + (cmy ? 5 : 0);
    const bool fastC = CX >= 0 && CY >= 0 && CX + cncols <= CW && CY + cnrows <= CH;
    const uint32_t tx = (fastY ? TILE_Y_BYTES : 0u) + (fastC ? 2 * TILE_C_BYTES : 0u);
    const int oY = fastY ? (X & 15) : 0, oC = fastC ? (CX & 15) : 0;  // window's byte offset in a tile row
    if (lane == 0) mbar_init(&S.bar, 1);
    __syncwarp();
    if (lane == 0 && tx) {
      const uint8_t* maps = static_cast<const uint8_t*>(J.ref_tmap[f.ref - 1]);  // Y, U, V maps, 128 bytes each
      mbar_expect_tx(&S.bar, tx);
      if (fastY) {
        tmap_acquire(maps);
        tma_load_2d(S.n.y, maps, X & ~15, Y, &S.bar);
      }
      if (fastC) {
        tmap_acquire(maps + 128);
        tmap_acquire(maps + 256);
        tma_load_2d(S.n.u, maps + 128, CX & ~15, CY, &S.bar);
        tma_load_2d(S.n.v, maps + 256, CX & ~15, CY, &S.bar);
      }
    }
    // ---- residuals while the tiles travel (Macroblock::has_nonzero_, macroblock.cc:579,593) ----
    if (f.tok_cnt) nz = build_residuals(J, f, S.coef, lane);
    if (!fastY) stage_clamped<TSY>(S.n.y, ref, g.y_pitch, g.W, g.H, X, Y, ncols, nrows, lane);
    if (!fastC) {
      stage_clamped<TSC>(S.n.u, refU, g.c_pitch, CW, CH, CX, CY, cncols, cnrows, lane);
      stage_clamped<TSC>(S.n.v, refV, g.c_pitch, CW, CH, CX, CY, cncols, cnrows, lane);
    }
    if (tx) mbar_wait(&S.bar, 0);
    __syncwarp();

    // ---- luma 16x16: rows (filter or re-aligned copy), then columns on aligned data ----
    if (my == 0) {
      if (mx) hpass2<16, TSY, 16>(S.n.y, oY, 16, mx, pix, lane);
      else hcopy<16, TSY, 16>(S.n.y, oY, 16, pix, lane);
    } else {
      if (mx) hpass2<16, TSY, 16>(S.n.y, oY, 21, mx, S.n.mid_y, lane);
      else hcopy<16, TSY, 16>(S.n.y, oY, 21, S.n.mid_y, lane);
      __syncwarp();
      const int cp = lane & 7, rg = lane >> 3;
      vitem<4>(S.n.mid_y + (4 * rg) * 16 + 2 * cp, 16, c_sixtap[my], pix + (4 * rg) * 16 + 2 * cp, 16);
    }
    // ---- chroma 8x8, both planes ----
    if (cmy == 0) {
      if (cmx) {
        hpass2<8, TSC, 8>(S.n.u, oC, 8, cmx, pix + 256, lane);
        hpass2<8, TSC, 8>(S.n.v, oC, 8, cmx, pix + 320, lane);
      } else {
        hcopy<8, TSC, 8>(lane < 16 ? S.n.u : S.n.v, oC, 8, pix + (lane < 16 ? 256 : 320), lane & 15);
      }
    } else {
      if (cmx) {
        hpass2<8, TSC, 8>(S.n.u, oC, 13, cmx, S.n.mid_c[0], lane);
        hpass2<8, TSC, 8>(S.n.v, oC, 13, cmx, S.n.mid_c[1], lane);
      } else {
        hcopy<8, TSC, 8>(S.n.u, oC, 13, S.n.mid_c[0], lane);
        hcopy<8, TSC, 8>(S.n.v, oC, 13, S.n.mid_c[1], lane);
      }
      __syncwarp();
      const int plane = lane >> 4, cp = lane & 3, rg = (lane >> 2) & 3;
      vitem<2>(S.n.mid_c[plane] + (2 * rg) * 8 + 2 * cp, 8, c_sixtap[cmy], pix + 256 + 64 * plane + (2 * rg) * 8 + 2 * cp, 8);
    }
    __syncwarp();
  } else {
    // ---- SPLITMV (macroblock.cc:560-575): lane b < 24 owns block b: 0-15 luma, 16-19 U, 20-23 V ----
    if (f.tok_cnt) nz = build_residuals(J, f, S.coef, lane);
    int lmx = 0, lmy = 0;
    if (lane < 16) {
      const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(J.split + f.split_idx) + lane);
      lmx = (int16_t)(v & 0xFFFF);
      lmy = (int16_t)(v >> 16);
    }
    // chroma vector of 2x2 group q = (lane & 3): rounded average of four luma vectors (macroblock.cc:289-299)
    const int qa = ((lane >> 1) & 1) * 8 + (lane & 1) * 2;
    const int sx = __shfl_sync(0xffffffffu, lmx, qa) + __shfl_sync(0xffffffffu, lmx, qa + 1) + __shfl_sync(0xffffffffu, lmx, qa + 4) +
                   __shfl_sync(0xffffffffu, lmx, qa + 5);
    const int sy = __shfl_sync(0xffffffffu, lmy, qa) + __shfl_sync(0xffffffffu, lmy, qa + 1) + __shfl_sync(0xffffffffu, lmy, qa + 4) +
                   __shfl_sync(0xffffffffu, lmy, qa + 5);
    int bmvx = lmx, bmvy = lmy, bx0 = 16 * col + 4 * (lane & 3), by0 = 16 * row + 4 * ((lane >> 2) & 3);
    if (lane >= 16) {
      bmvx = chroma_component(sx), bmvy = chroma_component(sy);
      bx0 = 8 * col + 4 * (lane & 1), by0 = 8 * row + 4 * ((lane >> 1) & 1);
    }
    const int bX = bx0 + (bmvx >> 3) - 2, bY = by0 + (bmvy >> 3) - 2;  // window origin (always the full 9 x 9)
    const int bfx = bmvx & 7, bfy = bmvy & 7;
    // stage: item = (block, window row)
    for (int it = 0; it < 7; it++) {
      const int i = it * 32 + lane, b = min(i / 9, 23), r = i - 9 * (i / 9);
      const int wx = __shfl_sync(0xffffffffu, bX, b), wy = __shfl_sync(0xffffffffu, bY, b);
      if (i < 216) {
        const uint8_t* plane = b < 16 ? ref : (b < 20 ? refU : refV);
        const int pitch = b < 16 ? g.y_pitch : g.c_pitch, PW = b < 16 ? g.W : CW, PH = b < 16 ? g.H : CH;
        const uint8_t* rowp = plane + (size_t)clampi(wy + r, 0, PH - 1) * pitch;
        uint32_t a0, a1, a2;
        if (wx >= 0 && wx + 9 <= PW) {
          const int o = wx & 3;
          const uint32_t* wp = reinterpret_cast<const uint32_t*>(rowp + (wx - o));
          const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
          a0 = vp8m::bytes_at(w0, w1, 8 * o), a1 = vp8m::bytes_at(w1, w2, 8 * o), a2 = w2 >> (8 * o);
        } else {
          uint32_t px[9];
#pragma unroll
          for (int k = 0; k < 9; k++) px[k] = __ldg(rowp + clampi(wx + k, 0, PW - 1));
          a0 = px[0] | (px[1] << 8) | (px[2] << 16) | (px[3] << 24);
          a1 = px[4] | (px[5] << 8) | (px[6] << 16) | (px[7] << 24);
          a2 = px[8];
        }
        uint32_t* d = reinterpret_cast<uint32_t*>(S.s.win[b][r]);
        d[0] = a0, d[1] = a1, d[2] = a2;
      }
    }
    __syncwarp();
    // rows: item = (block, window row) -> 4 pixels of mid
    for (int it = 0; it < 7; it++) {
      const int i = it * 32 + lane, b = min(i / 9, 23), r = i - 9 * (i / 9);
      const int fx = __shfl_sync(0xffffffffu, bfx, b);
      if (i < 216) {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(S.s.win[b][r]);
        *reinterpret_cast<uint32_t*>(S.s.mid[b][r]) =
            fx ? vp8m::sixtap_h4(w[0], w[1], w[2], c_taps03[fx], c_taps45[fx]) : vp8m::bytes_at(w[0], w[1], 16);
      }
    }
    __syncwarp();
    // columns: item = (block, pixel pair) -> 4 rows x 2 pixels of the macroblock buffer
    for (int it = 0; it < 2; it++) {
      const int i = it * 32 + lane, b = min(i >> 1, 23), cp = i & 1;
      const int fy = __shfl_sync(0xffffffffu, bfy, b);
      if (i < 48) {
        uint8_t* d;
        int ds;
        if (b < 16) d = pix + ((b >> 2) * 4) * 16 + (b & 3) * 4 + 2 * cp, ds = 16;
        else d = pix + 256 + 64 * ((b - 16) >> 2) + (((b >> 1) & 1) * 4) * 8 + (b & 1) * 4 + 2 * cp, ds = 8;
        const uint8_t* m = &S.s.mid[b][0][2 * cp];
        if (fy) {
          vitem<4>(m, 4, c_sixtap[fy], d, ds);
        } else {
#pragma unroll
          for (int j = 0; j < 4; j++) *reinterpret_cast<uint16_t*>(d + j * ds) = *reinterpret_cast<const uint16_t*>(m + (j + 2) * 4);
        }
      }
    }
    __syncwarp();
  }

  if (nz) add_residuals(pix, S.coef, nz, S.nzlist, lane);
  store_mb(pix, J.out, g, col, row, lane);
}

// ================================================================================================
// wavefront plumbing
// ================================================================================================
#ifndef VP8GPU_SIMT_EMUL
__device__ __forceinline__ int ld_progress(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_progress(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
#else
__device__ __forceinline__ int ld_progress(const int* p) {
  simt::yield();  // tests/simt: a poll lets the other threads of the CTA run
  return *reinterpret_cast<const volatile int*>(p);
}
__device__ __forceinline__ void st_progress(int* p, int v) { *reinterpret_cast<volatile int*>(p) = v; }
#endif
// wait until the row above has finished every macroblock left of `need`
__device__ __forceinline__ void wait_row(const int* progress_above, int need, int lane) {
  if (lane == 0) {
    unsigned ns = 20;
    while (ld_progress(progress_above) < need) {
      __nanosleep(ns);
      if (ns < 160) ns += ns;  // mild back-off: a step of the row above takes a few microseconds
    }
  }
  __syncwarp();  // the other lanes' later loads are ordered after lane 0's acquire through this barrier
}
__device__ __forceinline__ void publish_row(int* progress, int value, int lane) {
  __syncwarp();  // every lane's stores happen-before lane 0's release store (cumulative at gpu scope)
  if (lane == 0) st_progress(progress, value);
}
__device__ __forceinline__ uint8_t ldcg_u8(const uint8_t* p) { return __ldcg(p); }

// next set bit at position >= from in a bitmask spread one 32-bit word per lane; -1 if none
__device__ __forceinline__ int next_marked(uint32_t my_word, int from, int nwords) {
  for (int w = from >> 5; w < nwords; w++) {
    uint32_t bits = __shfl_sync(0xffffffffu, my_word, w);
    if (w == (from >> 5)) bits &= 0xffffffffu << (from & 31);
    if (bits) return w * 32 + __ffs(bits) - 1;
  }
  return -1;
}

// ================================================================================================
// k_intra
// ================================================================================================
// Luma workspace with its borders, so that every edge of every sub-block is one address formula:
//   row 0            = the pixel row above the macroblock, x = -1 .. 19 (corner, 16 above, 4 above-right)
//   rows 1..16       = macroblock rows, byte 15 = the pixel left of the row, bytes 16..31 = the row
//   rows 4, 8, 12    additionally carry the 4 above-right pixels at bytes 32..35 (prediction.cc:153-160:
//                    the right-column sub-blocks of rows 1-3 use the row above the MACROBLOCK)
// pixel (x, y) lives at (y + 1) * WS + 16 + x; rows are 16-byte aligned for the vector stores.
constexpr int WS = 48;

__device__ __forceinline__ void add_residuals_intra(uint8_t* W, uint8_t* pixc, const int16_t* coef, int lane,
                                                    bool luma_too) {
  for (int g4 = (luma_too ? lane : 64 + lane); g4 < 96; g4 += 32) {
    int blk, ry;
    uint8_t* p;
    if (g4 < 64) {
      const int y = g4 >> 2, x4 = (g4 & 3) * 4;
      blk = (y >> 2) * 4 + (x4 >> 2);
      ry = y & 3;
      p = W + (y + 1) * WS + 16 + x4;
    } else {
      const int c = g4 - 64, plane = c >> 4, cc = c & 15;
      const int y = cc >> 1, x4 = (cc & 1) * 4;
      blk = 16 + plane * 4 + (y >> 2) * 2 + (x4 >> 2);
      ry = y & 3;
      p = pixc + plane * 64 + y * 8 + x4;
    }
    const int16_t* r = coef + blk * CS + ry * 4;
    const uint32_t v = *reinterpret_cast<uint32_t*>(p);
    uint32_t o = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) o |= (uint32_t)vp8m::clamp255((int)((v >> (8 * k)) & 0xFF) + r[k]) << (8 * k);
    *reinterpret_cast<uint32_t*>(p) = o;
  }
  __syncwarp();
}

// Two row-warps per CTA: an SM holds at most 32 CTAs, so single-warp CTAs would cap the rows in
// flight at 32 per SM (69 frames of 1080p per GPU); with two it is the full 64 warps per SM.
constexpr int WF_WARPS = 2;

// 24 CTAs x 2 warps resident per SM (40 registers per thread, no spills)
__global__ void __launch_bounds__(32 * WF_WARPS, 24) k_intra(const DevJob* __restrict__ jobs, int njobs, Geom g, int* ticket) {
  __shared__ __align__(16) uint8_t s_W[WF_WARPS][17 * WS];
  __shared__ __align__(16) uint8_t s_pixc[WF_WARPS][128];  // U 8x8, V 8x8
  __shared__ __align__(16) int16_t s_coef[WF_WARPS][COEF_I16];
  __shared__ uint8_t s_aboveC[WF_WARPS][2][12];  // [0] = above-left, [1..8] = above
  __shared__ uint8_t s_leftC[WF_WARPS][2][8];
  __shared__ uint16_t s_lut[WF_WARPS][128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* const W = s_W[warp];
  uint8_t* const pixc = s_pixc[warp];
  int16_t* const coef = s_coef[warp];
  uint8_t (*const aboveC)[12] = s_aboveC[warp];
  uint8_t (*const leftC)[8] = s_leftC[warp];
  uint16_t* const lut = s_lut[warp];
  for (int i = lane; i < 128; i += 32) lut[i] = k_bpred_lut[i];
  int t = 0;
  if (lane == 0) t = atomicAdd(ticket, 1);
  t = __shfl_sync(0xffffffffu, t, 0);
  const int row = t / njobs, job = t - row * njobs;
  if (row >= g.mb_rows) return;
  const DevJob& J = jobs[job];
  if (J.n_intra == 0) return;
  const int cols = g.mb_cols;
  const vp8gpu_mb* row_mbs = J.mbs + (size_t)row * cols;

  // which macroblocks of this row are intra-coded: bit c of a mask spread one word per lane
  const int nwords = (cols + 31) >> 5;
  uint32_t my_word = 0;
  for (int w = 0; w < nwords; w++) {
    const int c = w * 32 + lane;
    const bool intra = c < cols && (__ldg(reinterpret_cast<const uint32_t*>(row_mbs + c) + 2) & 0xFF) == VP8GPU_REF_CURRENT;
    const uint32_t bits = __ballot_sync(0xffffffffu, intra);
    if (lane == w) my_word = bits;
  }
  // the same mask for the row above: a macroblock only has to wait for the row above when one of the
  // macroblocks it predicts from (above-left, above, above-right) is intra-coded too -- inter-coded
  // neighbours were finished by k_inter before this kernel started
  uint32_t above_word = 0;
  if (row > 0)
    for (int w = 0; w < nwords; w++) {
      const int c = w * 32 + lane;
      const bool intra = c < cols && (__ldg(reinterpret_cast<const uint32_t*>(row_mbs - cols + c) + 2) & 0xFF) == VP8GPU_REF_CURRENT;
      const uint32_t bits = __ballot_sync(0xffffffffu, intra);
      if (lane == w) above_word = bits;
    }
  int col = next_marked(my_word, 0, nwords);
  int* progress = J.intra_progress + row;
  // progress = P means: every macroblock of this row with column < P is reconstructed
  publish_row(progress, col < 0 ? cols : col, lane);

  uint8_t* const Y = J.out;
  uint8_t* const U = J.out + g.u_off;
  uint8_t* const V = J.out + g.v_off;

  PROF_DECL;
  while (col >= 0) {
    PROF(7);
    const MbFields f = load_mb(row_mbs + col);
    // the residual only depends on this macroblock's tokens: build it before waiting on the row above
    const bool has_res = f.tok_cnt != 0;
    PROF(0);
    if (has_res) build_residuals(J, f, coef, lane);
    PROF(1);
    if (row > 0) {
      // highest intra-coded column among col-1, col, col+1 of the row above (-1: none, nothing to wait for)
      int dep = -1;
#pragma unroll
      for (int d = -1; d <= 1; d++) {
        const int c = col + d;
        const uint32_t word = __shfl_sync(0xffffffffu, above_word, (c >> 5) & 31);
        if (c >= 0 && c < cols && ((word >> (c & 31)) & 1)) dep = c;
      }
      if (dep >= 0) wait_row(progress - 1, dep + 1, lane);
    }
    PROF(2);

    // ---- edges (prediction.cc:99-167), read through L2; the three loads of a lane are issued
    //      back to back so their latencies overlap ----
    {
      const int outside_above = row == 0 ? 127 : 129;  // value of above[-1] when it is not a pixel
      // (a) luma above row incl. corner and above-right: lanes 0..20
      const uint8_t* pa = Y;
      bool va = false;
      if (lane < 21 && row > 0 && !(lane == 0 && col == 0)) {
        const int x = (lane >= 17 && col == cols - 1) ? 15 : lane - 1;  // replicate at the right frame edge
        pa = Y + (size_t)(16 * row - 1) * g.y_pitch + 16 * col + x;
        va = true;
      }
      // (b) left columns: lanes 0..15 luma, 16..23 U, 24..31 V
      const uint8_t* pb = Y;
      if (col > 0) {
        if (lane < 16) pb = Y + (size_t)(16 * row + lane) * g.y_pitch + 16 * col - 1;
        else pb = ((lane & 8) ? V : U) + (size_t)(8 * row + (lane & 7)) * g.c_pitch + 8 * col - 1;
      }
      // (c) chroma above rows incl. corner: lanes 0..17
      const uint8_t* pc = Y;
      bool vc = false;
      const int cpl = lane >= 9, ck = lane - 9 * cpl;
      if (lane < 18 && row > 0 && !(ck == 0 && col == 0)) {
        pc = (cpl ? V : U) + (size_t)(8 * row - 1) * g.c_pitch + 8 * col + ck - 1;
        vc = true;
      }
      const int a = va ? (int)ldcg_u8(pa) : outside_above;
      const int b = col > 0 ? (int)ldcg_u8(pb) : 129;
      const int c = vc ? (int)ldcg_u8(pc) : outside_above;
      if (lane < 21) W[15 + lane] = (uint8_t)a;
      if (lane < 16) W[(lane + 1) * WS + 15] = (uint8_t)b;
      else leftC[(lane >> 3) & 1][lane & 7] = (uint8_t)b;
      if (lane < 18) aboveC[cpl][ck] = (uint8_t)c;
    }
    __syncwarp();
    PROF(3);

    // ---- chroma 8x8 prediction (prediction.cc:435-449): one 4-pixel word per lane ----
    {
      const int plane = lane >> 4, y = (lane >> 1) & 7, x4 = (lane & 1) * 4;
      const uint8_t* A = aboveC[plane] + 1;
      const uint8_t* L = leftC[plane];
      uint32_t word;
      if (f.uv_mode == VP8GPU_DC_PRED) {
        int s = 0, n = 0;
        if (row > 0) { for (int k = 0; k < 8; k++) s += A[k]; n += 8; }
        if (col > 0) { for (int k = 0; k < 8; k++) s += L[k]; n += 8; }
        word = (uint32_t)(n == 16 ? (s + 8) >> 4 : (n == 8 ? (s + 4) >> 3 : 128)) * 0x01010101u;
      } else if (f.uv_mode == VP8GPU_V_PRED) {
        word = (uint32_t)A[x4] | ((uint32_t)A[x4 + 1] << 8) | ((uint32_t)A[x4 + 2] << 16) | ((uint32_t)A[x4 + 3] << 24);
      } else if (f.uv_mode == VP8GPU_H_PRED) {
        word = (uint32_t)L[y] * 0x01010101u;
      } else {
        const int base = L[y] - A[-1];
        word = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) word |= (uint32_t)vp8m::clamp255(base + A[x4 + k]) << (8 * k);
      }
      *reinterpret_cast<uint32_t*>(pixc + plane * 64 + y * 8 + x4) = word;
    }

    if (f.y_mode != VP8GPU_B_PRED) {
      // ---- luma 16x16 prediction (prediction.cc:451-467): 8 pixels (two words) per lane ----
      const int y = lane >> 1, x8 = (lane & 1) * 8;
      const uint8_t* A = W + 16;  // above[x]
      const int left = W[(y + 1) * WS + 15];
      uint32_t w0, w1;
      if (f.y_mode == VP8GPU_DC_PRED) {
        int s = 0, n = 0;
        if (row > 0) { for (int k = 0; k < 16; k++) s += A[k]; n += 16; }
        if (col > 0) { for (int k = 0; k < 16; k++) s += W[(k + 1) * WS + 15]; n += 16; }
        w0 = w1 = (uint32_t)(n == 32 ? (s + 16) >> 5 : (n == 16 ? (s + 8) >> 4 : 128)) * 0x01010101u;
      } else if (f.y_mode == VP8GPU_V_PRED) {
        w0 = *reinterpret_cast<const uint32_t*>(A + x8);
        w1 = *reinterpret_cast<const uint32_t*>(A + x8 + 4);
      } else if (f.y_mode == VP8GPU_H_PRED) {
        w0 = w1 = (uint32_t)left * 0x01010101u;
      } else {
        const int base = left - W[15];
        w0 = w1 = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          w0 |= (uint32_t)vp8m::clamp255(base + A[x8 + k]) << (8 * k);
          w1 |= (uint32_t)vp8m::clamp255(base + A[x8 + 4 + k]) << (8 * k);
        }
      }
      __syncwarp();  // all lanes have read the left column / above row they need
      *reinterpret_cast<uint32_t*>(W + (y + 1) * WS + 16 + x8) = w0;
      *reinterpret_cast<uint32_t*>(W + (y + 1) * WS + 20 + x8) = w1;
      __syncwarp();
      if (has_res) add_residuals_intra(W, pixc, coef, lane, true);
    } else {
      // ---- B_PRED: 16 sub-blocks in raster order, each predicted from reconstructed
      //      neighbours, residual added before the next one starts (macroblock.cc:540-545) ----
      if (lane < 12) W[(4 + 4 * (lane >> 2)) * WS + 32 + (lane & 3)] = W[32 + (lane & 3)];  // above-right copies
      __syncwarp();
      if (has_res) add_residuals_intra(W, pixc, coef, lane, false);  // chroma only
      const uint64_t modes = ((uint64_t)f.bm_hi << 32) | f.bm_lo;
      const int x = lane & 3, y = (lane >> 2) & 3;
#pragma unroll
      for (int b = 0; b < 16; b++) {  // fully unrolled: table entries and residuals load ahead of the chain
        const int bx = b & 3, by = b >> 2;
        const int mode = (int)((modes >> (4 * b)) & 15);
        // edge entry i of this sub-block: i < 4 -> left[3 - i], i = 4 -> above[-1], i > 4 -> above[i - 5]
        const uint8_t* e0 = W + (4 * by) * WS + 15 + 4 * bx;  // = above[-1]
        if (lane < 16) {
          int v;
          if (mode == VP8GPU_B_DC_PRED) {
            int s4 = 4;
#pragma unroll
            for (int k = 0; k < 4; k++) s4 += e0[1 + k] + e0[(1 + k) * WS];
            v = s4 >> 3;
          } else if (mode == VP8GPU_B_TM_PRED) {
            v = vp8m::clamp255(e0[(1 + y) * WS] + e0[1 + x] - e0[0]);
          } else {
            const unsigned entry = lut[(mode - 2) * 16 + lane];
            const int ia = entry & 15, ib = (entry >> 4) & 15, ic = (entry >> 8) & 15;
            const int pa = e0[ia < 4 ? (4 - ia) * WS : ia - 4];
            const int pb = e0[ib < 4 ? (4 - ib) * WS : ib - 4];
            const int pc = e0[ic < 4 ? (4 - ic) * WS : ic - 4];
            v = (entry & 0x1000) ? ((pa + 2 * pb + pc + 2) >> 2) : ((pa + pb + 1) >> 1);
          }
          if (has_res) v = vp8m::clamp255(v + coef[b * CS + lane]);
          W[(4 * by + y + 1) * WS + 16 + 4 * bx + x] = (uint8_t)v;
        }
        __syncwarp();
      }
    }
    __syncwarp();
    PROF(4);
    // ---- macroblock -> frame: 16-byte luma rows by lanes 0-15, 8-byte chroma rows by 16-31 ----
    if (lane < 16) {
      *reinterpret_cast<uint4*>(Y + (size_t)(16 * row + lane) * g.y_pitch + 16 * col) =
          *reinterpret_cast<const uint4*>(W + (lane + 1) * WS + 16);
    } else {
      const int plane = (lane - 16) >> 3, yy = lane & 7;
      *reinterpret_cast<uint2*>((plane ? V : U) + (size_t)(8 * row + yy) * g.c_pitch + 8 * col) =
          *reinterpret_cast<const uint2*>(pixc + plane * 64 + yy * 8);
    }
    const int next = next_marked(my_word, col + 1, nwords);
    PROF(5);
    publish_row(progress, next < 0 ? cols : next, lane);
    PROF(6);
    PROF_COUNT();
    col = next;
  }
  PROF_FLUSH(0);
}

// ================================================================================================
// k_loopfilter
// ================================================================================================
// One line of pixels across edges (a row for vertical edges, a column for horizontal ones), held in
// registers: px[0..3] = the 4 pixels before the macroblock, px[4..] = the macroblock's own.
// Edge order along the line = the reference's order for this direction (loopfilter.cc:133-154):
// macroblock edge (position 4) first, then the sub-block edges at 8, 12, 16 (chroma: 8 only).
__device__ __forceinline__ void filter_edge_at(int* px, int q, const vp8m::LfParams& lp, bool mb_edge) {
  const int mask = vp8m::lf_mask(lp.interior, mb_edge ? lp.mb_edge : lp.sub_edge, px[q - 4], px[q - 3], px[q - 2],
                                 px[q - 1], px[q], px[q + 1], px[q + 2], px[q + 3]);
  if (!mask) return;  // both filters are the identity when the mask is 0
  const int hev = vp8m::lf_hev(lp.hev, px[q - 2], px[q - 1], px[q], px[q + 1]);
  if (mb_edge) vp8m::lf_mbedge(mask, hev, px[q - 3], px[q - 2], px[q - 1], px[q], px[q + 1], px[q + 2]);
  else vp8m::lf_inner(mask, hev, px[q - 2], px[q - 1], px[q], px[q + 1]);
}
__device__ __forceinline__ void filter_line(int* px, bool luma, bool do_mb_edge, bool do_inner,
                                            const vp8m::LfParams& lp) {
  if (do_mb_edge) filter_edge_at(px, 4, lp, true);
  if (do_inner) {
    filter_edge_at(px, 8, lp, false);
    if (luma) {
      filter_edge_at(px, 12, lp, false);
      filter_edge_at(px, 16, lp, false);
    }
  }
}

// 16 CTAs x 2 warps resident per SM (64 registers per thread: a 20-pixel line lives in registers)
__global__ void __launch_bounds__(32 * WF_WARPS, 16) k_loopfilter(const DevJob* __restrict__ jobs, int njobs, Geom g, int* ticket) {
  // region = the macroblock plus 4 pixels above and to the left: luma 20x20, chroma 12x12
  constexpr int YS = 20, CSZ = 12;
  __shared__ __align__(16) uint8_t s_ry[WF_WARPS][20 * YS];
  __shared__ __align__(16) uint8_t s_rc[WF_WARPS][2][12 * CSZ];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* const ry = s_ry[warp];
  uint8_t (*const rc)[12 * CSZ] = s_rc[warp];
  int t = 0;
  if (lane == 0) t = atomicAdd(ticket, 1);
  t = __shfl_sync(0xffffffffu, t, 0);
  const int row = t / njobs, job = t - row * njobs;
  if (row >= g.mb_rows) return;
  const DevJob& J = jobs[job];
  if (!J.lf_enabled) return;
  const int cols = g.mb_cols;
  const vp8gpu_mb* row_mbs = J.mbs + (size_t)row * cols;

  const int nwords = (cols + 31) >> 5;
  uint32_t my_word = 0;
  for (int w = 0; w < nwords; w++) {
    const int c = w * 32 + lane;
    const bool filtered = c < cols && (J.lf_force || ((__ldg(reinterpret_cast<const uint32_t*>(row_mbs + c) + 2) >> 16) & 0xFF) != 0);
    const uint32_t bits = __ballot_sync(0xffffffffu, filtered);
    if (lane == w) my_word = bits;
  }
  int col = next_marked(my_word, 0, nwords);
  int* progress = J.lf_progress + row;
  publish_row(progress, col < 0 ? cols : col, lane);

  uint8_t* const Y = J.out;
  uint8_t* const U = J.out + g.u_off;
  uint8_t* const V = J.out + g.v_off;
  const int y_lo = row > 0 ? 0 : 4;  // first region row that exists in the frame

  // per-lane addressing of the three transfer patterns (all in 32-bit words)
  //  own block (3 words per lane): words 0-63 luma 16 rows x 4, 64-95 chroma 2 planes x 8 rows x 2
  //  top rows  (1 word per lane):  lanes 0-15 luma 4 rows x 4, lanes 16-31 chroma 2 x 4 rows x 2
  auto own_ptr = [&](int k, int c, const uint8_t*& gp, uint8_t*& sp) {
    const int w = lane + 32 * k;
    if (w < 64) {
      const int r = w >> 2, wx = w & 3;
      gp = Y + (size_t)(16 * row + r) * g.y_pitch + 16 * c + 4 * wx;
      sp = ry + (4 + r) * YS + 4 + 4 * wx;
    } else {
      const int cw = w - 64, plane = cw >> 4, k2 = cw & 15, r = k2 >> 1, wx = k2 & 1;
      gp = (plane ? V : U) + (size_t)(8 * row + r) * g.c_pitch + 8 * c + 4 * wx;
      sp = rc[plane] + (4 + r) * CSZ + 4 + 4 * wx;
    }
  };
  uint32_t own[3];
  auto prefetch_own = [&](int c) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const uint8_t* gp;
      uint8_t* sp;
      own_ptr(k, c, gp, sp);
      own[k] = __ldcg(reinterpret_cast<const uint32_t*>(gp));
    }
  };
  if (col >= 0) prefetch_own(col);
  int prev = -2;  // last column this warp filtered (its right 4 columns are still in shared memory)

  PROF_DECL;
  while (col >= 0) {
    PROF(7);
    const MbFields f = load_mb(row_mbs + col);
    const bool have_left = prev == col - 1;
    PROF(0);
    if (row > 0) wait_row(progress - 1, min(col + 2, cols), lane);
    PROF(1);

    // ---- top 4 rows (final output of the row above), through L2: one word per lane ----
    uint32_t top = 0;
    if (row > 0) {
      if (lane < 16) {
        const int r = lane >> 2, wx = lane & 3;
        top = __ldcg(reinterpret_cast<const uint32_t*>(Y + (size_t)(16 * row - 4 + r) * g.y_pitch + 16 * col + 4 * wx));
      } else {
        const int cw = lane - 16, plane = cw >> 3, k2 = cw & 7, r = k2 >> 1, wx = k2 & 1;
        top = __ldcg(reinterpret_cast<const uint32_t*>((plane ? V : U) + (size_t)(8 * row - 4 + r) * g.c_pitch + 8 * col + 4 * wx));
      }
    }
    // ---- left 4 columns: slide them over from the previous macroblock, or fetch them ----
    uint32_t left0 = 0, left1 = 0;
    if (col > 0) {
      if (have_left) {
        if (lane < 20) left0 = *reinterpret_cast<const uint32_t*>(ry + lane * YS + 16);
        if (lane < 24) left1 = *reinterpret_cast<const uint32_t*>(rc[lane / 12] + (lane % 12) * CSZ + 8);
      } else {
        if (lane < 20 && lane >= y_lo)
          left0 = __ldcg(reinterpret_cast<const uint32_t*>(Y + (size_t)(16 * row - 4 + lane) * g.y_pitch + 16 * col - 4));
        if (lane < 24 && (lane % 12) >= y_lo)
          left1 = __ldcg(reinterpret_cast<const uint32_t*>((lane / 12 ? V : U) + (size_t)(8 * row - 4 + lane % 12) * g.c_pitch + 8 * col - 4));
      }
    }
    __syncwarp();  // everybody has read the old region before it is overwritten
    if (col > 0) {
      if (lane < 20) *reinterpret_cast<uint32_t*>(ry + lane * YS) = left0;
      if (lane < 24) *reinterpret_cast<uint32_t*>(rc[lane / 12] + (lane % 12) * CSZ) = left1;
    }
    if (row > 0) {
      if (lane < 16) *reinterpret_cast<uint32_t*>(ry + (lane >> 2) * YS + 4 + 4 * (lane & 3)) = top;
      else {
        const int cw = lane - 16, plane = cw >> 3, k2 = cw & 7;
        *reinterpret_cast<uint32_t*>(rc[plane] + (k2 >> 1) * CSZ + 4 + 4 * (k2 & 1)) = top;
      }
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const uint8_t* gp;
      uint8_t* sp;
      own_ptr(k, col, gp, sp);
      *reinterpret_cast<uint32_t*>(sp) = own[k];
    }
    __syncwarp();
    PROF(2);
    const int next = next_marked(my_word, col + 1, nwords);
    if (next >= 0) prefetch_own(next);  // in flight while this macroblock is filtered

    const vp8m::LfParams lp = vp8m::lf_params(J.lf_force ? J.lf_force : f.lf_level, J.sharpness, J.key_frame);
    const bool do_inner = !((f.flags & VP8GPU_MB_HAS_Y2) && f.tok_cnt == 0);  // macroblock.cc:608
    // lane roles on an edge: 0-15 luma positions, 16-23 U, 24-31 V
    const bool luma = lane < 16;
    uint8_t* const plane_base = luma ? ry : rc[(lane - 16) >> 3];
    const int stride = luma ? YS : CSZ, idx = luma ? lane : (lane & 7), len = luma ? 20 : 12;
    int px[20];

    // ---- vertical edges: one region row (4 + idx) per lane, in registers ----
    {
      const uint32_t* rw = reinterpret_cast<const uint32_t*>(plane_base + (4 + idx) * stride);
#pragma unroll
      for (int k = 0; k < 5; k++) {
        const uint32_t v = (k < 3 || luma) ? rw[k] : 0u;
        px[4 * k] = v & 0xFF, px[4 * k + 1] = (v >> 8) & 0xFF, px[4 * k + 2] = (v >> 16) & 0xFF, px[4 * k + 3] = v >> 24;
      }
      filter_line(px, luma, col > 0, do_inner, lp);
      uint32_t* ww = reinterpret_cast<uint32_t*>(plane_base + (4 + idx) * stride);
#pragma unroll
      for (int k = 0; k < 5; k++)
        if (k < 3 || luma) ww[k] = (uint32_t)px[4 * k] | ((uint32_t)px[4 * k + 1] << 8) | ((uint32_t)px[4 * k + 2] << 16) | ((uint32_t)px[4 * k + 3] << 24);
    }
    __syncwarp();
    // ---- horizontal edges: one region column (4 + idx) per lane ----
    {
      uint8_t* cp = plane_base + 4 + idx;
#pragma unroll
      for (int k = 0; k < 20; k++) px[k] = k < len ? cp[k * stride] : 0;
      filter_line(px, luma, row > 0, do_inner, lp);
#pragma unroll
      for (int k = 1; k < 19; k++)
        if (k < len - 1) cp[k * stride] = (uint8_t)px[k];
    }
    __syncwarp();

    PROF(3);
    // ---- write back: region columns 0..15 (x -4..11); the last 4 columns travel with the next
    //      macroblock unless this warp will not filter it ----
    const int x_lo = col > 0 ? 0 : 1;
    const bool flush_right = next != col + 1;
    {
      uint8_t* const gy = Y + (size_t)(16 * row - 4) * g.y_pitch + 16 * col - 4;
#pragma unroll
      for (int k = 0; k < 3; k++) {  // luma words 0..79: 20 rows x 4 words
        const int w = lane + 32 * k, r = w >> 2, wx = w & 3;
        if (w < 80 && r >= y_lo && wx >= x_lo)
          *reinterpret_cast<uint32_t*>(gy + (size_t)r * g.y_pitch + 4 * wx) = *reinterpret_cast<const uint32_t*>(ry + r * YS + 4 * wx);
      }
#pragma unroll
      for (int k = 0; k < 2; k++) {  // chroma words 0..47: 2 planes x 12 rows x 2 words
        const int w = lane + 32 * k, plane = w >= 24, kk = w - 24 * plane, r = kk >> 1, wx = kk & 1;
        if (w < 48 && r >= y_lo && wx >= x_lo)
          *reinterpret_cast<uint32_t*>((plane ? V : U) + (size_t)(8 * row - 4 + r) * g.c_pitch + 8 * col - 4 + 4 * wx) =
              *reinterpret_cast<const uint32_t*>(rc[plane] + r * CSZ + 4 * wx);
      }
      if (flush_right) {
        if (lane < 20 && lane >= y_lo)
          *reinterpret_cast<uint32_t*>(gy + (size_t)lane * g.y_pitch + 16) = *reinterpret_cast<const uint32_t*>(ry + lane * YS + 16);
        if (lane < 24) {
          const int plane = lane >= 12, r = lane - 12 * plane;
          if (r >= y_lo)
            *reinterpret_cast<uint32_t*>((plane ? V : U) + (size_t)(8 * row - 4 + r) * g.c_pitch + 8 * col + 4) =
                *reinterpret_cast<const uint32_t*>(rc[plane] + r * CSZ + 8);
        }
      }
    }
    PROF(4);
    publish_row(progress, next < 0 ? cols : next, lane);
    PROF(5);
    PROF_COUNT();
    prev = col;
    col = next;
  }
  PROF_FLUSH(16);
}

#include "wavefront_ll.cuh"

// ================================================================================================
// ENCODER kernel (SURVEY.md 8a row a16): the reference's macroblock decision loop on the device.
//   key frames    luma_mb_best_prediction_mode incl. the B_PRED trial (encode_intra.cc:83-161, 360-387),
//                 chroma by minimum distortion (:250-285)
//   inter frames  16x16 intra modes against ZEROMV / NEARESTMV / NEARMV / NEWMV of the LAST frame with the
//                 motion-vector census, mode costs of the census, diamond search (encode_inter.cc:172-369)
//   both          rdcost (encoder.cc:410-416), variance / sse / sad (variance.cc:34-82), subtract_dct / wht
//                 (dct.cc:45-164), truncating quantiser (quantization.cc:148-178), and the reconstruction a
//                 decoder will perform (macroblock.cc:504-601).
// The decisions are the reference's integers in the reference's order (ties go to the earlier candidate), so
// at the same quantiser the records equal the ones parsed back from the reference encoder's own output
// (tests/test_gpu_encoder.py).  One warp per macroblock ROW, rows chained by progress counters (2-macroblock
// lag: intra prediction reads the above-right macroblock, the census the above and above-left records).
// ================================================================================================
__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }
__device__ __forceinline__ uint32_t rdcost(uint32_t rate, uint32_t distortion, uint32_t rm, uint32_t dm) {
  return ((128u + rate * rm) / 256u) + distortion * dm;
}
// Encoder::variance over 16x16: lanes hold partial sums of the differences and of their squares
__device__ __forceinline__ uint32_t variance256(int sum, int sse) {
  const long long s = warp_sum(sum);
  const uint32_t q = (uint32_t)warp_sum(sse);
  return q - (uint32_t)((s * s) / 256);
}

struct __align__(16) EncSmem {  // per warp
  uint8_t W[17 * WS];      // luma workspace with borders (see k_intra): final prediction / reconstruction
  uint8_t Wb[17 * WS];     // B_PRED trial reconstruction
  uint8_t src[384];
  uint8_t pcand[2][256];   // inter candidates: the one being tried, the best so far
  uint8_t pixc[128];
  uint8_t tile[21 * 24];
  uint8_t mid[21 * 16];
  int16_t coef[COEF_I16];
  int16_t qb[16][16];      // quantised coefficients of the B_PRED trial
  int16_t tmp[16];
  uint8_t aboveC[2][12];
  uint8_t leftC[2][8];
};

// 16x16 luma prediction of `mv` from the reference into dst (stride 16): Block<16>::inter_predict on a SafeRaster
// The window is staged like mc_block's (aligned words, or pixel by pixel with clamped coordinates when it leaves the
// plane), the filters are k_inter's packed ones (rows: two dp4a per output on re-aligned words, columns: 32-bit
// multiply-adds on pixel pairs) -- the motion search evaluates this a hundred times per searched macroblock.
__device__ __forceinline__ void enc_mc16_finish(const McPlan<16>& p, const EncJob& J, const Geom& g, uint8_t* dst, EncSmem& S, int lane) {
  constexpr int TS = Mc<16>::TS, NW = Mc<16>::NW;
  if (p.fast) {
    uint32_t* tw = reinterpret_cast<uint32_t*>(S.tile);
#pragma unroll
    for (int k = 0; k < McPlan<16>::K; k++) {
      const int i = lane + 32 * k;
      if (i < p.wsize * NW) tw[i] = p.regs[k];
    }
  } else {
    for (int i = lane; i < p.wsize * p.wsize; i += 32) {
      const int r = i / p.wsize, c = i - r * p.wsize;
      S.tile[r * TS + c] = __ldg(J.ref + (size_t)clampi(p.wy + r, 0, g.H - 1) * g.y_pitch + clampi(p.wx + c, 0, g.W - 1));
    }
  }
  __syncwarp();
  // window column / row 0 is pixel -2 of the block unless the vector is whole-pel (then it is the block itself)
  if ((p.mx | p.my) == 0) {
    hcopy<16, TS, 16>(S.tile, p.o, 16, dst, lane);
  } else if (p.my == 0) {
    hpass2<16, TS, 16>(S.tile + 2 * TS, p.o, 16, p.mx, dst, lane);
  } else {
    if (p.mx) hpass2<16, TS, 16>(S.tile, p.o, 21, p.mx, S.mid, lane);
    else hcopy<16, TS, 16>(S.tile, p.o + 2, 21, S.mid, lane);
    __syncwarp();
    const int cp = lane & 7, rg = lane >> 3;
    vitem<4>(S.mid + (4 * rg) * 16 + 2 * cp, 16, c_sixtap[p.my], dst + (4 * rg) * 16 + 2 * cp, 16);
  }
  __syncwarp();
}
__device__ __forceinline__ void enc_mc16(const EncJob& J, const Geom& g, int px, int py, int mvx, int mvy, uint8_t* dst,
                                         EncSmem& S, int lane) {
  McPlan<16> p;
  mc_plan<16>(p, J.ref, g.y_pitch, g.W, g.H, px, py, mvx, mvy, lane);
  enc_mc16_finish(p, J, g, dst, S, lane);
}
// both 8x8 chroma predictions of a macroblock (same vector): dst = U 8x8, dst + 64 = V 8x8, stride 8.  The two windows
// are requested together; staging and filtering as in enc_mc16.
__device__ __forceinline__ void enc_mc8_pair(const EncJob& J, const Geom& g, int CW, int CH, int px, int py, int mvx, int mvy,
                                             uint8_t* dst, EncSmem& S, int lane) {
  constexpr int TS = Mc<8>::TS, NW = Mc<8>::NW;
  McPlan<8> pl[2];
  mc_plan<8>(pl[0], J.ref + g.u_off, g.c_pitch, CW, CH, px, py, mvx, mvy, lane);
  mc_plan<8>(pl[1], J.ref + g.v_off, g.c_pitch, CW, CH, px, py, mvx, mvy, lane);
#pragma unroll
  for (int plane = 0; plane < 2; plane++) {
    const McPlan<8>& p = pl[plane];
    const uint8_t* ref = J.ref + (plane ? g.v_off : g.u_off);
    uint8_t* d = dst + 64 * plane;
    if (p.fast) {
      uint32_t* tw = reinterpret_cast<uint32_t*>(S.tile);
#pragma unroll
      for (int k = 0; k < McPlan<8>::K; k++) {
        const int i = lane + 32 * k;
        if (i < p.wsize * NW) tw[i] = p.regs[k];
      }
    } else {
      for (int i = lane; i < p.wsize * p.wsize; i += 32) {
        const int r = i / p.wsize, c = i - r * p.wsize;
        S.tile[r * TS + c] = __ldg(ref + (size_t)clampi(p.wy + r, 0, CH - 1) * g.c_pitch + clampi(p.wx + c, 0, CW - 1));
      }
    }
    __syncwarp();
    if ((p.mx | p.my) == 0) {
      hcopy<8, TS, 8>(S.tile, p.o, 8, d, lane);
    } else if (p.my == 0) {
      hpass2<8, TS, 8>(S.tile + 2 * TS, p.o, 8, p.mx, d, lane);
    } else {
      if (p.mx) hpass2<8, TS, 8>(S.tile, p.o, 13, p.mx, S.mid, lane);
      else hcopy<8, TS, 8>(S.tile, p.o + 2, 13, S.mid, lane);
      __syncwarp();
      if (lane < 16) {
        const int cp = lane & 3, rg = lane >> 2;
        vitem<2>(S.mid + (2 * rg) * 8 + 2 * cp, 8, c_sixtap[p.my], d + (2 * rg) * 8 + 2 * cp, 8);
      }
    }
    __syncwarp();
  }
}
__device__ __forceinline__ uint32_t enc_variance(const uint8_t* src, const uint8_t* pred, int lane) {
  const int o = (lane >> 1) * 16 + (lane & 1) * 8;
  int sum = 0, sse = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const int d = (int)src[o + k] - (int)pred[o + k];
    sum += d;
    sse += d * d;
  }
  return variance256(sum, sse);
}
__device__ __forceinline__ uint32_t enc_sad(const uint8_t* src, const uint8_t* pred, int lane) {
  const int o = (lane >> 1) * 16 + (lane & 1) * 8;
  int acc = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) acc += abs((int)src[o + k] - (int)pred[o + k]);
  return (uint32_t)warp_sum(acc);
}
// Scorer::clamp (macroblock.cc:183-195)
__device__ __forceinline__ void clamp_mv(int& x, int& y, int col, int row, int cols, int rows) {
  const int to_left = max(-((col * 16) << 3) - 128, -32768), to_right = min((((cols - 1 - col) * 16) << 3) + 128, 32767);
  const int to_top = max(-((row * 16) << 3) - 128, -32768), to_bottom = min((((rows - 1 - row) * 16) << 3) + 128, 32767);
  x = min(max(x, to_left), to_right);
  y = min(max(y, to_top), to_bottom);
}
// KeyFrameMacroblock::implied_subblock_mode
__device__ __forceinline__ int implied_bmode(int y_mode) {
  return y_mode == VP8GPU_V_PRED ? VP8GPU_B_VE_PRED : (y_mode == VP8GPU_H_PRED ? VP8GPU_B_HE_PRED : (y_mode == VP8GPU_TM_PRED ? VP8GPU_B_TM_PRED : VP8GPU_B_DC_PRED));
}

// Encoder::trellis_quantize (encoder.cc:220-408) of one block by one lane.  c: the block's transform coefficients in
// raster order (Y after Y2: DC already 0); on return the quantised values the trellis chose.  type: 0 Y after Y2,
// 1 Y2, 2 U / V, 3 Y without Y2; ctx: has_nonzero of the block above + of the block to the left.  Returns whether
// any value is non-zero.  Two candidate levels per position ({q, q - 1} towards zero), Viterbi from the last coded
// position back to the first with the reference's integer rate / distortion arithmetic.
__device__ __attribute__((noinline)) bool trellis_block(int16_t* c, int type, int dcq, int acq, int ctx, const TrellisTables& T, uint32_t RM, uint32_t DM) {
  constexpr uint8_t kZig[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
  constexpr uint8_t kBandOf[17] = {0, 1, 2, 3, 6, 4, 5, 6, 6, 6, 6, 6, 6, 6, 6, 7, 0};
  constexpr uint8_t kPrevClass[12] = {0, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 0};
  constexpr int EOB = 11;
  const int first = type == 0 ? 1 : 0;
  int coded = 0;
  for (int i = first; i < 16; i++)
    if (c[kZig[i]]) coded = i + 1;
  if (coded == 0) {
    for (int i = 0; i < 16; i++) c[i] = 0;
    return false;
  }
  uint32_t rate[17][2], dist[17][2], cost[17][2];
  int16_t coeff[17][2];
  uint8_t token[17][2], nxt[17][2];
  for (int i = 0; i < 2; i++) {
    rate[coded][i] = 0, dist[coded][i] = 0, cost[coded][i] = 0;
    token[coded][i] = EOB, coeff[coded][i] = 0, nxt[coded][i] = 255;
  }
  for (int idx = coded - 1; idx >= first; idx--) {
    const int factor = idx == 0 ? dcq : acq;
    const int16_t orig = c[kZig[idx]];
    const int16_t quantized = (int16_t)(orig / factor);
    for (int qs = 0; qs < 2; qs++) {
      int16_t cand = quantized;
      if (cand < 0) {
        cand = (int16_t)(cand + qs);
        if (cand > 0) cand = 0;
      } else if (cand > 0 || qs == 0) {
        cand = (int16_t)(cand - qs);
        if (cand < 0) cand = 0;
      } else {  // cand == 0 and qs != 0: the same node as level 0
        rate[idx][1] = rate[idx][0], dist[idx][1] = dist[idx][0], cost[idx][1] = cost[idx][0];
        coeff[idx][1] = coeff[idx][0], token[idx][1] = token[idx][0], nxt[idx][1] = nxt[idx][0];
        continue;
      }
      const int16_t diff = (int16_t)(orig - cand * factor);
      const uint32_t sse = (uint32_t)((int)diff * (int)diff);
      const int a = cand < 0 ? -cand : cand;
      const int tok = a <= 4 ? a : (a <= 6 ? 5 : (a <= 10 ? 6 : (a <= 18 ? 7 : (a <= 34 ? 8 : (a <= 66 ? 9 : 10)))));  // Costs::token_for_coeff
      uint32_t d2[2], r2[2], c2[2];
      int best_next = 255;
      uint32_t best_cost = 0xFFFFFFFFu;
      for (int n = 0; n < 2; n++) {
        d2[n] = dist[idx + 1][n] + sse;
        r2[n] = rate[idx + 1][n];
        if (idx < 15) r2[n] += T.token_cost[type][kBandOf[idx + 1]][kPrevClass[tok]][token[idx + 1][n]];
        c2[n] = rdcost(r2[n], d2[n], RM, DM);
        if (c2[n] < best_cost) best_cost = c2[n], best_next = n;
      }
      if (cand != 0 || token[idx + 1][best_next] != EOB) {
        coeff[idx][qs] = cand, token[idx][qs] = (uint8_t)tok;
        rate[idx][qs] = r2[best_next] + T.value_cost[cand + 2048];
        dist[idx][qs] = d2[best_next];
        cost[idx][qs] = c2[best_next];
        nxt[idx][qs] = (uint8_t)best_next;
      } else {  // a zero followed by the end of the block: the block ends here
        coeff[idx][qs] = 0, token[idx][qs] = EOB;
        rate[idx][qs] = 0;
        dist[idx][qs] = sse;
        cost[idx][qs] = rdcost(0, sse, RM, DM);
        nxt[idx][qs] = 255;
      }
    }
  }
  uint32_t min_cost = 0xFFFFFFFFu;
  int choice = 0;
  for (int i = 0; i < 2; i++) {
    rate[first][i] += T.token_cost[type][kBandOf[first]][ctx][token[first][i]];
    cost[first][i] = rdcost(rate[first][i], dist[first][i], RM, DM);
    if (cost[first][i] < min_cost) min_cost = cost[first][i], choice = i;
  }
  bool any = false;
  int i = first;
  for (; i < 16; i++) {
    if (token[i][choice] == EOB) break;
    c[kZig[i]] = coeff[i][choice];
    any |= coeff[i][choice] != 0;
    choice = nxt[i][choice];
  }
  for (; i < 16; i++) c[kZig[i]] = 0;
  return any;
}

template <bool TRELLIS>
__global__ void __launch_bounds__(32 * WF_WARPS, 8) k_enc_rd(const EncJob* __restrict__ jobp, int njobs, Geom g, int* ticket) {
  __shared__ EncSmem s_all[WF_WARPS];
  __shared__ uint16_t s_lut[128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 128; i += blockDim.x) s_lut[i] = k_bpred_lut[i];
  __syncthreads();
  EncSmem& S = s_all[warp];
  uint8_t* const W = S.W;
  uint8_t* const pixc = S.pixc;
  uint8_t* const src = S.src;
  int16_t* const coef = S.coef;
  int t = 0;
  if (lane == 0) t = atomicAdd(ticket, 1);
  t = __shfl_sync(0xffffffffu, t, 0);
  // ticket t -> row t / njobs of job t % njobs: the jobs of one launch are passes of the same shape (the size
  // estimates of a target-size search at different quantisers, encoder.cu estimate_batch), each with its own
  // output raster, records, token pool and progress counters; the row a warp waits for was claimed earlier
  const EncJob& J = jobp[t % njobs];
  const int row = t / njobs;
  const int cols = J.cols, rows = J.rows, sub = J.sub;
  if (row >= rows) return;
  int* progress = J.progress + row;
  uint8_t* const Y = J.out;
  uint8_t* const U = J.out + g.u_off;
  uint8_t* const V = J.out + g.v_off;
  const int CW = g.W >> 1, CH = g.H >> 1;
  const vp8gpu_quant q = J.q;
  const EncTables& T = *J.tab;
  const uint32_t RM = J.rate_mult, DM = J.dist_mult;
  const bool key = J.key_frame != 0;

  // what the census and the B_PRED contexts need from the macroblock to the left (this warp's previous one)
  bool left_inter = false;
  int left_mvx = 0, left_mvy = 0, left_ymode = VP8GPU_DC_PRED;
  unsigned long long left_bm = 0;
  // second pass of a two-pass key frame: has_nonzero of the 25 blocks of the macroblock to the left (bits 0-15 Y,
  // 16-19 U, 20-23 V, 24 Y2), the token contexts of the trellis (encoder.cc:362-363)
  uint32_t left_nz = 0;
  __shared__ uint8_t s_nz[TRELLIS ? WF_WARPS : 1][TRELLIS ? 32 : 1];

  for (int col = 0; col < cols; col++) {
    const int mbi = row * cols + col;
    const int scol = sub * col, srow = sub * row;  // source / reference position of this macroblock
    // ---- source macroblock (96 words) ----
    for (int i = lane; i < 96; i += 32) {
      const uint8_t* gp;
      if (i < 64) gp = J.src + (size_t)(16 * srow + (i >> 2)) * g.y_pitch + 16 * scol + 4 * (i & 3);
      else {
        const int c = i - 64, plane = c >> 4, k = c & 15;
        gp = J.src + (plane ? g.v_off : g.u_off) + (size_t)(8 * srow + (k >> 1)) * g.c_pitch + 8 * scol + 4 * (k & 1);
      }
      reinterpret_cast<uint32_t*>(src)[i] = __ldg(reinterpret_cast<const uint32_t*>(gp));
    }
    __syncwarp();
    // The row above must have finished the macroblock above; the one above-right too, but only where its pixels can
    // be used: by the sub-blocks of a B_PRED macroblock (prediction.cc:143-167).  Inter frames at REALTIME_QUALITY
    // never try B_PRED (encode_inter.cc:281), so their rows follow each other one macroblock apart instead of two --
    // (cols + rows) dependent steps per pass instead of (cols + 2 rows).  The above-right pixels are still fetched
    // below, possibly before they are final, and then not looked at.
    if (row > 0) wait_row(progress - 1, min(col + ((key || !J.realtime) ? 2 : 1), cols), lane);

    // ---- edges of the reconstruction so far (prediction.cc:99-167; same rules as k_intra) ----
    {
      const int outside_above = row == 0 ? 127 : 129;
      const uint8_t* pa = Y;
      bool va = false;
      if (lane < 21 && row > 0 && !(lane == 0 && col == 0)) {
        const int x = (lane >= 17 && col == cols - 1) ? 15 : lane - 1;
        pa = Y + (size_t)(16 * row - 1) * g.y_pitch + 16 * col + x;
        va = true;
      }
      const uint8_t* pb = Y;
      if (col > 0) {
        if (lane < 16) pb = Y + (size_t)(16 * row + lane) * g.y_pitch + 16 * col - 1;
        else pb = ((lane & 8) ? V : U) + (size_t)(8 * row + (lane & 7)) * g.c_pitch + 8 * col - 1;
      }
      const uint8_t* pc = Y;
      bool vc = false;
      const int cpl = lane >= 9, ck = lane - 9 * cpl;
      if (lane < 18 && row > 0 && !(ck == 0 && col == 0)) {
        pc = (cpl ? V : U) + (size_t)(8 * row - 1) * g.c_pitch + 8 * col + ck - 1;
        vc = true;
      }
      const int a = va ? (int)ldcg_u8(pa) : outside_above;
      const int b = col > 0 ? (int)ldcg_u8(pb) : 129;
      const int c = vc ? (int)ldcg_u8(pc) : outside_above;
      if (lane < 21) W[15 + lane] = (uint8_t)a;
      if (lane < 16) W[(lane + 1) * WS + 15] = (uint8_t)b;
      else S.leftC[(lane >> 3) & 1][lane & 7] = (uint8_t)b;
      if (lane < 18) S.aboveC[cpl][ck] = (uint8_t)c;
    }
    // the records above (census, B_PRED contexts): published by the row above before its progress moved on
    uint4 rec_a = make_uint4(0, 0, 0, 0), rec_al = make_uint4(0, 0, 0, 0);
    unsigned long long above_bm = 0;
    if (row > 0) {
      rec_a = __ldcg(reinterpret_cast<const uint4*>(J.mbs + mbi - cols));
      above_bm = __ldcg(reinterpret_cast<const unsigned long long*>(J.mbs + mbi - cols) + 3);
      if (col > 0) rec_al = __ldcg(reinterpret_cast<const uint4*>(J.mbs + mbi - cols - 1));
    }
    uint32_t above_nz = 0;
    if constexpr (TRELLIS) {
      if (row > 0) above_nz = __ldcg(reinterpret_cast<const uint32_t*>(J.mbs + mbi - cols) + 5);  // vp8gpu_mb::reserved
    }
    uint32_t trial_nz = 0;  // B_PRED trial: has_nonzero of its sub-blocks
    __syncwarp();

    const uint8_t* A = W + 16;  // above[x]
    // ================= luma: luma_mb_best_prediction_mode (encode_intra.cc:83-161) =================
    uint32_t best_cost = 0xFFFFFFFFu;
    int best_mode = VP8GPU_DC_PRED;
    unsigned long long bm = 0;  // B_PRED sub-block modes
    const bool try_bpred = key || !J.realtime;
    if (try_bpred) {
      // ---- B_PRED trial: sub-blocks in raster order, each chosen by rdcost(mode cost, sse of the prediction)
      //      and reconstructed before the next one is predicted ----
      uint8_t* const Wb = S.Wb;
      if (lane < 21) Wb[15 + lane] = W[15 + lane];
      if (lane < 16) Wb[(lane + 1) * WS + 15] = W[(lane + 1) * WS + 15];
      __syncwarp();
      if (lane < 12) Wb[(4 + 4 * (lane >> 2)) * WS + 32 + (lane & 3)] = Wb[32 + (lane & 3)];  // above-right copies
      __syncwarp();
      uint32_t rate = T.ymode_cost[key ? 0 : 1][VP8GPU_B_PRED], dist = 0;
      const int above_ymode = (rec_a.y >> 16) & 0xFF, above_ref = rec_a.z & 0xFF;
      const int half = lane >> 4, px = lane & 15, x = px & 3, y = px >> 2;
      for (int b = 0; b < 16; b++) {
        const int bx = b & 3, by = b >> 2;
        // context modes (encode_intra.cc:124-127): the sub-block above / to the left, B_DC_PRED outside the frame.
        // Those are the modes the reference's frame object holds: a 16x16 intra macroblock's implied ones
        // (encode_intra.cc:190), a B_PRED macroblock's own, and for an inter macroblock whatever its own losing B_PRED
        // trial wrote there (encode_intra.cc:65; luma_mb_apply_inter_prediction leaves them, encode_inter.cc:365-420)
        // -- the record's b_modes, which k_enc_rd fills for inter macroblocks of BEST_QUALITY inter frames
        int am, lm;
        if (by > 0) am = (int)((bm >> (4 * (b - 4))) & 15);
        else if (row == 0) am = VP8GPU_B_DC_PRED;
        else am = (above_ref != VP8GPU_REF_CURRENT || above_ymode == VP8GPU_B_PRED) ? (int)((above_bm >> (4 * (12 + bx))) & 15)
                                                                                   : implied_bmode(above_ymode);
        if (bx > 0) lm = (int)((bm >> (4 * (b - 1))) & 15);
        else if (col == 0) lm = VP8GPU_B_DC_PRED;
        else lm = (left_inter || left_ymode == VP8GPU_B_PRED) ? (int)((left_bm >> (4 * (4 * by + 3))) & 15) : implied_bmode(left_ymode);
        const uint16_t* mode_cost = T.bmode_cost[am][lm];
        const uint8_t* e0 = Wb + (4 * by) * WS + 15 + 4 * bx;  // = above[-1] of this sub-block
        const int sp = src[(4 * by + y) * 16 + 4 * bx + x];
        int pv[5];
        uint32_t best_err = 0xFFFFFFFFu, best_sse = 0;
        int best_b = 0;
#pragma unroll
        for (int r = 0; r < 5; r++) {  // two modes per round: lanes 0-15 mode 2r, lanes 16-31 mode 2r + 1
          const int mode = 2 * r + half;
          int v;
          if (mode == VP8GPU_B_DC_PRED) {
            int s4 = 4;
#pragma unroll
            for (int k = 0; k < 4; k++) s4 += e0[1 + k] + e0[(1 + k) * WS];
            v = s4 >> 3;
          } else if (mode == VP8GPU_B_TM_PRED) {
            v = vp8m::clamp255(e0[(1 + y) * WS] + e0[1 + x] - e0[0]);
          } else {
            const unsigned entry = s_lut[(mode - 2) * 16 + px];
            const int ia = entry & 15, ib = (entry >> 4) & 15, ic = (entry >> 8) & 15;
            const int pa = e0[ia < 4 ? (4 - ia) * WS : ia - 4];
            const int pb = e0[ib < 4 ? (4 - ib) * WS : ib - 4];
            const int pc = e0[ic < 4 ? (4 - ic) * WS : ic - 4];
            v = (entry & 0x1000) ? ((pa + 2 * pb + pc + 2) >> 2) : ((pa + pb + 1) >> 1);
          }
          pv[r] = v;
          int d2 = (sp - v) * (sp - v);
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
          const uint32_t sse_even = (uint32_t)__shfl_sync(0xffffffffu, d2, 0), sse_odd = (uint32_t)__shfl_sync(0xffffffffu, d2, 16);
          const uint32_t err_even = rdcost(mode_cost[2 * r], sse_even, RM, DM), err_odd = rdcost(mode_cost[2 * r + 1], sse_odd, RM, DM);
          if (err_even < best_err) best_err = err_even, best_b = 2 * r, best_sse = sse_even;
          if (err_odd < best_err) best_err = err_odd, best_b = 2 * r + 1, best_sse = sse_odd;
        }
        rate += mode_cost[best_b];
        dist += best_sse;
        bm |= (unsigned long long)best_b << (4 * b);
        // the chosen prediction of pixel px sits in lane (best_b & 1) * 16 + px, round best_b >> 1
        const int rr = best_b >> 1;
        const int mine = rr == 0 ? pv[0] : (rr == 1 ? pv[1] : (rr == 2 ? pv[2] : (rr == 3 ? pv[3] : pv[4])));
        const int pred = __shfl_sync(0xffffffffu, mine, (best_b & 1) * 16 + px);
        // luma_sb_apply_intra_prediction: subtract_dct, quantise (Y without Y2: the DC uses y_dc), reconstruct
        if (lane < 16) S.tmp[lane] = (int16_t)(sp - pred);
        __syncwarp();
        if (lane == 0) {
          int16_t d[16], o[16];
#pragma unroll
          for (int k = 0; k < 16; k++) d[k] = S.tmp[k];
          vp8m::fdct16(d, o);
          if constexpr (TRELLIS) {
            // luma_sb_apply_intra_prediction( ..., SECOND_PASS ) (encode_intra.cc:58-63): contexts from the sub-blocks
            // coded so far in this trial and from the neighbouring macroblocks
            const int ca = by > 0 ? (int)((trial_nz >> (b - 4)) & 1) : (row > 0 ? (int)((above_nz >> (12 + bx)) & 1) : 0);
            const int cl = bx > 0 ? (int)((trial_nz >> (b - 1)) & 1) : (col > 0 ? (int)((left_nz >> (4 * by + 3)) & 1) : 0);
            // trellis_quantize runs BEFORE set_Y_without_Y2 (encode_intra.cc:58-66): the sub-block still has the type
            // the FIRST pass left it with -- Y after Y2 unless that pass coded the macroblock as B_PRED -- and with
            // that type the trellis starts at position 1 and leaves the DC as the transform produced it
            const int ttype = (J.y2_prev[mbi] & 2) ? 3 : 0;
            bool any = trellis_block(o, ttype, q.y_dc, q.y_ac, ca + cl, *J.trellis, RM, DM);
            if (ttype == 0 && o[0] != 0) any = true;
            if (any) trial_nz |= 1u << b;
#pragma unroll
            for (int k = 0; k < 16; k++) {
              const int f = k ? q.y_ac : q.y_dc;
              S.qb[b][k] = o[k];
              d[k] = (int16_t)(o[k] * f);
            }
          } else {
#pragma unroll
            for (int k = 0; k < 16; k++) {
              const int f = k ? q.y_ac : q.y_dc;
              int qv = vp8m::quantize_trunc(o[k], f);
              qv = qv > 2047 ? 2047 : (qv < -2047 ? -2047 : qv);
              S.qb[b][k] = (int16_t)qv;
              d[k] = (int16_t)(qv * f);
            }
          }
          vp8m::idct16(d, o);
#pragma unroll
          for (int k = 0; k < 16; k++) S.tmp[k] = o[k];
        }
        __syncwarp();
        if (lane < 16) Wb[(4 * by + y + 1) * WS + 16 + 4 * bx + x] = (uint8_t)vp8m::clamp255(pred + S.tmp[lane]);
        __syncwarp();
      }
      best_cost = rdcost(rate, dist, RM, DM);
      best_mode = VP8GPU_B_PRED;
      if constexpr (TRELLIS) trial_nz = __shfl_sync(0xffffffffu, trial_nz, 0);  // lane 0 coded the sub-blocks
    }
    // ---- 16x16 modes, in the reference's order TM, H, V, DC; distortion = variance of the prediction ----
    {
      const int y = lane >> 1, x8 = (lane & 1) * 8;
      const int left = W[(y + 1) * WS + 15], corner = W[15];
      int dcY;
      {
        int s = 0, n = 0;
        if (row > 0) { for (int k = 0; k < 16; k++) s += A[k]; n += 16; }
        if (col > 0) { for (int k = 0; k < 16; k++) s += W[(k + 1) * WS + 15]; n += 16; }
        dcY = n == 32 ? (s + 16) >> 5 : (n == 16 ? (s + 8) >> 4 : 128);
      }
      int s_tm = 0, q_tm = 0, s_h = 0, q_h = 0, s_v = 0, q_v = 0, s_dc = 0, q_dc = 0;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int sp = src[y * 16 + x8 + k], ab = A[x8 + k];
        int d = sp - vp8m::clamp255(left + ab - corner);
        s_tm += d, q_tm += d * d;
        d = sp - left;
        s_h += d, q_h += d * d;
        d = sp - ab;
        s_v += d, q_v += d * d;
        d = sp - dcY;
        s_dc += d, q_dc += d * d;
      }
      const uint16_t* mc = T.ymode_cost[key ? 0 : 1];
      uint32_t c = rdcost(mc[VP8GPU_TM_PRED], variance256(s_tm, q_tm), RM, DM);
      if (c < best_cost) best_cost = c, best_mode = VP8GPU_TM_PRED;
      c = rdcost(mc[VP8GPU_H_PRED], variance256(s_h, q_h), RM, DM);
      if (c < best_cost) best_cost = c, best_mode = VP8GPU_H_PRED;
      c = rdcost(mc[VP8GPU_V_PRED], variance256(s_v, q_v), RM, DM);
      if (c < best_cost) best_cost = c, best_mode = VP8GPU_V_PRED;
      c = rdcost(mc[VP8GPU_DC_PRED], variance256(s_dc, q_dc), RM, DM);
      if (c < best_cost) best_cost = c, best_mode = VP8GPU_DC_PRED;
    }

    // ================= inter candidates: luma_mb_inter_predict (encode_inter.cc:231-369) =================
    int best_mvx = 0, best_mvy = 0, keep = 0;  // keep: which pcand buffer holds the best inter prediction
    if (!key) {
      // ---- census of the vectors above, left and above-left (Scorer, macroblock.cc:143-174; all LAST: no sign flips) ----
      int cmx[4] = {0, 0, 0, 0}, cmy[4] = {0, 0, 0, 0}, score[4] = {0, 0, 0, 0}, idx = 0;
      auto add = [&](int weight, bool inter, int vx, int vy) {
        if (!inter) return;
        if ((vx | vy) == 0) {
          score[0] += weight;
        } else {
          if (!(vx == cmx[idx] && vy == cmy[idx])) {
            idx++;
            cmx[idx] = vx, cmy[idx] = vy;
          }
          score[idx] += weight;
        }
      };
      if (row > 0) add(2, (rec_a.z & 0xFF) != VP8GPU_REF_CURRENT, (int16_t)(rec_a.w & 0xFFFF), (int16_t)(rec_a.w >> 16));
      if (col > 0) add(2, left_inter, left_mvx, left_mvy);
      if (row > 0 && col > 0) add(1, (rec_al.z & 0xFF) != VP8GPU_REF_CURRENT, (int16_t)(rec_al.w & 0xFFFF), (int16_t)(rec_al.w >> 16));
      if (score[3] && cmx[idx] == cmx[1] && cmy[idx] == cmy[1]) score[1] += score[3];
      if (score[2] > score[1]) {
        int tswap = score[1];
        score[1] = score[2], score[2] = tswap;
        tswap = cmx[1], cmx[1] = cmx[2], cmx[2] = tswap;
        tswap = cmy[1], cmy[1] = cmy[2], cmy[2] = tswap;
      }
      if (score[1] >= score[0]) cmx[0] = cmx[1], cmy[0] = cmy[1];
      int brx = cmx[0], bry = cmy[0], nrx = cmx[1], nry = cmy[1], nex = cmx[2], ney = cmy[2];
      clamp_mv(brx, bry, col, row, cols, rows);
      clamp_mv(nrx, nry, col, row, cols, rows);
      clamp_mv(nex, ney, col, row, cols, rows);
      // mode costs of this census (fill_mv_ref_costs; the split count is 0: the encoder never codes SPLITMV)
      const uint32_t c_zero = T.mvref_zero[0][score[0]];
      const uint32_t c_nearest = T.mvref_one[0][score[0]] + T.mvref_zero[1][score[1]];
      const uint32_t c_near = T.mvref_one[0][score[0]] + T.mvref_one[1][score[1]] + T.mvref_zero[2][score[2]];
      const uint32_t c_new = T.mvref_one[0][score[0]] + T.mvref_one[1][score[1]] + T.mvref_one[2][score[2]] + T.mvref_zero[3][0];
      const int px0 = 16 * scol, py0 = 16 * srow;
      int cur = 0;
      // a candidate = its prediction (window requested by mc_plan, filtered by enc_mc16_finish) and rdcost of its variance
      auto judge = [&](const McPlan<16>& pl, int mode, int vx, int vy, uint32_t rate) {
        enc_mc16_finish(pl, J, g, S.pcand[cur], S, lane);
        const uint32_t c = rdcost(rate, enc_variance(src, S.pcand[cur], lane), RM, DM);
        if (c < best_cost) {
          best_cost = c, best_mode = mode, best_mvx = vx, best_mvy = vy;
          keep = cur;
          cur ^= 1;
        }
      };
      auto consider = [&](int mode, int vx, int vy, uint32_t rate) {
        McPlan<16> pl;
        mc_plan<16>(pl, J.ref, g.y_pitch, g.W, g.H, px0, py0, vx, vy, lane);
        judge(pl, mode, vx, vy, rate);
      };
      {
        // ZEROMV, NEARESTMV, NEARMV in the reference's order, each window requested one candidate ahead
        const bool has_nearest = (nrx | nry) != 0, has_near = (nex | ney) != 0;
        McPlan<16> pa, pb;
        mc_plan<16>(pa, J.ref, g.y_pitch, g.W, g.H, px0, py0, 0, 0, lane);
        if (has_nearest) mc_plan<16>(pb, J.ref, g.y_pitch, g.W, g.H, px0, py0, nrx, nry, lane);
        judge(pa, VP8GPU_ZEROMV, 0, 0, c_zero);
        if (has_near) mc_plan<16>(pa, J.ref, g.y_pitch, g.W, g.H, px0, py0, nex, ney, lane);
        if (has_nearest) judge(pb, VP8GPU_NEARESTMV, nrx, nry, c_nearest);
        if (has_near) judge(pa, VP8GPU_NEARMV, nex, ney, c_near);
      }
      if (!J.realtime || ((col & 3) == 0 && (row & 3) == 0)) {
        // ---- NEWMV: repeated diamond searches around the census' best vector (encode_inter.cc:172-229, 279-293) ----
        int mvx = 0, mvy = 0;
        // The centre of a diamond is the best site of the diamond before it (or its centre again), whose cost was
        // computed then -- the cost of a site depends on its position only -- so it is remembered instead of predicted
        // and compared a second time; the comparison itself still happens in its place (third of five, strict <).
        uint32_t known_c = 0;
        int known_x = 0, known_y = 0;
        bool known = false;
        for (int step = 512; step > 1;) {
          int ox = mvx, oy = mvy, first_step = step / 2;
          for (int sz = step; sz > 1; sz >>= 1) {
            uint32_t bc = 0xFFFFFFFFu;
            int bx2 = 0, by2 = 0;  // MBPredictionData{}.mv: if every site is out of bounds the origin becomes (0, 0)
            // one site ahead: the window of site i + 1 is requested (mc_plan: loads into registers) before site i is
            // filtered and compared, so its latency hides behind that work
            McPlan<16> pending;
            int pcx = 0, pcy = 0;
            bool have = false, pcached = false;
#pragma unroll 1
            for (int site = 0; site <= 5; site++) {
              McPlan<16> next;
              int ncx = 0, ncy = 0;
              bool nvalid = false, ncached = false;
              if (site < 5) {
                const int dx = site == 0 ? -1 : (site == 4 ? 1 : 0), dy = site == 1 ? -1 : (site == 3 ? 1 : 0);
                ncx = ox + sz * dx, ncy = oy + sz * dy;
                nvalid = !(ncx > 1023 || ncx < -1023 || ncy > 1023 || ncy < -1023);
                ncached = nvalid && known && ncx == known_x && ncy == known_y;
                if (nvalid && !ncached) {
                  int tx = (int16_t)(ncx + brx), ty = (int16_t)(ncy + bry);
                  clamp_mv(tx, ty, col, row, cols, rows);
                  mc_plan<16>(next, J.ref, g.y_pitch, g.W, g.H, px0, py0, tx, ty, lane);
                }
              }
              if (have) {
                const int cx = pcx, cy = pcy;
                uint32_t c = known_c;
                if (!pcached) {
                  enc_mc16_finish(pending, J, g, S.pcand[cur], S, lane);
                  const uint32_t sad = enc_sad(src, S.pcand[cur], lane);
                  const int sx = max(min(cx >> 2, 255), -255), sy = max(min(cy >> 2, 255), -255);
                  const uint32_t rate =
                      J.mv_sad_zero ? 0u : ((uint32_t)(T.mv_sad_cost[abs(sy)] + T.mv_sad_cost[abs(sx)]) * J.sad_per_bit + 128u) / 256u;
                  c = ((128u + rate) / 256u) + sad;  // rdcost( rate, distortion, 1, 1 )
                }
                if (c < bc) bc = c, bx2 = cx, by2 = cy;
              }
              if (site < 5 && nvalid) {
                pending = next;
                pcx = ncx, pcy = ncy;
                pcached = ncached;
                have = true;
              } else if (site < 5) {
                have = false;
              }
            }
            known = bc != 0xFFFFFFFFu;
            known_c = bc, known_x = bx2, known_y = by2;
            if (bx2 == ox && by2 == oy) first_step = sz / 2;
            ox = bx2, oy = by2;
          }
          if (ox == mvx && oy == mvy) break;
          mvx = ox, mvy = oy;
          step = first_step;
        }
        const int dvx = mvx, dvy = mvy;  // mv - best_ref
        mvx = (int16_t)(mvx + brx), mvy = (int16_t)(mvy + bry);
        if (mvx | mvy) {
          const uint32_t mvc = J.mv_costs_zero ? 0u
                                               : (uint32_t)(T.mv_mag_cost[0][abs(dvy)] + (dvy ? T.mv_sign_cost[0][dvy < 0] : 0) +
                                                            T.mv_mag_cost[1][abs(dvx)] + (dvx ? T.mv_sign_cost[1][dvx < 0] : 0));
          consider(VP8GPU_NEWMV, mvx, mvy, c_new + (mvc * 96u) / 128u);
        }
      }
    }
    const bool inter = best_mode > VP8GPU_B_PRED;
    __syncwarp();

    // ================= chroma =================
    int uv_mode = VP8GPU_DC_PRED;
    const int cplane = lane >> 4, cy = (lane >> 1) & 7, cx4 = (lane & 1) * 4;
    if (inter) {
      const int cmvx = chroma_component(4 * best_mvx), cmvy = chroma_component(4 * best_mvy);
      enc_mc8_pair(J, g, CW, CH, 8 * scol, 8 * srow, cmvx, cmvy, pixc, S, lane);
    } else {
      // chroma_mb_best_prediction_mode (encode_intra.cc:250-285): smallest sse( U ) + sse( V ), DC V H TM, first wins
      int cdc[2];
#pragma unroll
      for (int plane = 0; plane < 2; plane++) {
        int s = 0, n = 0;
        if (row > 0) { for (int k = 0; k < 8; k++) s += S.aboveC[plane][1 + k]; n += 8; }
        if (col > 0) { for (int k = 0; k < 8; k++) s += S.leftC[plane][k]; n += 8; }
        cdc[plane] = n == 16 ? (s + 8) >> 4 : (n == 8 ? (s + 4) >> 3 : 128);
      }
      const uint8_t* CA = S.aboveC[cplane] + 1;
      const int cl = S.leftC[cplane][cy], ccorner = CA[-1], cd = cplane ? cdc[1] : cdc[0];
      int e0 = 0, e1 = 0, e2 = 0, e3 = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int sp = src[256 + cplane * 64 + cy * 8 + cx4 + k], ab = CA[cx4 + k];
        int d = sp - cd;
        e0 += d * d;
        d = sp - ab;
        e1 += d * d;
        d = sp - cl;
        e2 += d * d;
        d = sp - vp8m::clamp255(cl + ab - ccorner);
        e3 += d * d;
      }
      e0 = warp_sum(e0), e1 = warp_sum(e1), e2 = warp_sum(e2), e3 = warp_sum(e3);
      uint32_t bd = (uint32_t)e0;
      if ((uint32_t)e1 < bd) bd = e1, uv_mode = VP8GPU_V_PRED;
      if ((uint32_t)e2 < bd) bd = e2, uv_mode = VP8GPU_H_PRED;
      if ((uint32_t)e3 < bd) bd = e3, uv_mode = VP8GPU_TM_PRED;
      uint32_t word;
      if (uv_mode == VP8GPU_DC_PRED) word = (uint32_t)cd * 0x01010101u;
      else if (uv_mode == VP8GPU_V_PRED) word = (uint32_t)CA[cx4] | ((uint32_t)CA[cx4 + 1] << 8) | ((uint32_t)CA[cx4 + 2] << 16) | ((uint32_t)CA[cx4 + 3] << 24);
      else if (uv_mode == VP8GPU_H_PRED) word = (uint32_t)cl * 0x01010101u;
      else {
        const int base = cl - ccorner;
        word = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) word |= (uint32_t)vp8m::clamp255(base + CA[cx4 + k]) << (8 * k);
      }
      *reinterpret_cast<uint32_t*>(pixc + cplane * 64 + cy * 8 + cx4) = word;
    }
    __syncwarp();

    // ================= luma prediction into the workspace, residual, transforms =================
    const bool bpred = best_mode == VP8GPU_B_PRED;
    if (inter) {
      const uint8_t* pbest = S.pcand[keep];
      for (int i = lane; i < 64; i += 32) {
        const int y = i >> 2, x4 = (i & 3) * 4;
        *reinterpret_cast<uint32_t*>(W + (y + 1) * WS + 16 + x4) = *reinterpret_cast<const uint32_t*>(pbest + y * 16 + x4);
      }
    } else if (!bpred) {
      const int y = lane >> 1, x8 = (lane & 1) * 8;
      const int left = W[(y + 1) * WS + 15];
      uint32_t w0, w1;
      if (best_mode == VP8GPU_DC_PRED) {
        int s = 0, n = 0;
        if (row > 0) { for (int k = 0; k < 16; k++) s += A[k]; n += 16; }
        if (col > 0) { for (int k = 0; k < 16; k++) s += W[(k + 1) * WS + 15]; n += 16; }
        w0 = w1 = (uint32_t)(n == 32 ? (s + 16) >> 5 : (n == 16 ? (s + 8) >> 4 : 128)) * 0x01010101u;
      } else if (best_mode == VP8GPU_V_PRED) {
        w0 = *reinterpret_cast<const uint32_t*>(A + x8);
        w1 = *reinterpret_cast<const uint32_t*>(A + x8 + 4);
      } else if (best_mode == VP8GPU_H_PRED) {
        w0 = w1 = (uint32_t)left * 0x01010101u;
      } else {
        const int base = left - W[15];
        w0 = w1 = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          w0 |= (uint32_t)vp8m::clamp255(base + A[x8 + k]) << (8 * k);
          w1 |= (uint32_t)vp8m::clamp255(base + A[x8 + 4 + k]) << (8 * k);
        }
      }
      __syncwarp();
      *reinterpret_cast<uint32_t*>(W + (y + 1) * WS + 16 + x8) = w0;
      *reinterpret_cast<uint32_t*>(W + (y + 1) * WS + 20 + x8) = w1;
    }
    __syncwarp();
    // forward DCT, one 4x4 block per lane (B_PRED: the luma blocks were coded during the trial)
    if (lane < 24 && !(bpred && lane < 16)) {
      int16_t d[16], o[16];
      if (lane < 16) {
        const int bx = lane & 3, by = lane >> 2;
#pragma unroll
        for (int k = 0; k < 16; k++)
          d[k] = (int16_t)((int)src[(4 * by + (k >> 2)) * 16 + 4 * bx + (k & 3)] - (int)W[(4 * by + (k >> 2) + 1) * WS + 16 + 4 * bx + (k & 3)]);
      } else {
        const int c = lane - 16, plane = c >> 2, bx = c & 1, by = (c >> 1) & 1;
#pragma unroll
        for (int k = 0; k < 16; k++)
          d[k] = (int16_t)((int)src[256 + plane * 64 + (4 * by + (k >> 2)) * 8 + 4 * bx + (k & 3)] -
                           (int)pixc[plane * 64 + (4 * by + (k >> 2)) * 8 + 4 * bx + (k & 3)]);
      }
      vp8m::fdct16(d, o);
#pragma unroll
      for (int k = 0; k < 16; k++) coef[lane * CS + k] = o[k];
    }
    __syncwarp();
    if (!bpred && lane == 24) {  // Y2 = WHT of the sixteen luma DCs
      int16_t in[16], o[16];
#pragma unroll
      for (int k = 0; k < 16; k++) in[k] = coef[k * CS];
      vp8m::fwht16(in, o);
#pragma unroll
      for (int k = 0; k < 16; k++) coef[24 * CS + k] = o[k];
    }
    __syncwarp();
    // ---- quantise (truncating division), count tokens, dequantise in place ----
    int cnt = 0;
    int16_t qv[16];
    const bool has_blk = lane < 24 || (lane == 24 && !bpred);
    uint32_t mb_nz = 0;
    if constexpr (TRELLIS) {
      // SECOND_PASS (encode_intra.cc:199-219, 305-330): every block through trellis_quantize, whose first token is
      // priced in the context of the blocks above and to the left -- already requantised ones.  Blocks on the same
      // anti-diagonal of their plane are independent: seven rounds; Y2 (check_reset_y2 first) in the first one.
      uint8_t* const nz = s_nz[warp];
      if (lane < 25) nz[lane] = (bpred && lane < 16) ? (uint8_t)((trial_nz >> lane) & 1) : 0;
      __syncwarp();
      const int gx = lane < 16 ? (lane & 3) : (lane & 1), gy = lane < 16 ? (lane >> 2) : ((lane >> 1) & 1);
      const int diag = lane == 24 ? 0 : gx + gy;
      for (int round = 0; round < 7; round++) {
        if (has_blk && diag == round && !(bpred && lane < 16)) {
          int ca, cl, type;
          if (lane < 16) {
            type = 0;
            ca = gy > 0 ? nz[lane - 4] : (row > 0 ? (int)((above_nz >> (12 + gx)) & 1) : 0);
            cl = gx > 0 ? nz[lane - 1] : (col > 0 ? (int)((left_nz >> (4 * gy + 3)) & 1) : 0);
          } else if (lane < 24) {
            type = 2;
            const int base = lane & ~3;  // 16: U, 20: V
            ca = gy > 0 ? nz[lane - 2] : (row > 0 ? (int)((above_nz >> (base + 2 + gx)) & 1) : 0);
            cl = gx > 0 ? nz[lane - 1] : (col > 0 ? (int)((left_nz >> (base + 2 * gy + 1)) & 1) : 0);
          } else {
            type = 1;
            ca = row > 0 ? (int)((above_nz >> 24) & 1) : 0;
            cl = col > 0 ? (int)((left_nz >> 24) & 1) : 0;
          }
          const int dcq = lane < 16 ? q.y_dc : (lane < 24 ? q.uv_dc : q.y2_dc);
          const int acq = lane < 16 ? q.y_ac : (lane < 24 ? q.uv_ac : q.y2_ac);
          int16_t cc[16];
#pragma unroll
          for (int k = 0; k < 16; k++) cc[k] = coef[lane * CS + k];
          if (lane < 16) cc[0] = 0;  // Y after Y2: the DC travels in Y2
          if (lane == 24 && !(q.y2_dc >= 35 && q.y2_ac >= 35)) {  // Encoder::check_reset_y2 (encoder.cc:198-218)
            int sum = 0;
            bool keep = false;
            for (int k = 0; k < 16; k++) {
              sum += cc[k] < 0 ? -cc[k] : cc[k];
              if (sum >= 35) {
                keep = true;
                break;
              }
            }
            if (!keep)
              for (int k = 0; k < 16; k++) cc[k] = 0;
          }
          nz[lane] = trellis_block(cc, type, dcq, acq, ca + cl, *J.trellis, RM, DM) ? 1 : 0;
#pragma unroll
          for (int k = 0; k < 16; k++) {
            qv[k] = cc[k];
            cnt += cc[k] != 0;
            coef[lane * CS + k] = (int16_t)(cc[k] * (k ? acq : dcq));
          }
        }
        __syncwarp();
      }
      if (bpred && lane < 16) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
          const int v = S.qb[lane][k];
          qv[k] = (int16_t)v;
          cnt += v != 0;
          coef[lane * CS + k] = (int16_t)(v * (k ? q.y_ac : q.y_dc));
        }
      }
      // what the macroblocks to the right and below will see: a B_PRED macroblock leaves its Y2 block alone, so that
      // block still says what the first pass left there
      mb_nz = __ballot_sync(0xffffffffu, lane < 24 && nz[lane]);
      const uint32_t y2_flag = bpred ? (uint32_t)(J.y2_prev[mbi] & 1) : (uint32_t)nz[24];
      mb_nz = (mb_nz & 0x00FFFFFFu) | ((y2_flag & 1u) << 24);
    } else if (has_blk) {
      const int dcq = lane < 16 ? q.y_dc : (lane < 24 ? q.uv_dc : q.y2_dc);
      const int acq = lane < 16 ? q.y_ac : (lane < 24 ? q.uv_ac : q.y2_ac);
#pragma unroll
      for (int k = 0; k < 16; k++) {
        int v;
        if (bpred && lane < 16) {
          v = S.qb[lane][k];
        } else {
          int c = coef[lane * CS + k];
          if (lane < 16 && k == 0) c = 0;  // the luma DCs travel in Y2
          v = vp8m::quantize_trunc(c, k ? acq : dcq);
          v = v > 2047 ? 2047 : (v < -2047 ? -2047 : v);  // largest magnitude a DCT token carries is 2114
        }
        qv[k] = (int16_t)v;
        cnt += v != 0;
        coef[lane * CS + k] = (int16_t)(v * (k ? acq : dcq));  // DCTCoefficients::dequantize
      }
    }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t base = 0;
    if (lane == 0 && total) base = atomicAdd(J.tok_counter, (uint32_t)total);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (has_blk && cnt && base + total <= J.tok_cap) {
      uint32_t at = base + incl - cnt;
#pragma unroll
      for (int k = 0; k < 16; k++)
        if (qv[k]) J.tokens[at++] = VP8GPU_TOKEN(lane, k, qv[k]);
    }
    __syncwarp();
    if (inter && sub != 1) {
      // Encoder::estimate_size hands Macroblock::reconstruct_inter the macroblock of the SAMPLED grid, and
      // reconstruct_inter predicts from the raster position it is given (macroblock.cc:589-591): the
      // reconstruction of a sampled inter macroblock is the reference at (col, row) -- not (4 col, 4 row),
      // where the residual was taken -- plus that residual.  Reproduced, because the next macroblocks'
      // intra candidates are predicted from it and the size estimate steers the quantiser search.
      enc_mc16(J, g, 16 * col, 16 * row, best_mvx, best_mvy, S.pcand[0], S, lane);
      for (int i = lane; i < 64; i += 32) {
        const int y = i >> 2, x4 = (i & 3) * 4;
        *reinterpret_cast<uint32_t*>(W + (y + 1) * WS + 16 + x4) = *reinterpret_cast<const uint32_t*>(S.pcand[0] + y * 16 + x4);
      }
      const int cmvx = chroma_component(4 * best_mvx), cmvy = chroma_component(4 * best_mvy);
      enc_mc8_pair(J, g, CW, CH, 8 * col, 8 * row, cmvx, cmvy, pixc, S, lane);
      __syncwarp();
    }
    // ---- reconstruct exactly like a decoder will ----
    if (bpred) {
      // luma is the trial's reconstruction; chroma residual through the shared inverse transforms
      for (int i = lane; i < 64; i += 32) {
        const int y = i >> 2, x4 = (i & 3) * 4;
        *reinterpret_cast<uint32_t*>(W + (y + 1) * WS + 16 + x4) = *reinterpret_cast<const uint32_t*>(S.Wb + (y + 1) * WS + 16 + x4);
      }
      __syncwarp();
      if (total) {
        if (lane < 16) {  // no residual left to add to luma: blank the (dequantised) luma blocks
          uint2* cv = reinterpret_cast<uint2*>(coef + lane * CS);
#pragma unroll
          for (int k = 0; k < 4; k++) cv[k] = make_uint2(0u, 0u);
        }
        __syncwarp();
        inverse_transforms(coef, false, lane);
        add_residuals_intra(W, pixc, coef, lane, false);
      }
    } else if (total) {
      inverse_transforms(coef, true, lane);
      add_residuals_intra(W, pixc, coef, lane, true);
    }
    if (lane < 16) {
      *reinterpret_cast<uint4*>(Y + (size_t)(16 * row + lane) * g.y_pitch + 16 * col) = *reinterpret_cast<const uint4*>(W + (lane + 1) * WS + 16);
    } else {
      const int plane = (lane - 16) >> 3, yy = lane & 7;
      *reinterpret_cast<uint2*>((plane ? V : U) + (size_t)(8 * row + yy) * g.c_pitch + 8 * col) = *reinterpret_cast<const uint2*>(pixc + plane * 64 + yy * 8);
    }
    if (lane == 0) {
      vp8gpu_mb m;
      m.tok_off = base;
      m.tok_cnt = (uint16_t)total;
      m.y_mode = (uint8_t)best_mode;
      m.uv_mode = (uint8_t)(inter ? 0 : uv_mode);
      m.ref_frame = inter ? VP8GPU_REF_LAST : VP8GPU_REF_CURRENT;
      m.segment_id = 0;
      m.lf_level = J.lf_level;
      m.flags = bpred ? 0 : VP8GPU_MB_HAS_Y2;
      m.mv_x = (int16_t)(inter ? best_mvx : 0);
      m.mv_y = (int16_t)(inter ? best_mvy : 0);
      m.split_idx = 0;
      m.reserved = TRELLIS ? mb_nz : 0;  // second pass: the blocks' has_nonzero for the row below (cleared by the host)
      m.b_modes = (bpred || inter) ? bm : 0;  // inter: the trial's modes at BEST_QUALITY (context of the next trials), else 0
      J.mbs[mbi] = m;
    }
    left_inter = inter;
    left_mvx = inter ? best_mvx : 0;
    left_mvy = inter ? best_mvy : 0;
    left_ymode = best_mode;
    left_bm = (bpred || inter) ? bm : 0;
    if constexpr (TRELLIS) left_nz = mb_nz;
    publish_row(progress, col + 1, lane);
  }
}

#include "reencode.cuh"

// ================================================================================================
// k_compare: References::operator== (decoder.cc:249-254) on the device; flag != 0 when any visible
// pixel of the MB-aligned planes differs (pitch padding is ignored).
// ================================================================================================
__global__ void k_compare(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, Geom g, int* flag) {
  const int words_y = g.W / 4, words_c = g.W / 8;
  const int rows_total = g.H + g.H;  // H luma rows + H/2 U rows + H/2 V rows
  int diff = 0;
  for (int r = blockIdx.x; r < rows_total; r += gridDim.x) {
    size_t off;
    int nw;
    if (r < g.H) off = (size_t)r * g.y_pitch, nw = words_y;
    else if (r < g.H + g.H / 2) off = g.u_off + (size_t)(r - g.H) * g.c_pitch, nw = words_c;
    else off = g.v_off + (size_t)(r - g.H - g.H / 2) * g.c_pitch, nw = words_c;
    const uint32_t* pa = reinterpret_cast<const uint32_t*>(a + off);
    const uint32_t* pb = reinterpret_cast<const uint32_t*>(b + off);
    for (int i = threadIdx.x; i < nw; i += blockDim.x) diff |= (pa[i] != pb[i]);
  }
  if (diff) atomicOr(flag, 1);
}

// ================================================================================================
// k_ssim: BaseRaster::quality (util/raster.cc:63-66) = ssim( Y, other.Y ) over the macroblock-aligned
// luma planes, the measure the reference encoder maximises when it picks the loop-filter level
// (encoder.cc:489-508).  util/ssim.cc binds x264's pixel_ssim_wxh: sums over 4x4 blocks, combined over
// every 8x8 window at a 4-pixel step, float ratio per window, mean over (W/4-1)(H/4-1) windows
// (restated in oracle/ref_shim/ssim_stub.cc; parity with x264 itself is unpinned in this image).
// One thread per window writes the window's float (the same expression as x264's ssim_end1, no fused
// multiply-add in it); the host adds them in float in raster order like pixel_ssim_wxh does, so the value
// equals the CPU restatement's bit for bit (Engine::frames_ssim).
// ================================================================================================
__global__ void k_ssim(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, Geom g, float* out) {
  const int nx = g.W / 4 - 1, ny = g.H / 4 - 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nx * ny) {
    const int wy = i / nx, wx = i - wy * nx;
    const uint8_t* pa = a + (size_t)(4 * wy) * g.y_pitch + 4 * wx;
    const uint8_t* pb = b + (size_t)(4 * wy) * g.y_pitch + 4 * wx;
    int s1 = 0, s2 = 0, ss = 0, s12 = 0;
#pragma unroll
    for (int y = 0; y < 8; y++) {
      const uint32_t* ra = reinterpret_cast<const uint32_t*>(pa + (size_t)y * g.y_pitch);
      const uint32_t* rb = reinterpret_cast<const uint32_t*>(pb + (size_t)y * g.y_pitch);
#pragma unroll
      for (int w = 0; w < 2; w++) {
        const uint32_t xa = __ldg(ra + w), xb = __ldg(rb + w);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const int p = (xa >> (8 * k)) & 0xFF, q = (xb >> (8 * k)) & 0xFF;
          s1 += p;
          s2 += q;
          ss += p * p + q * q;
          s12 += p * q;
        }
      }
    }
    const int c1 = (int)(.01 * .01 * 255 * 255 * 64 + .5);
    const int c2 = (int)(.03 * .03 * 255 * 255 * 64 * 63 + .5);
    const int vars = ss * 64 - s1 * s1 - s2 * s2, covar = s12 * 64 - s1 * s2;
    out[i] = __fdiv_rn(__fmul_rn((float)(2 * s1 * s2 + c1), (float)(2 * covar + c2)),
                       __fmul_rn((float)(s1 * s1 + s2 * s2 + c1), (float)(vars + c2)));
  }
}

// ================================================================================================
// k_hash: a 64-bit content hash of the visible pixels of a raster (HashCachedRaster::hash,
// raster_handle.hh:60-75, is the reference's analogue; the value is ours, not boost's).  Position
// dependent, order independent in evaluation: sum over 32-bit words of mix(word, plane row, index).
// ================================================================================================
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x ^= x >> 33;
  x *= 0xff51afd7ed558ccdull;
  x ^= x >> 33;
  x *= 0xc4ceb9fe1a85ec53ull;
  x ^= x >> 33;
  return x;
}
__global__ void k_hash(const uint8_t* __restrict__ a, Geom g, unsigned long long* out) {
  const int words_y = g.W / 4, words_c = g.W / 8;
  const int rows_total = g.H + g.H;
  unsigned long long acc = 0;
  for (int r = blockIdx.x; r < rows_total; r += gridDim.x) {
    size_t off;
    int nw;
    if (r < g.H) off = (size_t)r * g.y_pitch, nw = words_y;
    else if (r < g.H + g.H / 2) off = g.u_off + (size_t)(r - g.H) * g.c_pitch, nw = words_c;
    else off = g.v_off + (size_t)(r - g.H - g.H / 2) * g.c_pitch, nw = words_c;
    const uint32_t* pa = reinterpret_cast<const uint32_t*>(a + off);
    for (int i = threadIdx.x; i < nw; i += blockDim.x)
      acc += mix64(((unsigned long long)pa[i] << 32) ^ ((unsigned long long)r << 16) ^ (unsigned long long)i);
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

}  // namespace

// ================================================================================================
// launchers
// ================================================================================================
int launch_inter(const DevJob* jobs, int njobs, const Geom& g, void* stream) {
  const int n_mbs = g.mb_cols * g.mb_rows;
  dim3 grid((n_mbs + INTER_WARPS - 1) / INTER_WARPS, njobs);
  VP8_LAUNCH(k_inter, grid, INTER_WARPS * 32, 0, static_cast<cudaStream_t>(stream))(jobs, g);
  return (int)cudaGetLastError();
}
int launch_intra(const DevJob* jobs, int njobs, const Geom& g, int* ticket, uint32_t epoch, void* stream) {
  const int grid = (g.mb_rows * njobs + WF_WARPS - 1) / WF_WARPS;
  if (epoch) VP8_LAUNCH(k_intra_ll, grid, 32 * WF_WARPS, 0, static_cast<cudaStream_t>(stream))(jobs, njobs, g, ticket, epoch);
  else VP8_LAUNCH(k_intra, grid, 32 * WF_WARPS, 0, static_cast<cudaStream_t>(stream))(jobs, njobs, g, ticket);
  return (int)cudaGetLastError();
}
int launch_loopfilter(const DevJob* jobs, int njobs, const Geom& g, int* ticket, uint32_t epoch, void* stream) {
  const int grid = (g.mb_rows * njobs + WF_WARPS - 1) / WF_WARPS;
  if (epoch) VP8_LAUNCH(k_loopfilter_ll, grid, 32 * WF_WARPS, 0, static_cast<cudaStream_t>(stream))(jobs, njobs, g, ticket, epoch);
  else VP8_LAUNCH(k_loopfilter, grid, 32 * WF_WARPS, 0, static_cast<cudaStream_t>(stream))(jobs, njobs, g, ticket);
  return (int)cudaGetLastError();
}

int launch_enc_rd(const EncJob* jobs, int njobs, int rows, const Geom& g, int* ticket, void* stream) {
  VP8_LAUNCH(k_enc_rd<false>, (njobs * rows + WF_WARPS - 1) / WF_WARPS, 32 * WF_WARPS, 0, static_cast<cudaStream_t>(stream))(jobs, njobs, g, ticket);
  return (int)cudaGetLastError();
}
int launch_enc_rd_trellis(const EncJob* job, int rows, const Geom& g, int* ticket, void* stream) {
  VP8_LAUNCH(k_enc_rd<true>, (rows + WF_WARPS - 1) / WF_WARPS, 32 * WF_WARPS, 0, static_cast<cudaStream_t>(stream))(job, 1, g, ticket);
  return (int)cudaGetLastError();
}

int launch_reenc_inter(const ReencJob* job, int n_mbs, const Geom& g, void* stream) {
  VP8_LAUNCH(k_reenc_inter, (n_mbs + REENC_WARPS - 1) / REENC_WARPS, 32 * REENC_WARPS, 0, static_cast<cudaStream_t>(stream))(job, g);
  return (int)cudaGetLastError();
}
int launch_reenc_intra(const ReencJob* job, int rows, const Geom& g, int* ticket, void* stream) {
  VP8_LAUNCH(k_reenc_intra, (rows + WF_WARPS - 1) / WF_WARPS, 32 * WF_WARPS, 0, static_cast<cudaStream_t>(stream))(job, g, ticket);
  return (int)cudaGetLastError();
}

#ifdef VP8_PROFILE
extern "C" void vp8gpu_debug_profile(unsigned long long out[32], int reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, g_prof, sizeof(unsigned long long) * 32);
  if (reset) {
    unsigned long long z[32] = {0};
    cudaMemcpyToSymbol(g_prof, z, sizeof(z));
  }
}
#endif

// Batch header (job descriptors + zeroed tickets / counters) from mapped pinned host memory into HBM, read over
// PCIe by one thread block.  A cudaMemcpyAsync would queue behind whatever the copy engines are busy with -- in
// vp8gpu_decode_ivf that is megabytes of bitstream staged by the workers -- and stall the pixel batch for
// milliseconds (profiles/r2_notes.md); a 30 KB read by the SMs takes microseconds.
__global__ void k_fetch_header(uint4* __restrict__ dst, const uint4* __restrict__ src_host, int n16) {
  for (int i = threadIdx.x; i < n16; i += blockDim.x) dst[i] = src_host[i];
}
int launch_fetch_header(void* dst, const void* src_host_devptr, size_t bytes, void* stream) {
  VP8_LAUNCH(k_fetch_header, 1, 512, 0, static_cast<cudaStream_t>(stream))(static_cast<uint4*>(dst), static_cast<const uint4*>(src_host_devptr),
                                                                 (int)(bytes / 16));
  return (int)cudaGetLastError();
}

int launch_hash(const uint8_t* a, const Geom& g, unsigned long long* d_out, void* stream) {
  VP8_LAUNCH(k_hash, 296, 128, 0, static_cast<cudaStream_t>(stream))(a, g, d_out);
  return (int)cudaGetLastError();
}

int launch_ssim(const uint8_t* a, const uint8_t* b, const Geom& g, float* d_windows, void* stream) {
  const int n = (g.W / 4 - 1) * (g.H / 4 - 1);
  if (n <= 0) return 0;
  VP8_LAUNCH(k_ssim, (n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream))(a, b, g, d_windows);
  return (int)cudaGetLastError();
}

int launch_compare(const uint8_t* a, const uint8_t* b, const Geom& g, int* d_flag, void* stream) {
  VP8_LAUNCH(k_compare, 296, 128, 0, static_cast<cudaStream_t>(stream))(a, b, g, d_flag);
  return (int)cudaGetLastError();
}

}  // namespace vp8
