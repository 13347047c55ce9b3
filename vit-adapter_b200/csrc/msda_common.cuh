// msda_common.cuh — shared device helpers for the sm_100a multi-scale deformable attention kernels.
//
// Arithmetic contract (what the reference computes; SURVEY.md App. A):
//   reference forward  : detection/ops/src/cuda/ms_deform_im2col_cuda.cuh:237-299 (+ bilinear :33-84)
//   reference backward : detection/ops/src/cuda/ms_deform_im2col_cuda.cuh:301-510 (+ bilinear :87-159)
// The pixel coordinate is ONE fused multiply-add, fmaf(loc, (float)H, -0.5f): that is how nvcc
// compiles the reference's `loc_h * spatial_h - 0.5` (SASS: FFMA R, (float)H, loc, -0.5), and
// bit-exact index parity with the reference kernel depends on it.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <type_traits>

#include "../../include/msda_b200.h"

namespace msda {

// SMs of the current device (cudaDevAttrMultiProcessorCount, cached per device ordinal; 148 - a B200 - if the query fails).
// Host side: the launchers size persistent grids and CTA chunks with it.
inline int device_sm_count() {
  static std::atomic<int> cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  int n = cache[dev].load();
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev].store(n);
  }
  return n;
}

constexpr int kThreads = 256;            // threads per CTA for every kernel in this library
constexpr int kWarps = kThreads / 32;
constexpr int kMaxLevels = MSDA_MAX_LEVELS;

// Kernel parameter block (passed by value; lives in constant bank).
struct Params {
  const void* value;
  const int64_t* shapes;  // [L,2] (H,W) on device
  const int64_t* lsi;     // [L]       on device
  const void* loc;
  const void* aw;
  void* out;               // fwd: out ; bwd: unused
  const void* grad_out;    // bwd
  void* grad_value;        // bwd: dtype T, or fp32 scratch when T = bf16
  void* grad_loc;          // bwd
  void* grad_aw;           // bwd
  int N, S, M, D, L, Lq, P;
  int qc;                  // queries per CTA chunk
  int nchunk;              // ceil(Lq / qc)
  // fused entry points only: `loc` holds RAW sampling offsets, `aw` RAW attention logits, and the
  // locations / softmax are formed in registers from the reference points below
  const float* ref;        // reference points [Nr, Lq, Lr, RD], RD = ref_dim
  long long ref_bstride;   // floats between batches (0 when Nr == 1: broadcast)
  int ref_qstride;         // floats between queries (= Lr * RD)
  int ref_lstride;         // floats between levels  (0 when Lr == 1: broadcast)
  long long off_rowstride;   // floats between the offsets of consecutive (b,q) rows (dense: M*L*P*2); same for their gradient
  long long logit_rowstride; // floats between the logits  of consecutive (b,q) rows (dense: M*L*P);   same for their gradient
  int ref_dim;             // 2: points (x, y); 4: boxes (x, y, w, h)
  float* ref_partial;      // fused bwd: NULL, or the per-(b, q, m, lr) reference-point gradient partials [N, Lq, M, Lr, RD]
};

// Host-made plan for the shared-memory forward (msda_fwd_smem.cu): which levels' [H*W, D] maps of one
// head are staged in shared memory, and where. Needs the level shapes on the HOST.
constexpr unsigned kSmemBudget = 226u * 1024u;  // dynamic shared memory a CTA may use (227 KB max per CTA)
struct SmemPlan {
  unsigned staged;       // bit l = level l is staged
  unsigned total_bytes;  // dynamic shared memory = sum of staged maps
  int H[kMaxLevels], W[kMaxLevels], start[kMaxLevels];
  unsigned smem_off[kMaxLevels];
};

// ---------------------------------------------------------------------------------------------
// Geometry of one sampling point. Mirrors ms_deform_im2col_cuda.cuh:285-288 (coordinate + bounds
// test) and :38-78 (floor, fractions, per-corner validity).
// mask bit0: corner1 (h_low ,w_low ) readable     bit1: corner2 (h_low ,w_high)
//      bit2: corner3 (h_high,w_low )              bit3: corner4 (h_high,w_high)
// mask == 0 when the sample fails the bounds test (the reference skips it entirely).
// ---------------------------------------------------------------------------------------------
template <typename F>
struct PointGeom {
  int h_low, w_low;
  F lh, lw;
  unsigned mask;
};

__device__ __forceinline__ float msda_fma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double msda_fma(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float msda_floor(float a) { return floorf(a); }
__device__ __forceinline__ double msda_floor(double a) { return floor(a); }

template <typename F>
__device__ __forceinline__ PointGeom<F> point_geom(F loc_w, F loc_h, int H, int W) {
  PointGeom<F> g;
  const F h_im = msda_fma(loc_h, (F)H, (F)-0.5);
  const F w_im = msda_fma(loc_w, (F)W, (F)-0.5);
  const bool inside = (h_im > (F)-1) && (w_im > (F)-1) && (h_im < (F)H) && (w_im < (F)W);
  const F hf = msda_floor(h_im);
  const F wf = msda_floor(w_im);
  g.h_low = inside ? (int)hf : 0;
  g.w_low = inside ? (int)wf : 0;
  g.lh = inside ? (h_im - hf) : (F)0;
  g.lw = inside ? (w_im - wf) : (F)0;
  unsigned m = 0;
  if (inside) {
    const bool t = g.h_low >= 0, b = g.h_low + 1 <= H - 1;
    const bool l = g.w_low >= 0, r = g.w_low + 1 <= W - 1;
    m = (unsigned)(t && l) | ((unsigned)(t && r) << 1) | ((unsigned)(b && l) << 2) |
        ((unsigned)(b && r) << 3);
  }
  g.mask = m;
  return g;
}

// ---------------------------------------------------------------------------------------------
// A sampling point prepared for the vector kernels: the four corner rows are CLAMPED into the level
// so they can be gathered without predicates; corners the reference does not read get weight 0
// (forward) / mask bit 0 (backward), which reproduces its zero padding exactly for finite inputs.
//   offf    byte offset of the clamped (h_low, w_low) row inside the (b, m) slab, 16-byte aligned,
//           with flags in the low bits: bit0 = the right-hand corner is a different token,
//           bit1 = the lower corners are a different row, bit2 = the sample passed the bounds test
//   rowstep bytes between rows of this level (W * M * D * sizeof(T))
// ---------------------------------------------------------------------------------------------
struct PointTap {
  unsigned offf, rowstep;
  float w[4];
};

__device__ __forceinline__ unsigned tap_offset(const PointGeom<float>& g, int H, int W, int start,
                                               unsigned MDb) {
  const int hl = max(g.h_low, 0), hh = min(g.h_low + 1, H - 1);
  const int wl = max(g.w_low, 0), wh = min(g.w_low + 1, W - 1);
  return (unsigned)(start + hl * W + wl) * MDb | (unsigned)(wh != wl) | ((unsigned)(hh != hl) << 1) |
         ((unsigned)(g.mask != 0u) << 2);
}

__device__ __forceinline__ PointTap point_tap(float x, float y, float a, int H, int W, int start,
                                              unsigned MDb) {
  const PointGeom<float> g = point_geom<float>(x, y, H, W);
  const float hh = 1.f - g.lh, hw = 1.f - g.lw;
  PointTap t;
  t.w[0] = (g.mask & 1u) ? (hh * hw) * a : 0.f;
  t.w[1] = (g.mask & 2u) ? (hh * g.lw) * a : 0.f;
  t.w[2] = (g.mask & 4u) ? (g.lh * hw) * a : 0.f;
  t.w[3] = (g.mask & 8u) ? (g.lh * g.lw) * a : 0.f;
  t.offf = tap_offset(g, H, W, start, MDb);
  t.rowstep = (unsigned)W * MDb;
  return t;
}

// ---------------------------------------------------------------------------------------------
// 16-byte channel vectors. One lane owns kCpl consecutive channels of a head:
//   float          : 4 channels  (LDG.E.128)
//   __nv_bfloat16  : 8 channels  (LDG.E.128), widened to fp32 in registers
//   __half         : 8 channels  (LDG.E.128), widened to fp32 in registers (opt-in fp16 I/O, set_amp_value_dtype)
// ---------------------------------------------------------------------------------------------
template <typename T>
struct Vec;

template <>
struct Vec<float> {
  static constexpr int kCpl = 4;
  float v[4];
  __device__ __forceinline__ static Vec load(const float* p) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    Vec r;
    r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
    return r;
  }
  __device__ __forceinline__ static Vec zero() {
    Vec r;
    r.v[0] = r.v[1] = r.v[2] = r.v[3] = 0.f;
    return r;
  }
  __device__ __forceinline__ void store(float* p) const {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

template <>
struct Vec<__nv_bfloat16> {
  static constexpr int kCpl = 8;
  float v[8];
  __device__ __forceinline__ static Vec load(const __nv_bfloat16* p) {
    const uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
    Vec r;
    r.v[0] = __uint_as_float(t.x << 16); r.v[1] = __uint_as_float(t.x & 0xffff0000u);
    r.v[2] = __uint_as_float(t.y << 16); r.v[3] = __uint_as_float(t.y & 0xffff0000u);
    r.v[4] = __uint_as_float(t.z << 16); r.v[5] = __uint_as_float(t.z & 0xffff0000u);
    r.v[6] = __uint_as_float(t.w << 16); r.v[7] = __uint_as_float(t.w & 0xffff0000u);
    return r;
  }
  __device__ __forceinline__ static Vec zero() {
    Vec r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.v[i] = 0.f;
    return r;
  }
  __device__ __forceinline__ static unsigned pack2(float lo, float hi) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);  // .x = lo (low 16 bits)
    return *reinterpret_cast<const unsigned*>(&h);
  }
  __device__ __forceinline__ void store(__nv_bfloat16* p) const {
    uint4 t;
    t.x = pack2(v[0], v[1]); t.y = pack2(v[2], v[3]);
    t.z = pack2(v[4], v[5]); t.w = pack2(v[6], v[7]);
    *reinterpret_cast<uint4*>(p) = t;
  }
};

template <>
struct Vec<__half> {
  static constexpr int kCpl = 8;
  float v[8];
  __device__ __forceinline__ static Vec load(const __half* p) {
    const uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
    const unsigned u[4] = {t.x, t.y, t.z, t.w};
    Vec r;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u[i]));
      r.v[2 * i] = f.x; r.v[2 * i + 1] = f.y;
    }
    return r;
  }
  __device__ __forceinline__ static Vec zero() {
    Vec r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.v[i] = 0.f;
    return r;
  }
  __device__ __forceinline__ static unsigned pack2(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);  // .x = lo (low 16 bits)
    return *reinterpret_cast<const unsigned*>(&h);
  }
  __device__ __forceinline__ void store(__half* p) const {
    uint4 t;
    t.x = pack2(v[0], v[1]); t.y = pack2(v[2], v[3]);
    t.z = pack2(v[4], v[5]); t.w = pack2(v[6], v[7]);
    *reinterpret_cast<uint4*>(p) = t;
  }
};

// Reference point of one level as the fused kernels hold it: (x, y) or, for boxes, (x, y, w, h) in one 16-byte load.
template <int RD>
using RefVec = std::conditional_t<RD == 4, float4, float2>;

// Fused module arithmetic (reference: detection/ops/modules/ms_deform_attn.py:108-119), done in registers:
//   attention_weights = softmax(logits over the L*P points of one (b,q,m))
//   sampling_location = reference_point + sampling_offset / (W_l, H_l)                 (RD = 2)
//   sampling_location = ref_xy + sampling_offset / P * ref_wh * 0.5                    (RD = 4, boxes)
// Lane j of a G-lane group holds points j, j+G, ... (R rounds): xy[r] = raw offset, a[r] = raw logit,
// rf[r] = reference point of that point's level. On return xy[r] = location, a[r] = softmax weight.
// The max / sum over the L*P points are warp-shuffle reductions inside the group (every lane of the warp
// must call this). The location arithmetic is the fp32 operations torch performs, in its order and with its
// roundings (a true division by the Python scalar P is torch's multiply by the reciprocal; the _rn intrinsics
// keep nvcc from contracting into an FMA), so the locations — and therefore the corner indices — are
// bit-identical to the unfused path.
template <int G, int R, int PT, typename RefV>
__device__ __forceinline__ void fused_resolve(float2 (&xy)[R], float (&a)[R], const RefV (&rf)[R],
                                              const int* sH, const int* sW, int j, int LP) {
  float m = -INFINITY;
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (r * G + j < LP) m = fmaxf(m, a[r]);
#pragma unroll
  for (int s = G / 2; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, s, G));
  float sum = 0.f;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    a[r] = (r * G + j < LP) ? expf(a[r] - m) : 0.f;
    sum += a[r];
  }
#pragma unroll
  for (int s = G / 2; s > 0; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s, G);
#pragma unroll
  for (int r = 0; r < R; ++r) {
    a[r] = __fdiv_rn(a[r], sum);
    const int pi = r * G + j;
    if (pi < LP) {
      if constexpr (sizeof(RefV) == 16) {
        constexpr float kInvP = 1.0f / PT;
        xy[r].x = __fadd_rn(rf[r].x, __fmul_rn(__fmul_rn(__fmul_rn(xy[r].x, kInvP), rf[r].z), 0.5f));
        xy[r].y = __fadd_rn(rf[r].y, __fmul_rn(__fmul_rn(__fmul_rn(xy[r].y, kInvP), rf[r].w), 0.5f));
      } else {
        const int l = pi / PT;
        xy[r].x = rf[r].x + __fdiv_rn(xy[r].x, (float)sW[l]);
        xy[r].y = rf[r].y + __fdiv_rn(xy[r].y, (float)sH[l]);
      }
    }
  }
}

// Lane vectors by width: 16 bytes per lane (above) or 32 bytes per lane (fp32 only: 8 channels, one
// LDG.E.ENL2.256 / STG.E.ENL2.256, the 256-bit global accesses new on sm_100). Wider lanes halve the lanes per
// (b,q,m), so a warp serves twice as many queries per instruction: the per-point broadcast shuffles and the
// address / weight arithmetic are amortised over 8 queries instead of 4.
template <typename T, int LANE_BYTES>
struct LaneVec;
template <>
struct LaneVec<float, 16> : Vec<float> {
  __device__ __forceinline__ static LaneVec load(const float* p) { LaneVec r; static_cast<Vec<float>&>(r) = Vec<float>::load(p); return r; }
  __device__ __forceinline__ static LaneVec zero() { LaneVec r; static_cast<Vec<float>&>(r) = Vec<float>::zero(); return r; }
};
template <>
struct LaneVec<__nv_bfloat16, 16> : Vec<__nv_bfloat16> {
  __device__ __forceinline__ static LaneVec load(const __nv_bfloat16* p) { LaneVec r; static_cast<Vec<__nv_bfloat16>&>(r) = Vec<__nv_bfloat16>::load(p); return r; }
  __device__ __forceinline__ static LaneVec zero() { LaneVec r; static_cast<Vec<__nv_bfloat16>&>(r) = Vec<__nv_bfloat16>::zero(); return r; }
};
template <>
struct LaneVec<__half, 16> : Vec<__half> {
  __device__ __forceinline__ static LaneVec load(const __half* p) { LaneVec r; static_cast<Vec<__half>&>(r) = Vec<__half>::load(p); return r; }
  __device__ __forceinline__ static LaneVec zero() { LaneVec r; static_cast<Vec<__half>&>(r) = Vec<__half>::zero(); return r; }
};
template <>
struct LaneVec<float, 32> {
  static constexpr int kCpl = 8;
  float v[8];
  __device__ __forceinline__ static LaneVec load(const float* p) {
    LaneVec r;
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                 : "l"(p));
    return r;
  }
  __device__ __forceinline__ static LaneVec zero() {
    LaneVec r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.v[i] = 0.f;
    return r;
  }
  __device__ __forceinline__ void store(float* p) const {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
  }
};

// 64-bit pointer + 32-bit offset in ONE instruction (IMAD.WIDE.U32) instead of IADD3 + IADD3.X: the
// gather kernels are issue-bound, and every corner needs its own address.
__device__ __forceinline__ const char* ptr_add(const char* base, unsigned off) {
  unsigned long long r;
  asm("mad.wide.u32 %0, %1, 1, %2;" : "=l"(r) : "r"(off), "l"(reinterpret_cast<unsigned long long>(base)));
  return reinterpret_cast<const char*>(r);
}
// base + a * b (a, b 32-bit unsigned), one IMAD.WIDE.U32
__device__ __forceinline__ const char* ptr_madd(const char* base, unsigned a, unsigned b) {
  unsigned long long r;
  asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(a), "r"(b), "l"(reinterpret_cast<unsigned long long>(base)));
  return reinterpret_cast<const char*>(r);
}

// acc[0..3] += a1*v1[0..3] + a2*v2[0..3] + a3*v3[0..3] + a4*v4[0..3], executed only when `on` != 0, as 16
// PREDICATED FFMAs (no branch, no select): an out-of-range sample must contribute exactly nothing even if
// the clamped rows it aliased hold Inf/NaN. Accumulation order per channel is corner 1,2,3,4.
__device__ __forceinline__ void fma4x4_if(unsigned on, float* acc, float a1, float a2, float a3, float a4,
                                          const float* v1, const float* v2, const float* v3, const float* v4) {
  asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %24, 0;\n\t"
      "@p fma.rn.f32 %0, %4, %8, %0;\n\t@p fma.rn.f32 %1, %4, %9, %1;\n\t"
      "@p fma.rn.f32 %2, %4, %10, %2;\n\t@p fma.rn.f32 %3, %4, %11, %3;\n\t"
      "@p fma.rn.f32 %0, %5, %12, %0;\n\t@p fma.rn.f32 %1, %5, %13, %1;\n\t"
      "@p fma.rn.f32 %2, %5, %14, %2;\n\t@p fma.rn.f32 %3, %5, %15, %3;\n\t"
      "@p fma.rn.f32 %0, %6, %16, %0;\n\t@p fma.rn.f32 %1, %6, %17, %1;\n\t"
      "@p fma.rn.f32 %2, %6, %18, %2;\n\t@p fma.rn.f32 %3, %6, %19, %3;\n\t"
      "@p fma.rn.f32 %0, %7, %20, %0;\n\t@p fma.rn.f32 %1, %7, %21, %1;\n\t"
      "@p fma.rn.f32 %2, %7, %22, %2;\n\t@p fma.rn.f32 %3, %7, %23, %3;\n\t}"
      : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
      : "f"(a1), "f"(a2), "f"(a3), "f"(a4),
        "f"(v1[0]), "f"(v1[1]), "f"(v1[2]), "f"(v1[3]), "f"(v2[0]), "f"(v2[1]), "f"(v2[2]), "f"(v2[3]),
        "f"(v3[0]), "f"(v3[1]), "f"(v3[2]), "f"(v3[3]), "f"(v4[0]), "f"(v4[1]), "f"(v4[2]), "f"(v4[3]),
        "r"(on));
}

// Vector reduction into global memory: one REDG.E.ADD.F32x4 per 16 bytes (sm_90+ PTX
// `red.global.add.v4.f32`) instead of the reference's one scalar atomicAdd per channel per corner
// (ms_deform_im2col_cuda.cuh:121,130,139,148).
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c),
               "f"(d)
               : "memory");
}

// scalar load / convert helpers for the generic (any-D) kernels
__device__ __forceinline__ float ld_scalar(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_scalar(const __nv_bfloat16* p) {
  return __bfloat162float(__ldg(p));
}
__device__ __forceinline__ double ld_scalar(const double* p) { return __ldg(p); }

__device__ __forceinline__ void st_scalar(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_scalar(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ float ld_scalar(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ void st_scalar(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ void st_scalar(double* p, double v) { *p = v; }

// Block -> (batch, query chunk, head) decomposition shared by forward and backward.
// Heads vary fastest so concurrently running CTAs cover the same spatial neighbourhood
// (their sampling_loc / attn_weight sectors and value rows are shared in L2).
struct BlockCoord {
  int b, m, q_begin, q_end;
};
// (Walking the batch back-to-front in the backward, so that the tail of the grad_value memset is still in L2
// when its atomics arrive, was measured: no change — 240.6 vs 240.6 us on the 132 MB Injector tensor.)
__device__ __forceinline__ BlockCoord block_coord(const Params& p) {
  BlockCoord c;
  const int bid = blockIdx.x;
  c.m = bid % p.M;
  const int t = bid / p.M;
  const int chunk = t % p.nchunk;
  c.b = t / p.nchunk;
  c.q_begin = chunk * p.qc;
  c.q_end = min(p.Lq, c.q_begin + p.qc);
  return c;
}

}  // namespace msda
