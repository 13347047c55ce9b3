// msda_fwd.cu — forward of multi-scale deformable attention for sm_100a.
//
// Replaces ms_deformable_im2col_gpu_kernel (reference: detection/ops/src/cuda/
// ms_deform_im2col_cuda.cuh:237-299) and its launcher (:923-954). Not a port: the reference runs
// one thread per output scalar and recomputes every coordinate D times; here
//   * a CTA owns (batch b, head m, a chunk of consecutive queries) so that the value rows its
//     warps gather stay hot in L1 (consecutive queries are spatial neighbours in the adapter),
//   * a group of G lanes owns one (b,q,m): each lane keeps 16 bytes of channels (4 fp32 / 8 bf16),
//     so a warp serves 32/G queries at once and every gather is an LDG.E.128 that covers whole
//     128-byte lines (one L1 wavefront per corner row),
//   * the geometry of a point is computed ONCE, by one lane of the group: corner rows are clamped
//     into the level (so the four gathers need no predicate and no zero-fill), the bilinear weights
//     are pre-multiplied with the attention weight and zeroed for corners the reference skips, and
//     the lot (packed offset+flags, 4 weights) is handed to the group through a 32-byte record in the
//     warp's shared-memory scratch: one LDS.128 + one LDS.32 per point instead of 5 warp shuffles on
//     the same LSU pipe the gathers saturate (round 1: 41 % of the pipe's wavefronts were shuffles),
//   * out is written exactly once (no at::zeros memset as in ms_deform_attn_cuda.cu:54).
#include "msda_common.cuh"

namespace msda {

// ---------------------------------------------------------------------------------------------
// Vector kernel. T = float | __nv_bfloat16, G = lanes per (b,q,m) (D = G * Vec<T>::kCpl),
// LT/PT = compile-time levels / points (0,0 = runtime), MINB = min resident CTAs per SM.
// ---------------------------------------------------------------------------------------------
// FUSED: `loc` / `aw` hold raw offsets / logits; locations and the softmax are formed in registers (static L,P only).
// RD (fused only): reference-point width, 2 = points (x, y), 4 = boxes (x, y, w, h).
template <typename T, int G, int LT, int PT, int MINB, int LB = 16, bool FUSED = false, int RD = 2>
__global__ void __launch_bounds__(kThreads, MINB) msda_fwd_vec_kernel(const Params p) {
  static_assert(!FUSED || LT > 0, "the fused entry needs compile-time L, P");
  static_assert(RD == 2 || (FUSED && RD == 4), "box references are a fused-entry input");
  using RefV = RefVec<RD>;
  using V = LaneVec<T, LB>;  // LB = bytes per lane: 16 (LDG.128) or 32 (LDG.256, fp32 only)
  constexpr int kCpl = V::kCpl;
  constexpr int kGpw = 32 / G;  // (b,q,m) groups per warp
  constexpr bool kStatic = (LT > 0);

  const int L = kStatic ? LT : p.L;
  const int P = kStatic ? PT : p.P;
  const int LP = L * P;
  const int MD = p.M * p.D;
  const unsigned MDb = (unsigned)MD * (unsigned)sizeof(T);  // bytes between neighbouring tokens

  __shared__ int sH[kMaxLevels], sW[kMaxLevels], sStart[kMaxLevels];
  // per-warp tap scratch: one row per (b,q,m) group of the warp, G records of 32 bytes (4 weights | offset+flags, row
  // step) + 16 bytes of padding, so that the records the 32/G groups read together sit in different bank groups
  constexpr int kTapRow = 2 * G + 1;  // uint4 per group row
  __shared__ uint4 s_tap[kWarps * kGpw * kTapRow];
  if (threadIdx.x < L) {
    sH[threadIdx.x] = (int)p.shapes[2 * threadIdx.x];
    sW[threadIdx.x] = (int)p.shapes[2 * threadIdx.x + 1];
    sStart[threadIdx.x] = (int)p.lsi[threadIdx.x];
  }
  __syncthreads();

  unsigned rsl[kStatic ? LT : 1];  // bytes between rows, per level (registers; static indexing only)
#pragma unroll
  for (int l = 0; l < (kStatic ? LT : 1); ++l) rsl[l] = (unsigned)sW[l] * MDb;

  const BlockCoord bc = block_coord(p);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = lane / G, j = lane % G;
  const unsigned tap_row = (unsigned)__cvta_generic_to_shared(s_tap) + (unsigned)((warp * kGpw + grp) * kTapRow) * 16u;
  const unsigned tap_mine = tap_row + (unsigned)j * 32u;

  // CTA-uniform slab base (batch b, head m) + this lane's 16 bytes inside a D-row
  const char* __restrict__ vb = reinterpret_cast<const char*>(p.value) +
                                ((size_t)bc.b * p.S * MD + (size_t)bc.m * p.D) * sizeof(T) + j * LB;
  const float* __restrict__ loc = reinterpret_cast<const float*>(p.loc);
  const float* __restrict__ aw = reinterpret_cast<const float*>(p.aw);
  T* __restrict__ out = reinterpret_cast<T*>(p.out);

  // Software pipeline over the query loop: sampling_loc / attn_weight stream from HBM once, so their load
  // latency (~800 cycles) would sit at the head of every iteration's dependency chain. The static
  // variants fetch the NEXT iteration's locations and weights before working on the current one.
  constexpr int kRounds = kStatic ? (LT * PT + G - 1) / G : 1;
  float2 nxy[kRounds];
  RefV nrf[kRounds];
  float na[kRounds];
  auto fetch = [&](int qw_, float2 (&xy_)[kRounds], float (&a_)[kRounds], RefV (&rf_)[kRounds]) {
    const int q_ = qw_ + grp;
    const bool act_ = q_ < bc.q_end;
    const int qq_ = act_ ? q_ : bc.q_begin;
    const size_t pair_ = ((size_t)bc.b * p.Lq + qq_) * p.M + bc.m;
#pragma unroll
    for (int r = 0; r < kRounds; ++r) {
      const int pi_ = r * G + j;
      xy_[r] = make_float2(0.f, 0.f);
      rf_[r] = RefV{};
      a_[r] = 0.f;
      if (pi_ < LP && act_) {
        if (FUSED) {  // raw offsets / logits may be two column blocks of ONE merged GEMM output: explicit row strides
          const size_t row_ = (size_t)bc.b * p.Lq + qq_;
          xy_[r] = __ldg(reinterpret_cast<const float2*>(loc + row_ * p.off_rowstride + (size_t)bc.m * LP * 2) + pi_);
          a_[r] = __ldg(aw + row_ * p.logit_rowstride + (size_t)bc.m * LP + pi_);
        } else {
          xy_[r] = __ldg(reinterpret_cast<const float2*>(loc + pair_ * LP * 2) + pi_);
          a_[r] = __ldg(aw + pair_ * LP + pi_);
        }
        if (FUSED)
          rf_[r] = __ldg(reinterpret_cast<const RefV*>(p.ref + (size_t)bc.b * p.ref_bstride + (size_t)qq_ * p.ref_qstride +
                                                       (pi_ / (FUSED ? PT : 1)) * p.ref_lstride));
      }
    }
  };
  if (kStatic) fetch(bc.q_begin + warp * kGpw, nxy, na, nrf);

  for (int qw = bc.q_begin + warp * kGpw; qw < bc.q_end; qw += kWarps * kGpw) {
    const int q = qw + grp;
    const bool active = q < bc.q_end;
    const size_t pair = ((size_t)bc.b * p.Lq + (active ? q : bc.q_begin)) * p.M + bc.m;
    const float* __restrict__ loc_pair = loc + pair * LP * 2;
    const float* __restrict__ aw_pair = aw + pair * LP;

    float2 cxy[kRounds];
    RefV crf[kRounds];
    float ca[kRounds];
    if (kStatic) {
#pragma unroll
      for (int r = 0; r < kRounds; ++r) { cxy[r] = nxy[r]; ca[r] = na[r]; crf[r] = nrf[r]; }
      if (qw + kWarps * kGpw < bc.q_end) fetch(qw + kWarps * kGpw, nxy, na, nrf);
      if constexpr (FUSED) fused_resolve<G, kRounds, (FUSED ? PT : 1)>(cxy, ca, crf, sH, sW, j, LP);
    }

    V acc = V::zero();

#pragma unroll
    for (int r0 = 0; r0 < (kStatic ? LT * PT : LP); r0 += G) {
      // ---- producer: lane j prepares point r0 + j --------------------------------------------
      const int pi = r0 + j;
      PointTap tap;
      tap.offf = 0u; tap.rowstep = 0u;
      tap.w[0] = tap.w[1] = tap.w[2] = tap.w[3] = 0.f;
      if (pi < LP && active) {
        const int l = pi / P;
        float2 xy;
        float a;
        if (kStatic) {
          xy = cxy[r0 / G];
          a = ca[r0 / G];
        } else {
          xy = __ldg(reinterpret_cast<const float2*>(loc_pair) + pi);
          a = __ldg(aw_pair + pi);
        }
        tap = point_tap(xy.x, xy.y, a, sH[l], sW[l], sStart[l], MDb);
      }
      // ---- hand-over: every lane publishes the point it prepared ------------------------------------
      __syncwarp();  // the previous round's readers are done with the records
      asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(tap_mine), "f"(tap.w[0]), "f"(tap.w[1]), "f"(tap.w[2]), "f"(tap.w[3]) : "memory");
      asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(tap_mine + 16u), "r"(tap.offf), "r"(tap.rowstep) : "memory");
      __syncwarp();
      // ---- consumers: every lane of the group gathers its 16 bytes for each prepared point ----
#pragma unroll
      for (int jj = 0; jj < G; ++jj) {
        if (r0 + jj < LP) {  // uniform
          float a1, a2, a3, a4;
          unsigned of, rs;
          asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a1), "=f"(a2), "=f"(a3), "=f"(a4) : "r"(tap_row + jj * 32u));
          if (kStatic) {
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(of) : "r"(tap_row + jj * 32u + 16u));
            rs = rsl[(r0 + jj) / (kStatic ? PT : 1)];  // level is a compile-time constant here
          } else {
            asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(of), "=r"(rs) : "r"(tap_row + jj * 32u + 16u));
          }
          // four corner addresses in 4 IMAD.WIDE (64-bit base + 32-bit offset / flag * step)
          const char* p1 = ptr_add(vb, of & ~15u);
          const char* p2 = ptr_madd(p1, of & 1u, MDb);
          const char* p3 = ptr_madd(p1, (of >> 1) & 1u, rs);
          const char* p4 = ptr_madd(p3, of & 1u, MDb);
          const V v1 = V::load(reinterpret_cast<const T*>(p1));
          const V v2 = V::load(reinterpret_cast<const T*>(p2));
          const V v3 = V::load(reinterpret_cast<const T*>(p3));
          const V v4 = V::load(reinterpret_cast<const T*>(p4));
          // the reference skips out-of-range samples entirely (:288): predicated FMAs, no branch
#pragma unroll
          for (int c0 = 0; c0 < kCpl; c0 += 4)
            fma4x4_if(of & 4u, &acc.v[c0], a1, a2, a3, a4, &v1.v[c0], &v2.v[c0], &v3.v[c0], &v4.v[c0]);
        }
      }
    }
    if (active) acc.store(out + pair * p.D + j * kCpl);
  }
}

// ---------------------------------------------------------------------------------------------
// Generic kernel: any D, any dtype (f32 / bf16 / f64), any L,P. One warp per (b,q,m); lanes stride
// over channels. Completeness path for the channel counts the reference's own test sweeps
// (ops/test.py:108: D in {30, 71, 1025, 2048, 3096}); the adapter shapes never take it.
// ---------------------------------------------------------------------------------------------
template <typename T, typename F>
__global__ void __launch_bounds__(kThreads) msda_fwd_generic_kernel(const Params p) {
  const int L = p.L, P = p.P, LP = L * P, MD = p.M * p.D;
  const BlockCoord bc = block_coord(p);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const T* __restrict__ vb =
      reinterpret_cast<const T*>(p.value) + (size_t)bc.b * p.S * MD + bc.m * p.D;
  const F* __restrict__ loc = reinterpret_cast<const F*>(p.loc);
  const F* __restrict__ aw = reinterpret_cast<const F*>(p.aw);
  T* __restrict__ out = reinterpret_cast<T*>(p.out);

  for (int q = bc.q_begin + warp; q < bc.q_end; q += kWarps) {
    const size_t pair = ((size_t)bc.b * p.Lq + q) * p.M + bc.m;
    for (int c = lane; c < p.D; c += 32) {
      F acc = 0;
      for (int l = 0; l < L; ++l) {
        const int H = (int)p.shapes[2 * l], W = (int)p.shapes[2 * l + 1];
        const int start = (int)p.lsi[l];
        for (int k = 0; k < P; ++k) {
          const size_t pi = pair * LP + l * P + k;
          const F x = loc[2 * pi], y = loc[2 * pi + 1], a = aw[pi];
          const PointGeom<F> g = point_geom<F>(x, y, H, W);
          if (g.mask == 0u) continue;
          const F hh = 1 - g.lh, hw = 1 - g.lw;
          const T* p1 = vb + (size_t)(start + g.h_low * W + g.w_low) * MD + c;
          const F v1 = (g.mask & 1u) ? (F)ld_scalar(p1) : (F)0;
          const F v2 = (g.mask & 2u) ? (F)ld_scalar(p1 + MD) : (F)0;
          const F v3 = (g.mask & 4u) ? (F)ld_scalar(p1 + (size_t)W * MD) : (F)0;
          const F v4 = (g.mask & 8u) ? (F)ld_scalar(p1 + (size_t)W * MD + MD) : (F)0;
          const F val = (hh * hw) * v1 + (hh * g.lw) * v2 + (g.lh * hw) * v3 + (g.lh * g.lw) * v4;
          acc += val * a;
        }
      }
      st_scalar(out + pair * p.D + c, acc);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Launchers
// ---------------------------------------------------------------------------------------------
template <typename T, int G, int MINB>
static cudaError_t launch_vec_gm(const Params& p, dim3 grid, cudaStream_t s) {
  if (p.L == 3 && p.P == 4) {
    msda_fwd_vec_kernel<T, G, 3, 4, MINB><<<grid, kThreads, 0, s>>>(p);
  } else if (p.L == 1 && p.P == 4) {
    msda_fwd_vec_kernel<T, G, 1, 4, MINB><<<grid, kThreads, 0, s>>>(p);
  } else {
    msda_fwd_vec_kernel<T, G, 0, 0, MINB><<<grid, kThreads, 0, s>>>(p);
  }
  return cudaGetLastError();
}

template <typename T, int G>
static cudaError_t launch_vec_g(const Params& p, int minb, dim3 grid, cudaStream_t s) {
  switch (minb) {
    case 3: return launch_vec_gm<T, G, 3>(p, grid, s);
    case 6: return launch_vec_gm<T, G, 6>(p, grid, s);
    // measured (tools/minctas_sweep.py, profiles/r2_minctas_sweep.jsonl): fp32 is fastest compiled for 4 resident CTAs
    // (64 registers), the 16-bit kernels - which also hold the unpacked rows - for 3 (80): Extractor forward bf16 B
    // 101 -> 96 us, S 88 -> 85, L bs 1 35.6 -> 33.6; 6 CTAs (40 registers) lose 20 % at fp32
    default: return launch_vec_gm<T, G, (sizeof(T) == 2 ? 3 : 4)>(p, grid, s);
  }
}

// ---------------------------------------------------------------------------------------------
// The file is compiled once per value dtype (build.py: -DMSDA_TU=0 f32 + f64 + dispatch, 1 bf16, 2 f16) so that the
// three sets of instantiations build in parallel; each part exports its entry points under a dtype suffix.
// ---------------------------------------------------------------------------------------------
#ifndef MSDA_TU
#define MSDA_TU 0
#endif

// fused entry (raw offsets + logits + reference points): static (L,P) in {(3,4),(1,4),(4,4)} only, points or boxes
template <typename T, int G, int RD>
static cudaError_t launch_fused_gr(const Params& p, dim3 grid, cudaStream_t s) {
  if (p.L == 3 && p.P == 4) msda_fwd_vec_kernel<T, G, 3, 4, 4, 16, true, RD><<<grid, kThreads, 0, s>>>(p);
  else if (p.L == 1 && p.P == 4) msda_fwd_vec_kernel<T, G, 1, 4, 4, 16, true, RD><<<grid, kThreads, 0, s>>>(p);
  else if (p.L == 4 && p.P == 4) msda_fwd_vec_kernel<T, G, 4, 4, 4, 16, true, RD><<<grid, kThreads, 0, s>>>(p);
  else return cudaErrorNotSupported;
  return cudaGetLastError();
}
template <typename T, int G>
static cudaError_t launch_fused_g(const Params& p, dim3 grid, cudaStream_t s) {
  return p.ref_dim == 4 ? launch_fused_gr<T, G, 4>(p, grid, s) : launch_fused_gr<T, G, 2>(p, grid, s);
}

template <typename T>
static cudaError_t launch_vec(const Params& p, int G, int minb, dim3 grid, cudaStream_t s) {
  switch (G) {
    case 2: return launch_vec_gm<T, 2, 4>(p, grid, s);
    case 4: return launch_vec_g<T, 4>(p, minb, grid, s);
    case 8: return launch_vec_g<T, 8>(p, minb, grid, s);
    case 16: return launch_vec_g<T, 16>(p, minb, grid, s);
    case 32: return launch_vec_gm<T, 32, 4>(p, grid, s);
    default: return cudaErrorInvalidValue;
  }
}

// 16-bit value types: 8 channels per lane -> fused kernels at G = 4 (D = 32) and 8 (D = 64)
template <typename T>
static cudaError_t launch_fused_lowp(const Params& p, int G, dim3 grid, cudaStream_t s) {
  if (G == 4) return launch_fused_g<T, 4>(p, grid, s);
  if (G == 8) return launch_fused_g<T, 8>(p, grid, s);
  return cudaErrorNotSupported;
}

cudaError_t fwd_vec_bf16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s);
cudaError_t fwd_fused_bf16(const Params& p, int G, dim3 grid, cudaStream_t s);
cudaError_t fwd_generic_bf16(const Params& p, dim3 grid, cudaStream_t s);
cudaError_t fwd_vec_f16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s);
cudaError_t fwd_fused_f16(const Params& p, int G, dim3 grid, cudaStream_t s);
cudaError_t fwd_generic_f16(const Params& p, dim3 grid, cudaStream_t s);

#if MSDA_TU == 1
cudaError_t fwd_vec_bf16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s) { return launch_vec<__nv_bfloat16>(p, G, minb, grid, s); }
cudaError_t fwd_fused_bf16(const Params& p, int G, dim3 grid, cudaStream_t s) { return launch_fused_lowp<__nv_bfloat16>(p, G, grid, s); }
cudaError_t fwd_generic_bf16(const Params& p, dim3 grid, cudaStream_t s) {
  msda_fwd_generic_kernel<__nv_bfloat16, float><<<grid, kThreads, 0, s>>>(p);
  return cudaGetLastError();
}
#elif MSDA_TU == 2
cudaError_t fwd_vec_f16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s) { return launch_vec<__half>(p, G, minb, grid, s); }
cudaError_t fwd_fused_f16(const Params& p, int G, dim3 grid, cudaStream_t s) { return launch_fused_lowp<__half>(p, G, grid, s); }
cudaError_t fwd_generic_f16(const Params& p, dim3 grid, cudaStream_t s) {
  msda_fwd_generic_kernel<__half, float><<<grid, kThreads, 0, s>>>(p);
  return cudaGetLastError();
}
#else
// 32-byte lanes (fp32): G = D / 8
template <int G>
static cudaError_t launch_wide_g(const Params& p, int minb, dim3 grid, cudaStream_t s) {
  if (p.L == 3 && p.P == 4) {
    if (minb == 3) msda_fwd_vec_kernel<float, G, 3, 4, 3, 32><<<grid, kThreads, 0, s>>>(p);
    else msda_fwd_vec_kernel<float, G, 3, 4, 4, 32><<<grid, kThreads, 0, s>>>(p);
  } else if (p.L == 1 && p.P == 4) {
    if (minb == 3) msda_fwd_vec_kernel<float, G, 1, 4, 3, 32><<<grid, kThreads, 0, s>>>(p);
    else msda_fwd_vec_kernel<float, G, 1, 4, 4, 32><<<grid, kThreads, 0, s>>>(p);
  } else {
    msda_fwd_vec_kernel<float, G, 0, 0, 4, 32><<<grid, kThreads, 0, s>>>(p);
  }
  return cudaGetLastError();
}

cudaError_t launch_forward_wide(const Params& p, int G, int minb, cudaStream_t s) {
  const dim3 grid((unsigned)((size_t)p.N * p.nchunk * p.M));
  switch (G) {
    case 2: return launch_wide_g<2>(p, minb, grid, s);
    case 4: return launch_wide_g<4>(p, minb, grid, s);
    case 8: return launch_wide_g<8>(p, minb, grid, s);
    default: return cudaErrorNotSupported;
  }
}

cudaError_t launch_forward_fused(const Params& p, int dtype, int G, cudaStream_t s) {
  const dim3 grid((unsigned)((size_t)p.N * p.nchunk * p.M));
  if (dtype == MSDA_F32) {
    if (G == 8) return launch_fused_g<float, 8>(p, grid, s);
    if (G == 16) return launch_fused_g<float, 16>(p, grid, s);
  } else if (dtype == MSDA_F16) {
    return fwd_fused_f16(p, G, grid, s);
  } else if (dtype == MSDA_BF16) {
    return fwd_fused_bf16(p, G, grid, s);
  }
  return cudaErrorNotSupported;
}

// Returns true when the vector kernels support (dtype, D): D*sizeof(T) is a multiple of 16 bytes and
// D / (16/sizeof(T)) is a power of two in [2, 32].
bool vec_supported(int dtype, int D, int* G_out) {
  int cpl = dtype == MSDA_F32 ? 4 : (dtype == MSDA_BF16 || dtype == MSDA_F16) ? 8 : 0;
  if (cpl == 0 || D % cpl != 0) return false;
  const int G = D / cpl;
  if (G < 2 || G > 32 || (G & (G - 1)) != 0) return false;
  *G_out = G;
  return true;
}

cudaError_t launch_forward(const Params& p, int dtype, bool vec_ok, int G, int minb, cudaStream_t s) {
  const dim3 grid((unsigned)((size_t)p.N * p.nchunk * p.M));
  if (vec_ok) {
    if (dtype == MSDA_F32) return launch_vec<float>(p, G, minb, grid, s);
    if (dtype == MSDA_F16) return fwd_vec_f16(p, G, minb, grid, s);
    return fwd_vec_bf16(p, G, minb, grid, s);
  }
  switch (dtype) {
    case MSDA_F32: msda_fwd_generic_kernel<float, float><<<grid, kThreads, 0, s>>>(p); break;
    case MSDA_BF16: return fwd_generic_bf16(p, grid, s);
    case MSDA_F16: return fwd_generic_f16(p, grid, s);
    case MSDA_F64: msda_fwd_generic_kernel<double, double><<<grid, kThreads, 0, s>>>(p); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}
#endif  // MSDA_TU

}  // namespace msda
