// msda_bwd.cu — backward of multi-scale deformable attention for sm_100a.
//
// Replaces the reference's col2im kernels (detection/ops/src/cuda/ms_deform_im2col_cuda.cuh:
// 301-403 `…blocksize_aware_reduce_v1` used at D=32, :406-510 `…reduce_v2` used at D=64, and the
// dynamic/global variants :513-920) plus the launcher switch (:956-1327). Not a port:
//   * the reference launches one D-thread block per (b,q,m), stages 3*D partials in shared memory
//     per point and reduces them serially (v1) or with a barrier tree (v2); here a group of G lanes
//     owns a (b,q,m) and each lane keeps 4/8 channels. Because everything is linear in the corner
//     values, a lane only accumulates u_k = sum_c grad_out[c] * v_k[c] for the four corners (4 FMAs
//     per channel) and turns (u_1..u_4) into its share of d/d(attn), d/dx, d/dy once per point;
//     the G shares of all G points of a round are then summed with ONE transposed shuffle
//     reduction (3G values -> 3 per lane in ~3G shuffles, instead of 3*log2(G) per point) — no
//     shared memory, no __syncthreads in the point loop;
//   * corner rows are clamped into the level, so the value gathers need no predicates;
//   * grad_value is scattered with one 16-byte vector reduction (REDG.E.ADD.F32x4) per lane per
//     corner instead of one scalar atomicAdd per channel per corner (:121,130,139,148);
//   * grad_sampling_loc / grad_attn_weight are written exactly once, so only grad_value is
//     zero-filled (the reference memsets all three, ms_deform_attn_cuda.cu:121-123).
// bf16 I/O accumulates grad_value in an fp32 scratch and converts once at the end.
#include "msda_common.cuh"

namespace msda {

// Backward lane layout: ALWAYS 4 channels per lane, for fp32 and bf16 alike (bf16 rows are read with
// 8-byte loads). The scatter then issues exactly one REDG.E.ADD.F32x4 per lane per corner and the G
// lanes of a group cover whole 32-byte sectors of the fp32 accumulator row in one instruction. (With
// 8 bf16 channels per lane the two halves of a lane's 32 bytes went out in two instructions, each
// touching every sector half-filled: twice the L2 atomic sector visits — measured 1.6x slower.)
template <typename T>
struct VecB;
template <>
struct VecB<float> : Vec<float> {
  static constexpr int kLaneBytes = 16;
  __device__ __forceinline__ static VecB load(const float* p) { VecB r; static_cast<Vec<float>&>(r) = Vec<float>::load(p); return r; }
  __device__ __forceinline__ static VecB zero() { VecB r; static_cast<Vec<float>&>(r) = Vec<float>::zero(); return r; }
};
template <>
struct VecB<__nv_bfloat16> {
  static constexpr int kCpl = 4;
  static constexpr int kLaneBytes = 8;
  float v[4];
  __device__ __forceinline__ static VecB load(const __nv_bfloat16* p) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    VecB r;
    r.v[0] = __uint_as_float(t.x << 16); r.v[1] = __uint_as_float(t.x & 0xffff0000u);
    r.v[2] = __uint_as_float(t.y << 16); r.v[3] = __uint_as_float(t.y & 0xffff0000u);
    return r;
  }
  __device__ __forceinline__ static VecB zero() {
    VecB r;
    r.v[0] = r.v[1] = r.v[2] = r.v[3] = 0.f;
    return r;
  }
};

template <>
struct VecB<__half> {
  static constexpr int kCpl = 4;
  static constexpr int kLaneBytes = 8;
  float v[4];
  __device__ __forceinline__ static VecB load(const __half* p) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
    VecB r;
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = b.x; r.v[3] = b.y;
    return r;
  }
  __device__ __forceinline__ static VecB zero() {
    VecB r;
    r.v[0] = r.v[1] = r.v[2] = r.v[3] = 0.f;
    return r;
  }
};

// OPT-IN scatter for 16-bit I/O (tuning key "bwd_packed16" = 2): 4 channels go out as ONE packed reduction straight into the
// bf16 / fp16 grad_value (REDG.E.ADD.BF16x4 / F16x4, 8 bytes per lane, 64-byte rows for D = 32) instead of an fp32 vector
// reduction into a scratch that is zero-filled before and converted after. Half the atomic payload (the L2 served 1.67x
// the rows per ns in the round-1 microbenchmark), no 4-byte-per-element memset, no convert kernel - but every CONTRIBUTION is
// rounded to 16 bits and the running sum is kept in 16 bits, instead of one rounding of an fp32 sum: ~sqrt(n) * 2^-9
// relative error for n contributions per element (n ~ 9 Injector, ~ 84 Extractor), outside the 1e-2 bf16 tolerance for
// long sums. Not the default for that reason; tests/test_op_gpu.py::test_packed16_backward states its tolerance.
template <typename T>
__device__ __forceinline__ void red_add_16x4(char* p, float a, float b, float c, float d);
template <>
__device__ __forceinline__ void red_add_16x4<__nv_bfloat16>(char* p, float a, float b, float c, float d) {
  asm volatile("red.global.v2.bf16x2.add.noftz [%0], {%1, %2};" ::"l"(p), "r"(Vec<__nv_bfloat16>::pack2(a, b)),
               "r"(Vec<__nv_bfloat16>::pack2(c, d)) : "memory");
}
template <>
__device__ __forceinline__ void red_add_16x4<__half>(char* p, float a, float b, float c, float d) {
  asm volatile("red.global.v2.f16x2.add.noftz [%0], {%1, %2};" ::"l"(p), "r"(Vec<__half>::pack2(a, b)), "r"(Vec<__half>::pack2(c, d)) : "memory");
}
template <>
__device__ __forceinline__ void red_add_16x4<float>(char*, float, float, float, float) {}

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int s = G / 2; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s, G);
  return v;
}

// Transposed reduction over a group of G lanes: every lane holds NV = 3*G partials laid out
// [point][component]; afterwards lane j holds the three totals of point j in v[0..2].
// Each step halves the live values: a lane keeps the half that belongs to its side of the split and
// receives the partner's partials for that half.
template <int G, int NV>
__device__ __forceinline__ void group_transpose_sum(float (&v)[NV], int j) {
  static_assert(NV == 3 * G, "layout is [G points][3 components]");
  int n = NV;
#pragma unroll
  for (int s = G / 2; s > 0; s >>= 1) {
    const bool upper = (j & s) != 0;
    const int half = n / 2;
#pragma unroll
    for (int i = 0; i < NV / 2; ++i) {
      if (i < half) {
        const float send = upper ? v[i] : v[i + half];
        const float keep = upper ? v[i + half] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s, G);
      }
    }
    n = half;
  }
}

// ---------------------------------------------------------------------------------------------
// Vector kernel (same work decomposition as the forward).
// ---------------------------------------------------------------------------------------------
// FUSED: `loc` / `aw` hold raw offsets / logits (see fused_resolve); grad_loc / grad_aw then receive the gradients
// w.r.t. the raw offsets / logits (softmax backward and the 1/(W,H) scaling folded in).
// PACK (16-bit T only): grad_value is T storage and the scatter uses packed 16-bit reductions (see red_add_16x4).
// RD (fused only): reference-point width, 2 = points (x, y), 4 = boxes (x, y, w, h).
// RGRAD (fused only): also write the reference-point gradient of every (b,q,m) to p.ref_partial, reduced inside the group
// over the P points of a level (and over the levels when the reference points broadcast over them); no atomics, so the
// result is bitwise reproducible. msda_ref_grad_reduce_kernel sums the partials over the heads (and the batch).
template <typename T, int G, int LT, int PT, int MINB, bool FUSED = false, bool PACK = false, int RD = 2, bool RGRAD = false>
__global__ void __launch_bounds__(kThreads, MINB) msda_bwd_vec_kernel(const Params p) {
  static_assert(!FUSED || LT > 0, "the fused entry needs compile-time L, P");
  static_assert(!PACK || sizeof(T) == 2, "packed reductions are for the 16-bit value types");
  static_assert((RD == 2 && !RGRAD) || (FUSED && (RD == 2 || RD == 4) && G % (PT > 0 ? PT : 1) == 0),
                "box references and reference-point gradients are fused-entry features; a level's points share a round");
  using RefV = RefVec<RD>;
  constexpr float kInvP = 1.0f / (PT > 0 ? PT : 1);
  using V = VecB<T>;
  constexpr int kCpl = V::kCpl;
  constexpr int kGpw = 32 / G;
  constexpr bool kStatic = (LT > 0);
  constexpr bool kTranspose = (G <= 8);  // 3*G partial registers per lane

  const int L = kStatic ? LT : p.L;
  const int P = kStatic ? PT : p.P;
  const int LP = L * P;
  const int MD = p.M * p.D;
  const unsigned MDb = (unsigned)MD * (unsigned)sizeof(T);  // bytes between neighbouring tokens (value)
  const unsigned MDf = PACK ? MDb : (unsigned)MD * 4u;       // same in the grad_value accumulator (fp32, or T when PACK)

  __shared__ int sH[kMaxLevels], sW[kMaxLevels], sStart[kMaxLevels];
  if (threadIdx.x < L) {
    sH[threadIdx.x] = (int)p.shapes[2 * threadIdx.x];
    sW[threadIdx.x] = (int)p.shapes[2 * threadIdx.x + 1];
    sStart[threadIdx.x] = (int)p.lsi[threadIdx.x];
  }
  __syncthreads();

  unsigned rsl[kStatic ? LT : 1];  // token rows: bytes between rows per level, in units of MDb
#pragma unroll
  for (int l = 0; l < (kStatic ? LT : 1); ++l) rsl[l] = (unsigned)sW[l];

  const BlockCoord bc = block_coord(p);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = lane / G, j = lane % G;

  const size_t slab = (size_t)bc.b * p.S * MD + (size_t)bc.m * p.D;
  const char* __restrict__ vb = reinterpret_cast<const char*>(p.value) + slab * sizeof(T) + j * V::kLaneBytes;
  char* __restrict__ gvb = reinterpret_cast<char*>(p.grad_value) + slab * (PACK ? sizeof(T) : 4u) + j * (kCpl * (PACK ? (int)sizeof(T) : 4));
  const float* __restrict__ loc = reinterpret_cast<const float*>(p.loc);
  const float* __restrict__ aw = reinterpret_cast<const float*>(p.aw);
  const T* __restrict__ gout = reinterpret_cast<const T*>(p.grad_out);
  float* __restrict__ gloc = reinterpret_cast<float*>(p.grad_loc);
  float* __restrict__ gaw = reinterpret_cast<float*>(p.grad_aw);

  // Software pipeline over the query loop (static variants): the next iteration's grad_out row, sampling
  // locations and attention weights are fetched before the current iteration is processed, so their HBM
  // latency is off the critical path.
  constexpr int kRounds = kStatic ? (LT * PT + G - 1) / G : 1;
  float2 nxy[kRounds];
  RefV nrf[kRounds];
  float na[kRounds];
  V ngo = V::zero();
  auto fetch = [&](int qw_, float2 (&xy_)[kRounds], float (&a_)[kRounds], RefV (&rf_)[kRounds], V& go_) {
    const int q_ = qw_ + grp;
    const bool act_ = q_ < bc.q_end;
    const int qq_ = act_ ? q_ : bc.q_begin;
    const size_t pair_ = ((size_t)bc.b * p.Lq + qq_) * p.M + bc.m;
    go_ = act_ ? V::load(gout + pair_ * p.D + j * kCpl) : V::zero();
#pragma unroll
    for (int r = 0; r < kRounds; ++r) {
      const int pi_ = r * G + j;
      xy_[r] = make_float2(0.f, 0.f);
      rf_[r] = RefV{};
      a_[r] = 0.f;
      if (pi_ < LP && act_) {
        if (FUSED) {  // explicit row strides: offsets / logits may be column blocks of one merged GEMM output
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
  if (kStatic) fetch(bc.q_begin + warp * kGpw, nxy, na, nrf, ngo);

  for (int qw = bc.q_begin + warp * kGpw; qw < bc.q_end; qw += kWarps * kGpw) {
    const int q = qw + grp;
    const bool active = q < bc.q_end;
    const size_t pair = ((size_t)bc.b * p.Lq + (active ? q : bc.q_begin)) * p.M + bc.m;
    const float* __restrict__ loc_pair = loc + pair * LP * 2;
    const float* __restrict__ aw_pair = aw + pair * LP;

    V go;
    float2 cxy[kRounds];
    RefV crf[kRounds];
    float ca[kRounds];
    float ga_keep[kRounds];  // fused: d/d(attention weight) of this lane's points, kept for the softmax backward
    float dot_part = 0.f;    // fused: this lane's share of sum_p a_p * dL/da_p
    float2 coff[RD == 4 && RGRAD ? kRounds : 1];  // boxes with RGRAD: the raw offsets (fused_resolve overwrites cxy)
    float rsum[RGRAD ? RD : 1];  // RGRAD, levels broadcast: this (b,q,m)'s reference-point gradient summed over all points
    if constexpr (RGRAD) {
#pragma unroll
      for (int c = 0; c < RD; ++c) rsum[c] = 0.f;
    }
    if (kStatic) {
      go = ngo;
#pragma unroll
      for (int r = 0; r < kRounds; ++r) { cxy[r] = nxy[r]; ca[r] = na[r]; crf[r] = nrf[r]; ga_keep[r] = 0.f; }
      if constexpr (RD == 4 && RGRAD) {
#pragma unroll
        for (int r = 0; r < kRounds; ++r) coff[r] = cxy[r];
      }
      if (qw + kWarps * kGpw < bc.q_end) fetch(qw + kWarps * kGpw, nxy, na, nrf, ngo);
      if constexpr (FUSED) fused_resolve<G, kRounds, (FUSED ? PT : 1)>(cxy, ca, crf, sH, sW, j, LP);
    } else {
      go = active ? V::load(gout + pair * p.D + j * kCpl) : V::zero();
    }

#pragma unroll
    for (int r0 = 0; r0 < (kStatic ? LT * PT : LP); r0 += G) {
      // ---- producer: lane j prepares point r0 + j -----------------------------------------------
      const int pi = r0 + j;
      const bool mine = (pi < LP) && active;
      unsigned tokf = 0u, wrow = 0u;  // clamped top-left token index << 4 | (rl, rh, cl, ch) validity bits
      float lh = 0.f, lw = 0.f, a = 0.f, fH = 0.f, fW = 0.f;
      if (mine) {
        const int l = pi / P;
        const int H = sH[l], W = sW[l];
        float2 xy;
        if (kStatic) {
          xy = cxy[r0 / G];
          a = ca[r0 / G];
        } else {
          xy = __ldg(reinterpret_cast<const float2*>(loc_pair) + pi);
          a = __ldg(aw_pair + pi);
        }
        const PointGeom<float> g = point_geom<float>(xy.x, xy.y, H, W);
        lh = g.lh; lw = g.lw;
        const unsigned rl = (g.mask & 3u) != 0u, rh = (g.mask & 12u) != 0u;  // row h_low / h_high readable
        const unsigned cl = (g.mask & 5u) != 0u, ch = (g.mask & 10u) != 0u;  // col w_low / w_high readable
        const int hl = max(g.h_low, 0), wl = max(g.w_low, 0);
        tokf = ((unsigned)(sStart[l] + hl * W + wl) << 4) | rl | (rh << 1) | (cl << 2) | (ch << 3);
        wrow = (unsigned)W;
        fH = (float)H; fW = (float)W;
      }
      float part[kTranspose ? 3 * G : 3];
      float my_ga = 0.f, my_gw = 0.f, my_gh = 0.f;
      // ---- consumers ------------------------------------------------------------------------------
#pragma unroll
      for (int jj = 0; jj < G; ++jj) {
        float s_a = 0.f, s_w = 0.f, s_h = 0.f;
        if (r0 + jj < LP) {  // uniform
          const unsigned tf = __shfl_sync(0xffffffffu, tokf, jj, G);
          const float flh = __shfl_sync(0xffffffffu, lh, jj, G);
          const float flw = __shfl_sync(0xffffffffu, lw, jj, G);
          const float fa = __shfl_sync(0xffffffffu, a, jj, G);
          unsigned wr;
          if (kStatic) {
            wr = rsl[(r0 + jj) / (kStatic ? PT : 1)];
          } else {
            wr = __shfl_sync(0xffffffffu, wrow, jj, G);
          }
          const bool rl = tf & 1u, rh = tf & 2u, cl = tf & 4u, ch = tf & 8u;
          const unsigned tok = tf >> 4;
          const unsigned dcol = (cl && ch) ? 1u : 0u;  // in tokens
          const unsigned drow = (rl && rh) ? wr : 0u;
          const unsigned t1 = tok, t2 = tok + dcol, t3 = tok + drow, t4 = tok + drow + dcol;
          const V v1 = V::load(reinterpret_cast<const T*>(ptr_madd(vb, t1, MDb)));
          const V v2 = V::load(reinterpret_cast<const T*>(ptr_madd(vb, t2, MDb)));
          const V v3 = V::load(reinterpret_cast<const T*>(ptr_madd(vb, t3, MDb)));
          const V v4 = V::load(reinterpret_cast<const T*>(ptr_madd(vb, t4, MDb)));
          float u1 = 0.f, u2 = 0.f, u3 = 0.f, u4 = 0.f;
#pragma unroll
          for (int c = 0; c < kCpl; ++c) {
            u1 = fmaf(go.v[c], v1.v[c], u1);
            u2 = fmaf(go.v[c], v2.v[c], u2);
            u3 = fmaf(go.v[c], v3.v[c], u3);
            u4 = fmaf(go.v[c], v4.v[c], u4);
          }
          const bool m1 = rl && cl, m2 = rl && ch, m3 = rh && cl, m4 = rh && ch;
          u1 = m1 ? u1 : 0.f; u2 = m2 ? u2 : 0.f; u3 = m3 ? u3 : 0.f; u4 = m4 ? u4 : 0.f;
          const float hh = 1.f - flh, hw = 1.f - flw;
          const float w1 = hh * hw, w2 = hh * flw, w3 = flh * hw, w4 = flh * flw;
          s_a = w1 * u1 + w2 * u2 + w3 * u3 + w4 * u4;
          s_w = hh * (u2 - u1) + flh * (u4 - u3);
          s_h = hw * (u3 - u1) + flw * (u4 - u2);
          // scatter: grad_value[corner k] += (w_k * attn) * grad_out
          const float a1 = w1 * fa, a2 = w2 * fa, a3 = w3 * fa, a4 = w4 * fa;
          if constexpr (PACK) {
            static_assert(kCpl == 4, "one packed reduction per lane per corner");
            if (m1) red_add_16x4<T>(const_cast<char*>(ptr_madd(gvb, t1, MDf)), a1 * go.v[0], a1 * go.v[1], a1 * go.v[2], a1 * go.v[3]);
            if (m2) red_add_16x4<T>(const_cast<char*>(ptr_madd(gvb, t2, MDf)), a2 * go.v[0], a2 * go.v[1], a2 * go.v[2], a2 * go.v[3]);
            if (m3) red_add_16x4<T>(const_cast<char*>(ptr_madd(gvb, t3, MDf)), a3 * go.v[0], a3 * go.v[1], a3 * go.v[2], a3 * go.v[3]);
            if (m4) red_add_16x4<T>(const_cast<char*>(ptr_madd(gvb, t4, MDf)), a4 * go.v[0], a4 * go.v[1], a4 * go.v[2], a4 * go.v[3]);
          } else {
#pragma unroll
            for (int c0 = 0; c0 < kCpl; c0 += 4) {
              if (m1) red_add_v4(reinterpret_cast<float*>(const_cast<char*>(ptr_madd(gvb, t1, MDf))) + c0, a1 * go.v[c0], a1 * go.v[c0 + 1], a1 * go.v[c0 + 2], a1 * go.v[c0 + 3]);
              if (m2) red_add_v4(reinterpret_cast<float*>(const_cast<char*>(ptr_madd(gvb, t2, MDf))) + c0, a2 * go.v[c0], a2 * go.v[c0 + 1], a2 * go.v[c0 + 2], a2 * go.v[c0 + 3]);
              if (m3) red_add_v4(reinterpret_cast<float*>(const_cast<char*>(ptr_madd(gvb, t3, MDf))) + c0, a3 * go.v[c0], a3 * go.v[c0 + 1], a3 * go.v[c0 + 2], a3 * go.v[c0 + 3]);
              if (m4) red_add_v4(reinterpret_cast<float*>(const_cast<char*>(ptr_madd(gvb, t4, MDf))) + c0, a4 * go.v[c0], a4 * go.v[c0 + 1], a4 * go.v[c0 + 2], a4 * go.v[c0 + 3]);
            }
          }
        }
        if constexpr (kTranspose) {
          part[3 * jj + 0] = s_a; part[3 * jj + 1] = s_w; part[3 * jj + 2] = s_h;
        } else if (r0 + jj < LP) {
          s_a = group_sum<G>(s_a);
          s_w = group_sum<G>(s_w);
          s_h = group_sum<G>(s_h);
          if (j == jj) { my_ga = s_a; my_gw = s_w; my_gh = s_h; }
        }
      }
      if constexpr (kTranspose) {
        group_transpose_sum<G, 3 * G>(part, j);
        my_ga = part[0]; my_gw = part[1]; my_gh = part[2];
      }
      if constexpr (FUSED) {
        // dL/dloc exactly as the plain kernel writes grad_sampling_loc (boxes and reference-point gradients need it)
        const float gx = fW * my_gw * a, gy = fH * my_gh * a;
        if constexpr (RD == 2) {
          // d loc / d offset = 1 / (W, H): the (W, H) factors of grad_sampling_loc cancel
          if (mine) {
            const size_t row = (size_t)bc.b * p.Lq + q;
            *reinterpret_cast<float2*>(gloc + row * p.off_rowstride + (size_t)bc.m * LP * 2 + 2 * pi) = make_float2(my_gw * a, my_gh * a);
          }
        } else {
          // boxes: d loc / d offset = ref_wh * 0.5 / P, applied in the order torch's autograd applies it
          if (mine) {
            const size_t row = (size_t)bc.b * p.Lq + q;
            const RefV rf = crf[r0 / G];
            *reinterpret_cast<float2*>(gloc + row * p.off_rowstride + (size_t)bc.m * LP * 2 + 2 * pi) =
                make_float2(__fmul_rn(__fmul_rn(__fmul_rn(gx, 0.5f), rf.z), kInvP), __fmul_rn(__fmul_rn(__fmul_rn(gy, 0.5f), rf.w), kInvP));
          }
        }
        if constexpr (RGRAD) {
          // d ref_xy = dL/dloc; boxes: d ref_wh = (dL/dloc * 0.5) * (offset / P)
          float gr[RD];
          gr[0] = mine ? gx : 0.f;
          gr[1] = mine ? gy : 0.f;
          if constexpr (RD == 4) {
            gr[2] = mine ? __fmul_rn(__fmul_rn(gx, 0.5f), __fmul_rn(coff[r0 / G].x, kInvP)) : 0.f;
            gr[3] = mine ? __fmul_rn(__fmul_rn(gy, 0.5f), __fmul_rn(coff[r0 / G].y, kInvP)) : 0.f;
          }
          // the PT points of a level are PT aligned consecutive lanes of this round: sum them
#pragma unroll
          for (int s = 1; s < PT; s <<= 1)
#pragma unroll
            for (int c = 0; c < RD; ++c) gr[c] += __shfl_xor_sync(0xffffffffu, gr[c], s, G);
          if (p.ref_lstride != 0) {  // one reference point per level: that level's partial is complete
            if (mine && j % PT == 0) {
              float* dst = p.ref_partial + ((((size_t)bc.b * p.Lq + q) * p.M + bc.m) * LT + pi / PT) * RD;
              if constexpr (RD == 4) *reinterpret_cast<float4*>(dst) = make_float4(gr[0], gr[1], gr[2], gr[3]);
              else *reinterpret_cast<float2*>(dst) = make_float2(gr[0], gr[1]);
            }
          } else {  // one reference point for all levels: sum the levels of this round, then the rounds
#pragma unroll
            for (int s = PT; s < G; s <<= 1)
#pragma unroll
              for (int c = 0; c < RD; ++c) gr[c] += __shfl_xor_sync(0xffffffffu, gr[c], s, G);
#pragma unroll
            for (int c = 0; c < RD; ++c) rsum[c] += gr[c];
          }
        }
        ga_keep[r0 / G] = mine ? my_ga : 0.f;
        dot_part = fmaf(a, ga_keep[r0 / G], dot_part);
      } else if (mine) {
        gaw[pair * LP + pi] = my_ga;
        reinterpret_cast<float2*>(gloc)[pair * LP + pi] = make_float2(fW * my_gw * a, fH * my_gh * a);
      }
    }
    if constexpr (RGRAD) {
      if (p.ref_lstride == 0 && active && j == 0) {
        float* dst = p.ref_partial + (((size_t)bc.b * p.Lq + q) * p.M + bc.m) * RD;
        if constexpr (RD == 4) *reinterpret_cast<float4*>(dst) = make_float4(rsum[0], rsum[1], rsum[2], rsum[3]);
        else *reinterpret_cast<float2*>(dst) = make_float2(rsum[0], rsum[1]);
      }
    }
    if constexpr (FUSED) {
      // softmax backward: d logit_p = a_p * (dL/da_p - sum_p' a_p' dL/da_p')
      const float dot = group_sum<G>(dot_part);
#pragma unroll
      for (int r = 0; r < kRounds; ++r) {
        const int pi = r * G + j;
        if (pi < LP && active)
          gaw[((size_t)bc.b * p.Lq + q) * p.logit_rowstride + (size_t)bc.m * LP + pi] = ca[r] * (ga_keep[r] - dot);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Generic kernel: any D / dtype / L,P. One warp per (b,q,m), lanes stride over channels, scalar
// atomics. AT = type of the grad_value accumulator (float scratch for bf16).
// ---------------------------------------------------------------------------------------------
template <typename T, typename F, typename AT>
__global__ void __launch_bounds__(kThreads) msda_bwd_generic_kernel(const Params p) {
  const int L = p.L, P = p.P, LP = L * P, MD = p.M * p.D;
  const BlockCoord bc = block_coord(p);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t img = (size_t)bc.b * p.S * MD + bc.m * p.D;
  const T* __restrict__ vb = reinterpret_cast<const T*>(p.value) + img;
  AT* __restrict__ gvb = reinterpret_cast<AT*>(p.grad_value) + img;
  const F* __restrict__ loc = reinterpret_cast<const F*>(p.loc);
  const F* __restrict__ aw = reinterpret_cast<const F*>(p.aw);
  const T* __restrict__ gout = reinterpret_cast<const T*>(p.grad_out);
  F* __restrict__ gloc = reinterpret_cast<F*>(p.grad_loc);
  F* __restrict__ gaw = reinterpret_cast<F*>(p.grad_aw);

  for (int q = bc.q_begin + warp; q < bc.q_end; q += kWarps) {
    const size_t pair = ((size_t)bc.b * p.Lq + q) * p.M + bc.m;
    for (int l = 0; l < L; ++l) {
      const int H = (int)p.shapes[2 * l], W = (int)p.shapes[2 * l + 1];
      const int start = (int)p.lsi[l];
      for (int k = 0; k < P; ++k) {
        const size_t pi = pair * LP + l * P + k;
        const F x = loc[2 * pi], y = loc[2 * pi + 1], a = aw[pi];
        const PointGeom<F> g = point_geom<F>(x, y, H, W);
        F s_a = 0, s_w = 0, s_h = 0;
        if (g.mask != 0u) {
          const F hh = 1 - g.lh, hw = 1 - g.lw;
          const F w1 = hh * hw, w2 = hh * g.lw, w3 = g.lh * hw, w4 = g.lh * g.lw;
          const size_t o = (size_t)(start + g.h_low * W + g.w_low) * MD;
          const size_t rs = (size_t)W * MD;
          for (int c = lane; c < p.D; c += 32) {
            const F go = (F)ld_scalar(gout + pair * p.D + c);
            const T* p1 = vb + o + c;
            AT* g1 = gvb + o + c;
            const F tg = go * a;
            F v1 = 0, v2 = 0, v3 = 0, v4 = 0;
            if (g.mask & 1u) { v1 = (F)ld_scalar(p1); atomicAdd(g1, (AT)(w1 * tg)); }
            if (g.mask & 2u) { v2 = (F)ld_scalar(p1 + MD); atomicAdd(g1 + MD, (AT)(w2 * tg)); }
            if (g.mask & 4u) { v3 = (F)ld_scalar(p1 + rs); atomicAdd(g1 + rs, (AT)(w3 * tg)); }
            if (g.mask & 8u) { v4 = (F)ld_scalar(p1 + rs + MD); atomicAdd(g1 + rs + MD, (AT)(w4 * tg)); }
            s_a += go * (w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4);
            s_w += go * (hh * (v2 - v1) + g.lh * (v4 - v3));
            s_h += go * (hw * (v3 - v1) + g.lw * (v4 - v2));
          }
        }
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
          s_a += __shfl_xor_sync(0xffffffffu, s_a, s);
          s_w += __shfl_xor_sync(0xffffffffu, s_w, s);
          s_h += __shfl_xor_sync(0xffffffffu, s_h, s);
        }
        if (lane == 0) {
          gaw[pi] = s_a;
          gloc[2 * pi] = (F)W * s_w * a;
          gloc[2 * pi + 1] = (F)H * s_h * a;
        }
      }
    }
  }
}

// fp32 scratch -> bf16 / fp16 grad_value (n is a multiple of 8 on the vector path; tail handled scalar).
template <typename TO>
__global__ void __launch_bounds__(kThreads) msda_cvt_f32_bf16_kernel(const float* __restrict__ src, TO* __restrict__ dst, size_t n) {
  const size_t nvec = n / 8;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(src) + 2 * i);
    const float4 b = __ldcs(reinterpret_cast<const float4*>(src) + 2 * i + 1);
    uint4 o;
    o.x = Vec<TO>::pack2(a.x, a.y);
    o.y = Vec<TO>::pack2(a.z, a.w);
    o.z = Vec<TO>::pack2(b.x, b.y);
    o.w = Vec<TO>::pack2(b.z, b.w);
    reinterpret_cast<uint4*>(dst)[i] = o;
  }
  for (size_t i = nvec * 8 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    st_scalar(dst + i, src[i]);
}

// The same conversion for a grad_value that is not 16-byte aligned: the C ABI only requires the element size.
template <typename TO>
__global__ void __launch_bounds__(kThreads) msda_cvt_f32_bf16_scalar_kernel(const float* __restrict__ src, TO* __restrict__ dst, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    st_scalar(dst + i, src[i]);
}

// ---------------------------------------------------------------------------------------------
// Launchers
// ---------------------------------------------------------------------------------------------
template <typename T, int G, int MINB>
static cudaError_t launch_vec_gm(const Params& p, dim3 grid, cudaStream_t s) {
  if (p.L == 3 && p.P == 4) {
    msda_bwd_vec_kernel<T, G, 3, 4, MINB><<<grid, kThreads, 0, s>>>(p);
  } else if (p.L == 1 && p.P == 4) {
    msda_bwd_vec_kernel<T, G, 1, 4, MINB><<<grid, kThreads, 0, s>>>(p);
  } else {
    msda_bwd_vec_kernel<T, G, 0, 0, MINB><<<grid, kThreads, 0, s>>>(p);
  }
  return cudaGetLastError();
}

template <typename T, int G>
static cudaError_t launch_vec_g(const Params& p, int minb, dim3 grid, cudaStream_t s) {
  switch (minb) {
    case 2: return launch_vec_gm<T, G, 2>(p, grid, s);
    case 4: return launch_vec_gm<T, G, 4>(p, grid, s);
    default: return launch_vec_gm<T, G, 3>(p, grid, s);
  }
}

// The fused kernel for the call's reference width (p.ref_dim) and whether it writes reference-point gradient partials
// (p.ref_partial): f(std::integral_constant<int, RD>, std::bool_constant<RGRAD>).
template <class F>
static cudaError_t with_ref_variant(const Params& p, F&& f) {
  if (p.ref_dim == 4)
    return p.ref_partial ? f(std::integral_constant<int, 4>{}, std::true_type{}) : f(std::integral_constant<int, 4>{}, std::false_type{});
  return p.ref_partial ? f(std::integral_constant<int, 2>{}, std::true_type{}) : f(std::integral_constant<int, 2>{}, std::false_type{});
}

template <typename T, int G>
static cudaError_t launch_fused_g(const Params& p, dim3 grid, cudaStream_t s) {
  return with_ref_variant(p, [&](auto rd, auto rg) {
    constexpr int RD = decltype(rd)::value;
    constexpr bool RG = decltype(rg)::value;
    if (p.L == 3 && p.P == 4) msda_bwd_vec_kernel<T, G, 3, 4, 3, true, false, RD, RG><<<grid, kThreads, 0, s>>>(p);
    else if (p.L == 1 && p.P == 4) msda_bwd_vec_kernel<T, G, 1, 4, 3, true, false, RD, RG><<<grid, kThreads, 0, s>>>(p);
    else if (p.L == 4 && p.P == 4) msda_bwd_vec_kernel<T, G, 4, 4, 3, true, false, RD, RG><<<grid, kThreads, 0, s>>>(p);
    else return cudaErrorNotSupported;
    return cudaGetLastError();
  });
}

template <typename T>
static cudaError_t launch_vec(const Params& p, int G, int minb, dim3 grid, cudaStream_t s) {
  switch (G) {
    case 2: return launch_vec_gm<T, 2, 3>(p, grid, s);
    case 4: return launch_vec_g<T, 4>(p, minb, grid, s);
    case 8: return launch_vec_g<T, 8>(p, minb, grid, s);
    case 16: return launch_vec_g<T, 16>(p, minb, grid, s);
    case 32: return launch_vec_gm<T, 32, 3>(p, grid, s);
    default: return cudaErrorInvalidValue;
  }
}

template <typename T>
static cudaError_t launch_fused_t(const Params& p, int G, dim3 grid, cudaStream_t s) {
  if (G == 8) return launch_fused_g<T, 8>(p, grid, s);
  if (G == 16) return launch_fused_g<T, 16>(p, grid, s);
  return cudaErrorNotSupported;
}

// opt-in packed 16-bit scatter (see red_add_16x4): the adapter configurations only - G in {8, 16}, (L, P) in {(3,4), (1,4)}
template <typename T, int G>
static cudaError_t launch_packed_g(const Params& p, bool fused, dim3 grid, cudaStream_t s) {
  if constexpr (sizeof(T) == 2) {
    const bool l3 = p.L == 3 && p.P == 4, l1 = p.L == 1 && p.P == 4;
    if (!l3 && !l1) return cudaErrorNotSupported;
    if (fused) {
      return with_ref_variant(p, [&](auto rd, auto rg) {
        constexpr int RD = decltype(rd)::value;
        constexpr bool RG = decltype(rg)::value;
        if (l3) msda_bwd_vec_kernel<T, G, 3, 4, 3, true, true, RD, RG><<<grid, kThreads, 0, s>>>(p);
        else msda_bwd_vec_kernel<T, G, 1, 4, 3, true, true, RD, RG><<<grid, kThreads, 0, s>>>(p);
        return cudaGetLastError();
      });
    } else {
      if (l3) msda_bwd_vec_kernel<T, G, 3, 4, 3, false, true><<<grid, kThreads, 0, s>>>(p);
      else msda_bwd_vec_kernel<T, G, 1, 4, 3, false, true><<<grid, kThreads, 0, s>>>(p);
    }
    return cudaGetLastError();
  } else {
    return cudaErrorNotSupported;
  }
}
template <typename T>
static cudaError_t launch_packed_t(const Params& p, int G, bool fused, dim3 grid, cudaStream_t s) {
  if (G == 8) return launch_packed_g<T, 8>(p, fused, grid, s);
  if (G == 16) return launch_packed_g<T, 16>(p, fused, grid, s);
  return cudaErrorNotSupported;
}

template <typename TO>
static cudaError_t launch_cvt_t(const float* src, void* dst, size_t n, cudaStream_t s) {
  const bool vec = reinterpret_cast<uintptr_t>(dst) % 16 == 0;  // 16-byte stores
  size_t blocks = ((vec ? n / 8 : n) + kThreads - 1) / kThreads;
  if (blocks < 1) blocks = 1;
  if (blocks > 148u * 16u) blocks = 148u * 16u;
  if (vec) msda_cvt_f32_bf16_kernel<TO><<<(unsigned)blocks, kThreads, 0, s>>>(src, reinterpret_cast<TO*>(dst), n);
  else msda_cvt_f32_bf16_scalar_kernel<TO><<<(unsigned)blocks, kThreads, 0, s>>>(src, reinterpret_cast<TO*>(dst), n);
  return cudaGetLastError();
}

// The file is compiled once per value dtype (build.py: -DMSDA_TU=0 f32 + f64 + dispatch, 1 bf16, 2 f16) so that the three
// sets of instantiations build in parallel; each part exports its entry points under a dtype suffix.
#ifndef MSDA_TU
#define MSDA_TU 0
#endif
cudaError_t bwd_vec_bf16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s);
cudaError_t bwd_fused_bf16(const Params& p, int G, dim3 grid, cudaStream_t s);
cudaError_t bwd_generic_bf16(const Params& p, dim3 grid, cudaStream_t s);
cudaError_t bwd_cvt_bf16(const float* src, void* dst, size_t n, cudaStream_t s);
cudaError_t bwd_vec_f16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s);
cudaError_t bwd_fused_f16(const Params& p, int G, dim3 grid, cudaStream_t s);
cudaError_t bwd_generic_f16(const Params& p, dim3 grid, cudaStream_t s);
cudaError_t bwd_cvt_f16(const float* src, void* dst, size_t n, cudaStream_t s);
cudaError_t bwd_packed_bf16(const Params& p, int G, bool fused, dim3 grid, cudaStream_t s);
cudaError_t bwd_packed_f16(const Params& p, int G, bool fused, dim3 grid, cudaStream_t s);

#if MSDA_TU == 1
cudaError_t bwd_packed_bf16(const Params& p, int G, bool fused, dim3 grid, cudaStream_t s) { return launch_packed_t<__nv_bfloat16>(p, G, fused, grid, s); }
cudaError_t bwd_vec_bf16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s) { return launch_vec<__nv_bfloat16>(p, G, minb, grid, s); }
cudaError_t bwd_fused_bf16(const Params& p, int G, dim3 grid, cudaStream_t s) { return launch_fused_t<__nv_bfloat16>(p, G, grid, s); }
cudaError_t bwd_generic_bf16(const Params& p, dim3 grid, cudaStream_t s) {
  msda_bwd_generic_kernel<__nv_bfloat16, float, float><<<grid, kThreads, 0, s>>>(p);
  return cudaGetLastError();
}
cudaError_t bwd_cvt_bf16(const float* src, void* dst, size_t n, cudaStream_t s) { return launch_cvt_t<__nv_bfloat16>(src, dst, n, s); }
#elif MSDA_TU == 2
cudaError_t bwd_packed_f16(const Params& p, int G, bool fused, dim3 grid, cudaStream_t s) { return launch_packed_t<__half>(p, G, fused, grid, s); }
cudaError_t bwd_vec_f16(const Params& p, int G, int minb, dim3 grid, cudaStream_t s) { return launch_vec<__half>(p, G, minb, grid, s); }
cudaError_t bwd_fused_f16(const Params& p, int G, dim3 grid, cudaStream_t s) { return launch_fused_t<__half>(p, G, grid, s); }
cudaError_t bwd_generic_f16(const Params& p, dim3 grid, cudaStream_t s) {
  msda_bwd_generic_kernel<__half, float, float><<<grid, kThreads, 0, s>>>(p);
  return cudaGetLastError();
}
cudaError_t bwd_cvt_f16(const float* src, void* dst, size_t n, cudaStream_t s) { return launch_cvt_t<__half>(src, dst, n, s); }
#else
// fused entry: `p.grad_value` is the zero-filled fp32 accumulator (as in launch_backward)
cudaError_t launch_backward_fused(const Params& p, int dtype, int G, cudaStream_t s) {
  const dim3 grid((unsigned)((size_t)p.N * p.nchunk * p.M));
  if (dtype == MSDA_F32) return launch_fused_t<float>(p, G, grid, s);
  if (dtype == MSDA_BF16) return bwd_fused_bf16(p, G, grid, s);
  if (dtype == MSDA_F16) return bwd_fused_f16(p, G, grid, s);
  return cudaErrorNotSupported;
}

// `p.grad_value` must point at the ACCUMULATOR (T storage for f32/f64, fp32 scratch for bf16 / f16),
// already zero-filled on `s`.
cudaError_t launch_backward(const Params& p, int dtype, bool vec_ok, int G, int minb, cudaStream_t s) {
  const dim3 grid((unsigned)((size_t)p.N * p.nchunk * p.M));
  if (vec_ok) {
    if (dtype == MSDA_F32) return launch_vec<float>(p, G, minb, grid, s);
    if (dtype == MSDA_F16) return bwd_vec_f16(p, G, minb, grid, s);
    return bwd_vec_bf16(p, G, minb, grid, s);
  }
  switch (dtype) {
    case MSDA_F32: msda_bwd_generic_kernel<float, float, float><<<grid, kThreads, 0, s>>>(p); break;
    case MSDA_BF16: return bwd_generic_bf16(p, grid, s);
    case MSDA_F16: return bwd_generic_f16(p, grid, s);
    case MSDA_F64: msda_bwd_generic_kernel<double, double, double><<<grid, kThreads, 0, s>>>(p); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// `p.grad_value` = the zero-filled bf16 / fp16 grad_value itself. cudaErrorNotSupported when there is no packed kernel.
cudaError_t launch_backward_packed16(const Params& p, int dtype, int G, bool fused, cudaStream_t s) {
  const dim3 grid((unsigned)((size_t)p.N * p.nchunk * p.M));
  if (dtype == MSDA_BF16) return bwd_packed_bf16(p, G, fused, grid, s);
  if (dtype == MSDA_F16) return bwd_packed_f16(p, G, fused, grid, s);
  return cudaErrorNotSupported;
}

cudaError_t launch_cvt_f32_bf16(const float* src, void* dst, size_t n, int dtype, cudaStream_t s) {
  return dtype == MSDA_F16 ? bwd_cvt_f16(src, dst, n, s) : bwd_cvt_bf16(src, dst, n, s);
}

// grad_reference_points [Nr, Lq, Lr, RD] from the partials [N, Lq, M, Lr, RD] of the RGRAD fused backward: one thread per
// output float sums over the heads (and over the batch when Nr == 1), always in the order b, then m.
__global__ void __launch_bounds__(kThreads) msda_ref_grad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ out,
                                                                        int N, int Lq, int M, int Nr, int Lr, int RD) {
  const size_t per_q = (size_t)Lr * RD;
  const size_t total = (size_t)Nr * Lq * per_q;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t lc = i % per_q;
    const size_t q = (i / per_q) % Lq;
    const int b0 = (int)(i / (per_q * Lq));
    const int b1 = Nr == 1 ? N : b0 + 1;
    float acc = 0.f;
    for (int b = b0; b < b1; ++b) {
      const float* src = partial + (((size_t)b * Lq + q) * M) * per_q + lc;
      for (int m = 0; m < M; ++m) acc += src[(size_t)m * per_q];
    }
    out[i] = acc;
  }
}

cudaError_t launch_ref_grad_reduce(const Params& p, int ref_batch, int ref_levels, float* grad_ref, cudaStream_t s) {
  const size_t total = (size_t)ref_batch * p.Lq * ref_levels * p.ref_dim;
  size_t blocks = (total + kThreads - 1) / kThreads;
  if (blocks > 148u * 16u) blocks = 148u * 16u;
  msda_ref_grad_reduce_kernel<<<(unsigned)blocks, kThreads, 0, s>>>(p.ref_partial, grad_ref, p.N, p.Lq, p.M, ref_batch, ref_levels,
                                                                   p.ref_dim);
  return cudaGetLastError();
}
#endif  // MSDA_TU

}  // namespace msda
