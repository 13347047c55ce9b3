// adapter_layernorm.cu — the LayerNorm prologues of the adapter's Injector / Extractor (SURVEY.md §8(f) N2).
//
// Reference: `self.query_norm(query)`, `self.feat_norm(feat)`, `self.ffn_norm(query)` — nn.LayerNorm(dim, eps=1e-6) on
// [B, tokens, C] with C = 384 / 768 / 1024 (*/mm*_custom/models/backbones/adapter_modules.py:101-103,110-116,133-134,
// 142-145). Every one of them feeds a Linear; under AMP torch runs the LayerNorm in fp32, writes fp32, and the Linear
// then casts its input to the low-precision type with another full pass. Measured on B200 (profiles/r1_block_profile_*):
// at ViT-Adapter-B, 16 x 512^2, bf16 autocast, torch's five LayerNorms + their backward + those casts are ~2.3 ms of a
// 6.9 ms interaction, more than three times the deformable-attention kernels themselves.
//
// Here one warp owns one row. The row lives in registers (VPL 16-byte quads per lane), so x is read exactly once:
//   forward : mean and the centred second moment by warp shuffles, y = (x - mean) * rstd * gamma + beta written directly in
//             the consumer's dtype (bf16 under AMP), mean / rstd saved as fp32.
//   backward: xhat recomputed from the saved statistics, the two row sums (gamma*dy, gamma*dy*xhat) by warp shuffles,
//             dx written in x's dtype; dgamma / dbeta accumulate per lane across the rows the warp walks, are reduced over
//             the CTA's warps through shared memory, written as one partial row per CTA and summed in a fixed order by a
//             second kernel (deterministic, no atomics). When x also feeds a residual connection (query + f(LN(query))), the
//             gradient arriving over that connection is added into dx here, which removes autograd's separate add pass.
// Compulsory traffic: forward rows*C*(e_in + e_out); backward rows*C*(e_in + e_out + e_in).
#include <cuda_fp16.h>

#include "msda_common.cuh"

namespace msda {

struct LnParams {
  const void* x;        // [rows, C] TI
  const void* gamma;    // [C] fp32
  const void* beta;     // [C] fp32 (forward only)
  void* y;              // forward: [rows, C] TO
  float* mean;          // [rows]
  float* rstd;          // [rows]
  const void* grad_y;   // backward: [rows, C] TO
  void* grad_x;         // backward: [rows, C] TI
  float* partial;       // backward: [gridDim.x][2][C] per-CTA partial sums of dgamma, dbeta
  long long rows;
  int C;
  float eps;
  const void* grad_res; // backward, optional: [rows, C] TI gradient of the residual branch that shares x, added into grad_x
};

constexpr int kLnWarps = 8;

template <typename T> struct LnQuad;
template <> struct LnQuad<float> {
  static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) {
    const float4 q = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
  static __device__ __forceinline__ void ld_shared(const float* p, float (&v)[4]) {
    const float4 q = *reinterpret_cast<const float4*>(p);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
  static __device__ __forceinline__ void st(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct LnQuad<__nv_bfloat16> {
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float (&v)[4]) {
    const uint2 q = __ldg(reinterpret_cast<const uint2*>(p));
    v[0] = __uint_as_float(q.x << 16); v[1] = __uint_as_float(q.x & 0xffff0000u);
    v[2] = __uint_as_float(q.y << 16); v[3] = __uint_as_float(q.y & 0xffff0000u);
  }
  static __device__ __forceinline__ void ld_shared(const __nv_bfloat16* p, float (&v)[4]) {
    const uint2 q = *reinterpret_cast<const uint2*>(p);
    v[0] = __uint_as_float(q.x << 16); v[1] = __uint_as_float(q.x & 0xffff0000u);
    v[2] = __uint_as_float(q.y << 16); v[3] = __uint_as_float(q.y & 0xffff0000u);
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[4]) {
    uint2 o;
    o.x = Vec<__nv_bfloat16>::pack2(v[0], v[1]); o.y = Vec<__nv_bfloat16>::pack2(v[2], v[3]);
    *reinterpret_cast<uint2*>(p) = o;
  }
};

template <> struct LnQuad<__half> {
  static __device__ __forceinline__ void cvt(const uint2& q, float (&v)[4]) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&q.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&q.y));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
  static __device__ __forceinline__ void ld(const __half* p, float (&v)[4]) { cvt(__ldg(reinterpret_cast<const uint2*>(p)), v); }
  static __device__ __forceinline__ void ld_shared(const __half* p, float (&v)[4]) { cvt(*reinterpret_cast<const uint2*>(p), v); }
  static __device__ __forceinline__ void st(__half* p, const float (&v)[4]) {
    uint2 o;
    const __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
    o.x = *reinterpret_cast<const unsigned*>(&a); o.y = *reinterpret_cast<const unsigned*>(&b);
    *reinterpret_cast<uint2*>(p) = o;
  }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// lane owns quads at columns (i * 32 + lane) * 4, i < VPL; quads past C are masked out
template <typename TI, typename TO, int VPL>
__global__ void __launch_bounds__(kLnWarps * 32, 2) adapter_ln_fwd_kernel(const LnParams p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const TI* __restrict__ x = reinterpret_cast<const TI*>(p.x);
  TO* __restrict__ y = reinterpret_cast<TO*>(p.y);
  const float* __restrict__ gamma = reinterpret_cast<const float*>(p.gamma);
  const float* __restrict__ beta = reinterpret_cast<const float*>(p.beta);
  bool ok[VPL];
  float g[VPL][4], bt[VPL][4];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int col = (i * 32 + lane) * 4;
    ok[i] = col < p.C;
#pragma unroll
    for (int v = 0; v < 4; ++v) { g[i][v] = 0.f; bt[i][v] = 0.f; }
    if (ok[i]) {
      LnQuad<float>::ld(gamma + col, g[i]);
      if (beta) LnQuad<float>::ld(beta + col, bt[i]);
    }
  }
  const float inv_c = 1.0f / (float)p.C;
  for (long long row = (long long)blockIdx.x * kLnWarps + warp; row < p.rows; row += (long long)gridDim.x * kLnWarps) {
    const TI* xr = x + row * p.C;
    float xv[VPL][4];
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
#pragma unroll
      for (int v = 0; v < 4; ++v) xv[i][v] = 0.f;
      if (ok[i]) LnQuad<TI>::ld(xr + (i * 32 + lane) * 4, xv[i]);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) s += (xv[i][0] + xv[i][1]) + (xv[i][2] + xv[i][3]);
    const float m0 = warp_sum(s) * inv_c;
    // second pass: mean = m0 + mean(x - m0). The row sum's rounding scales with |x|, the correction's with the spread
    // |x - m0|: a row with a large common offset gets its mean to within the spread's precision, and a constant row gets
    // exactly its value (so y == beta, as with torch's Welford statistics) instead of an error that 1/sqrt(eps) magnifies
    float sd = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (ok[i]) sd += ((xv[i][0] - m0) + (xv[i][1] - m0)) + ((xv[i][2] - m0) + (xv[i][3] - m0));
    const float mean = m0 + warp_sum(sd) * inv_c;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (ok[i]) {
#pragma unroll
        for (int v = 0; v < 4; ++v) { const float d = xv[i][v] - mean; q = fmaf(d, d, q); }
      }
    const float var = warp_sum(q) * inv_c;
    const float rstd = 1.0f / sqrtf(var + p.eps);
    TO* yr = y + row * p.C;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (ok[i]) {
        float o[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) o[v] = fmaf((xv[i][v] - mean) * rstd, g[i][v], bt[i][v]);
        LnQuad<TO>::st(yr + (i * 32 + lane) * 4, o);
      }
    if (lane == 0) { p.mean[row] = mean; p.rstd[row] = rstd; }
  }
}

template <typename TI, typename TO, int VPL>
__global__ void __launch_bounds__(kLnWarps * 32, (VPL <= 6 ? 2 : 1)) adapter_ln_bwd_kernel(const LnParams p) {
  // one buffer, two lives: while rows are walked, warp w stages the residual-gradient row it will need at the store
  // (cp.async: bytes in flight that cost no registers) in its VPL*512-byte slice; afterwards the same memory is the
  // tree reduction over the warps (at most 4 rows of dgamma | dbeta)
  __shared__ __align__(16) float ln_smem[kLnWarps / 2 * 2 * VPL * 128];
  float (*red)[2 * VPL * 128] = reinterpret_cast<float (*)[2 * VPL * 128]>(ln_smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  TI* stage = reinterpret_cast<TI*>(ln_smem + warp * VPL * 128);
  const TI* __restrict__ x = reinterpret_cast<const TI*>(p.x);
  const TO* __restrict__ dy = reinterpret_cast<const TO*>(p.grad_y);
  TI* __restrict__ dx = reinterpret_cast<TI*>(p.grad_x);
  const TI* __restrict__ gres = reinterpret_cast<const TI*>(p.grad_res);
  const float* __restrict__ gamma = reinterpret_cast<const float*>(p.gamma);
  bool ok[VPL];
  float dg[VPL][4], db[VPL][4];  // gamma is re-read per row (L1-resident): 4*VPL registers matter more here
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    ok[i] = (i * 32 + lane) * 4 < p.C;
#pragma unroll
    for (int v = 0; v < 4; ++v) { dg[i][v] = 0.f; db[i][v] = 0.f; }
  }
  const float inv_c = 1.0f / (float)p.C;
  for (long long row = (long long)blockIdx.x * kLnWarps + warp; row < p.rows; row += (long long)gridDim.x * kLnWarps) {
    const TI* xr = x + row * p.C;
    const TO* dyr = dy + row * p.C;
    float xh[VPL][4], gy[VPL][4];
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
#pragma unroll
      for (int v = 0; v < 4; ++v) { xh[i][v] = 0.f; gy[i][v] = 0.f; }
      if (ok[i]) {
        LnQuad<TI>::ld(xr + (i * 32 + lane) * 4, xh[i]);
        LnQuad<TO>::ld(dyr + (i * 32 + lane) * 4, gy[i]);
      }
    }
    if (gres) {  // the residual gradient is only needed at the store: start it towards shared memory now
#pragma unroll
      for (int i = 0; i < VPL; ++i)
        if (ok[i]) {
          const unsigned dst = (unsigned)__cvta_generic_to_shared(stage + (i * 32 + lane) * 4);
          const TI* src = gres + row * p.C + (i * 32 + lane) * 4;
          if constexpr (sizeof(TI) == 4) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
          else asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
        }
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    const float mean = p.mean[row], rstd = p.rstd[row];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (ok[i]) {
        float g[4];
        LnQuad<float>::ld(gamma + (i * 32 + lane) * 4, g);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const float h = (xh[i][v] - mean) * rstd;
          xh[i][v] = h;
          db[i][v] += gy[i][v];
          dg[i][v] = fmaf(gy[i][v], h, dg[i][v]);
          const float t = gy[i][v] * g[v];
          gy[i][v] = t;  // gamma * dy
          s1 += t;
          s2 = fmaf(t, h, s2);
        }
      }
    s1 = warp_sum(s1) * inv_c;
    s2 = warp_sum(s2) * inv_c;
    TI* dxr = dx + row * p.C;
    if (gres) asm volatile("cp.async.wait_group 0;" ::: "memory");  // each lane reads back only what it copied itself
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (ok[i]) {
        float o[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) o[v] = (gy[i][v] - fmaf(xh[i][v], s2, s1)) * rstd;
        if (gres) {  // x also feeds a residual connection: fold that branch's gradient in here instead of a separate add pass
          float r[4];
          LnQuad<TI>::ld_shared(stage + (i * 32 + lane) * 4, r);
#pragma unroll
          for (int v = 0; v < 4; ++v) o[v] += r[v];
        }
        LnQuad<TI>::st(dxr + (i * 32 + lane) * 4, o);
      }
  }
  __syncthreads();  // every warp is done with its staging slice before the buffer becomes the reduction tree
  // tree over the 8 warps: upper half writes, lower half adds, in a fixed order
#pragma unroll
  for (int half = kLnWarps / 2; half > 0; half >>= 1) {
    if (warp >= half && warp < 2 * half) {
      float* r = red[warp - half];
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        *reinterpret_cast<float4*>(r + (i * 32 + lane) * 4) = make_float4(dg[i][0], dg[i][1], dg[i][2], dg[i][3]);
        *reinterpret_cast<float4*>(r + VPL * 128 + (i * 32 + lane) * 4) = make_float4(db[i][0], db[i][1], db[i][2], db[i][3]);
      }
    }
    __syncthreads();
    if (warp < half) {
      const float* r = red[warp];
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        const float4 a = *reinterpret_cast<const float4*>(r + (i * 32 + lane) * 4);
        const float4 b = *reinterpret_cast<const float4*>(r + VPL * 128 + (i * 32 + lane) * 4);
        dg[i][0] += a.x; dg[i][1] += a.y; dg[i][2] += a.z; dg[i][3] += a.w;
        db[i][0] += b.x; db[i][1] += b.y; db[i][2] += b.z; db[i][3] += b.w;
      }
    }
    __syncthreads();
  }
  if (warp == 0) {
    float* out = p.partial + (size_t)blockIdx.x * 2 * p.C;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (ok[i]) {
        LnQuad<float>::st(out + (i * 32 + lane) * 4, dg[i]);
        LnQuad<float>::st(out + p.C + (i * 32 + lane) * 4, db[i]);
      }
  }
}

// dgamma[c] = sum_r partial[r][0][c], dbeta[c] = sum_r partial[r][1][c]; block = (32 columns, 32 row slices), four
// independent partial sums per thread
__global__ void __launch_bounds__(1024) adapter_ln_param_grad_kernel(const float* __restrict__ partial, int rows, int C,
                                                                     float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ float red[32][33];
  const int i = blockIdx.x * 32 + threadIdx.x;  // column of the [2*C] partial row
  const int n = 2 * C;
  float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
  if (i < n) {
    int r = threadIdx.y;
    for (; r + 96 < rows; r += 128) {
      t0 += partial[(size_t)r * n + i];
      t1 += partial[(size_t)(r + 32) * n + i];
      t2 += partial[(size_t)(r + 64) * n + i];
      t3 += partial[(size_t)(r + 96) * n + i];
    }
    for (; r < rows; r += 32) t0 += partial[(size_t)r * n + i];
  }
  red[threadIdx.y][threadIdx.x] = (t0 + t1) + (t2 + t3);
  __syncthreads();
  if (threadIdx.y == 0 && i < n) {
    float t = 0.f;
#pragma unroll
    for (int yy = 0; yy < 32; ++yy) t += red[yy][threadIdx.x];
    if (i < C) dgamma[i] = t; else dbeta[i - C] = t;
  }
}

static unsigned ln_grid(long long rows) {
  const long long need = (rows + kLnWarps - 1) / kLnWarps;
  const long long resident = device_sm_count() * 2;
  return (unsigned)(need < resident ? (need ? need : 1) : resident);
}

bool layernorm_supported(int C) { return C > 0 && C % 4 == 0 && C <= 8 * 128; }

size_t layernorm_backward_workspace_bytes(long long rows, int C) { return (size_t)ln_grid(rows) * 2 * C * sizeof(float); }

template <typename TI, typename TO, bool BWD>
static cudaError_t ln_launch(const LnParams& p, cudaStream_t s) {
  const unsigned grid = ln_grid(p.rows);
  const int vpl = (p.C + 127) / 128;
#define LN_CASE(V)                                                                     \
  case V:                                                                              \
    if (BWD) adapter_ln_bwd_kernel<TI, TO, V><<<grid, kLnWarps * 32, 0, s>>>(p);       \
    else adapter_ln_fwd_kernel<TI, TO, V><<<grid, kLnWarps * 32, 0, s>>>(p);           \
    break;
  switch (vpl) {
    LN_CASE(1) LN_CASE(2) LN_CASE(3) LN_CASE(4) LN_CASE(5) LN_CASE(6) LN_CASE(7) LN_CASE(8)
    default: return cudaErrorInvalidValue;
  }
#undef LN_CASE
  return cudaGetLastError();
}

template <bool BWD>
static cudaError_t ln_dispatch(const LnParams& p, int in_dtype, int out_dtype, cudaStream_t s) {
  if (in_dtype == MSDA_F32 && out_dtype == MSDA_F32) return ln_launch<float, float, BWD>(p, s);
  if (in_dtype == MSDA_F32 && out_dtype == MSDA_BF16) return ln_launch<float, __nv_bfloat16, BWD>(p, s);
  if (in_dtype == MSDA_BF16 && out_dtype == MSDA_BF16) return ln_launch<__nv_bfloat16, __nv_bfloat16, BWD>(p, s);
  if (in_dtype == MSDA_F32 && out_dtype == MSDA_F16) return ln_launch<float, __half, BWD>(p, s);
  if (in_dtype == MSDA_F16 && out_dtype == MSDA_F16) return ln_launch<__half, __half, BWD>(p, s);
  return cudaErrorInvalidValue;
}

cudaError_t launch_layernorm_forward(const LnParams& p, int in_dtype, int out_dtype, cudaStream_t s) {
  return ln_dispatch<false>(p, in_dtype, out_dtype, s);
}

// two launches: the row kernel, then the parameter-gradient sum over its per-CTA partial rows
cudaError_t launch_layernorm_backward(const LnParams& p, int in_dtype, int out_dtype, float* dgamma, float* dbeta, cudaStream_t s) {
  cudaError_t e = ln_dispatch<true>(p, in_dtype, out_dtype, s);
  if (e != cudaSuccess) return e;
  adapter_ln_param_grad_kernel<<<(2 * p.C + 31) / 32, dim3(32, 32), 0, s>>>(p.partial, (int)ln_grid(p.rows), p.C, dgamma, dbeta);
  return cudaGetLastError();
}

}  // namespace msda
