// msda_abi.cu — extern "C" boundary declared in include/msda_b200.h.
//
// Host-side role of the reference's ms_deform_attn_cuda.cu:20-153 (argument checks, dimension
// extraction, launches on the caller's stream) without any ATen type: raw pointers in, error code
// out. No allocation, no synchronisation, no global mutable state besides two tuning knobs and a
// launch counter (all atomics).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "msda_common.cuh"

namespace msda {
bool vec_supported(int dtype, int D, int* G_out);
cudaError_t launch_forward(const Params& p, int dtype, bool vec_ok, int G, int minb, cudaStream_t s);
cudaError_t launch_backward(const Params& p, int dtype, bool vec_ok, int G, int minb, cudaStream_t s);
cudaError_t launch_cvt_f32_bf16(const float* src, void* dst, size_t n, int dtype, cudaStream_t s);
cudaError_t launch_backward_packed16(const Params& p, int dtype, int G, bool fused, cudaStream_t s);
cudaError_t launch_forward_fused(const Params& p, int dtype, int G, cudaStream_t s);
cudaError_t launch_backward_fused(const Params& p, int dtype, int G, cudaStream_t s);
cudaError_t launch_ref_grad_reduce(const Params& p, int ref_batch, int ref_levels, float* grad_ref, cudaStream_t s);
struct DwParams {
  const void* x;
  const void* w;
  const void* bias;
  void* y;
  int B, Ntok, C, H, W;
};
cudaError_t launch_dwconv(const DwParams& p, int dtype, bool flip, cudaStream_t s);
size_t dwconv_wgrad_workspace_bytes(const DwParams& p, int dtype);
cudaError_t launch_dwconv_wgrad(const DwParams& p, int dtype, const void* grad_y, void* gw, void* gb, void* workspace,
                                size_t workspace_bytes, int* launches, cudaStream_t s);
struct LnParams {
  const void* x;
  const void* gamma;
  const void* beta;
  void* y;
  float* mean;
  float* rstd;
  const void* grad_y;
  void* grad_x;
  float* partial;
  long long rows;
  int C;
  float eps;
  const void* grad_res;
};
cudaError_t launch_residual_add(int branch_dtype, const float* res, const void* branch, float* out, long long n, cudaStream_t s);
bool layernorm_supported(int C);
size_t layernorm_backward_workspace_bytes(long long rows, int C);
cudaError_t launch_layernorm_forward(const LnParams& p, int in_dtype, int out_dtype, cudaStream_t s);
cudaError_t launch_layernorm_backward(const LnParams& p, int in_dtype, int out_dtype, float* dgamma, float* dbeta, cudaStream_t s);
bool colsum_supported(int dtype, int C);
size_t colsum_workspace_bytes(int dtype, long long rows, int C);
cudaError_t launch_colsum(int dtype, const void* x, long long rows, int C, float* out, float* partial, cudaStream_t s);
cudaError_t launch_forward_wide(const Params& p, int G, int minb, cudaStream_t s);
struct CellPlan {
  unsigned off_tl, off_go, off_scr, off_ubuf, off_hist, total;
  int hist_cap;
};
int backward_cell_max_points();
bool plan_backward_cell(int D, int LP, int esize, int qc, int hist_cap, unsigned budget, CellPlan* cp);
cudaError_t launch_backward_cell(const Params& p, const CellPlan& cp, int dtype, cudaStream_t s);
size_t backward_sorted_workspace_bytes(int N, int S, int M, int D, int L, int Lq, int P, int sm_count);
cudaError_t launch_backward_sorted(const Params& p, int dtype, void* ws, int sm_count, int* launches, cudaStream_t s);
cudaError_t launch_forward_smem(const Params& p, const SmemPlan& plan, int dtype, int G, int nt, cudaStream_t s);

static thread_local char g_err[512] = "";
constexpr bool kFwdWideDefault = false;  // flipped once measured faster (tuning key "fwd_wide" = 2 forces it)
static std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_qc_fwd{0}, g_qc_bwd{0}, g_minb_fwd{0}, g_minb_bwd{0}, g_smem_mode{0}, g_smem_nt{0}, g_smem_chunks{0}, g_fwd_wide{0}, g_bwd_cell{0}, g_bwd_cell_qc{0}, g_bwd_packed16{0}, g_bwd_sorted{0};

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

static int cuda_fail(cudaError_t e, const char* fmt, ...) {
  char what[256];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(what, sizeof(what), fmt, ap);
  va_end(ap);
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  return (int)e;
}

// 0, or the return code of a failed launch
static int launched(cudaError_t e, const char* what) { return e == cudaSuccess ? 0 : cuda_fail(e, "%s", what); }

// The fused launchers return cudaErrorNotSupported when they have no kernel for G.
static int fused_launched(cudaError_t e, const char* who, int G) {
  if (e == cudaErrorNotSupported) return fail(MSDA_E_UNSUPPORTED, "%s: no fused kernel for G=%d", who, G);
  return e == cudaSuccess ? 0 : cuda_fail(e, "%s launch", who);
}

static size_t elem_size(int dtype) {
  return dtype == MSDA_F32 ? 4 : (dtype == MSDA_BF16 || dtype == MSDA_F16) ? 2 : dtype == MSDA_F64 ? 8 : 0;
}

static int check_dims(const msda_dims* d, int dtype) {
  if (!d) return fail(MSDA_E_NULL, "dims is NULL");
  if (elem_size(dtype) == 0) return fail(MSDA_E_DTYPE, "unknown dtype %d", dtype);
  if (d->batch <= 0 || d->spatial_size <= 0 || d->num_heads <= 0 || d->channels <= 0 ||
      d->num_levels <= 0 || d->num_query <= 0 || d->num_point <= 0)
    return fail(MSDA_E_DIMS, "non-positive dimension (N=%d S=%d M=%d D=%d L=%d Lq=%d P=%d)", d->batch,
                d->spatial_size, d->num_heads, d->channels, d->num_levels, d->num_query, d->num_point);
  if (d->num_levels > MSDA_MAX_LEVELS)
    return fail(MSDA_E_LEVELS, "num_levels=%d exceeds MSDA_MAX_LEVELS=%d", d->num_levels, MSDA_MAX_LEVELS);
  // in-image byte offsets are uint32 in the kernels (the reference is int32 element offsets throughout);
  // the token index shares a register with 4 flag bits.
  const int64_t per_image = (int64_t)d->spatial_size * d->num_heads * d->channels;
  const int64_t per_pair = (int64_t)d->num_levels * d->num_point;
  if (per_image >= (1ll << 29) || per_pair >= (1ll << 20) || d->spatial_size >= (1 << 27) ||
      (int64_t)d->num_heads * d->channels >= (1ll << 24))
    return fail(MSDA_E_DIMS, "S*M*D=%lld does not fit the 32-bit in-image byte offset", (long long)per_image);
  return 0;
}

static bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

static int sm_count() { return device_sm_count(); }

// Queries per CTA chunk of the query-order kernels (a multiple of the queries one pass of the CTA serves). Two regimes,
// MEASURED at every chunk size (tools/chunk_sweep.py, profiles/r2_chunk_sweep.jsonl; B / S / L, fp32 and bf16):
//   dense calls (>= 8 samples per value token and head: the Extractors, 21): consecutive queries gather the same value rows,
//     so long chunks keep them in L1 - ViT-Adapter-B Extractor forward 124 us at 256 queries per CTA, 140 at 64, 166 at 32:
//     enough CTAs to fill the SMs ~8 times over, chunks as long as possible otherwise (<= 256);
//   sparse calls (the Injectors, 2.3): nothing to reuse, and a CTA's time is proportional to its queries, so the shortest
//     chunk gives the evenest last round - ViT-Adapter-B Injector, 1 024 queries x 192 slabs: 7 chunks of 160 (the last one 64
//     long) were 1 344 CTAs = 3.03 rounds of 3 x 148 -> backward 239 us, 32 chunks of 32 are 13.8 rounds -> 226 us; S
//     226 -> 216 us, forward 86 -> 80; L bs 1 forward 37.7 -> 32.8 us.
static int pick_chunk(const msda_dims* d, int per_iter, int override_qc) {
  int qc;
  if (override_qc > 0) {
    qc = override_qc;
  } else if ((int64_t)d->num_query * d->num_levels * d->num_point < 8 * (int64_t)d->spatial_size) {
    qc = per_iter > 32 ? per_iter : 32;
  } else {
    const int64_t bm = (int64_t)d->batch * d->num_heads;
    const int64_t target_ctas = (int64_t)sm_count() * 8;
    int64_t chunks = (target_ctas + bm - 1) / bm;
    if (chunks < 1) chunks = 1;
    qc = (int)((d->num_query + chunks - 1) / chunks);
    if (qc > 256) qc = 256;
  }
  qc = ((qc + per_iter - 1) / per_iter) * per_iter;
  if (qc < per_iter) qc = per_iter;
  return qc;
}

// Plan the shared-memory forward from host-known level shapes: the set of levels (smallest first) whose
// [H*W, D] maps of one head fit the budget, and the number of query chunks per (b, m).
// MEASURED OUTCOME (profiles/r1_fwd_smem_vs_l1.md): not a robust win over the L1-path forward at the adapter
// shapes (B 512^2 bs16 Extractor 115.6 vs 121.8 us fp32, 77.8 vs 97.3 us bf16; Injector 98-115 vs 97 us): with
// the row gathers down to one LSU wavefront each, the 5 broadcast shuffles per point keep the kernel at ~79 % of
// the same LSU data pipe. So it is OPT-IN (tuning key "fwd_smem" = 2).
static bool plan_forward_smem(const msda_dims* d, int dtype, int G, const int64_t* hs, int nt, SmemPlan* plan,
                              int* qc_out, int* nchunk_out) {
  if (!hs || dtype == MSDA_F16) return false;   // the staged forward is instantiated for f32 / bf16
  const int L = d->num_levels;
  if (!((L == 3 || L == 1) && d->num_point == 4)) return false;
  const int mode = g_smem_mode.load();
  if (mode != 2) return false;  // opt-in only, see above
  const unsigned rowB = (unsigned)G * 16u;
  memset(plan, 0, sizeof(*plan));
  int64_t start = 0;
  int order[kMaxLevels];
  int64_t bytes[kMaxLevels];
  for (int l = 0; l < L; ++l) {
    const int64_t H = hs[2 * l], W = hs[2 * l + 1];
    if (H <= 0 || W <= 0 || H > (1 << 20) || W > (1 << 20)) return false;
    plan->H[l] = (int)H; plan->W[l] = (int)W; plan->start[l] = (int)start;
    start += H * W;
    bytes[l] = (H + 2) * (W + 2) * (int64_t)rowB;  // zero-padded by one token on every side
    order[l] = l;
  }
  if (start != d->spatial_size) return false;  // host shapes do not describe this value tensor
  for (int a = 0; a < L; ++a)
    for (int b = a + 1; b < L; ++b)
      if (bytes[order[b]] < bytes[order[a]]) { const int t = order[a]; order[a] = order[b]; order[b] = t; }
  // Layout: [null block of zeros | staged level maps]. The null block is where skipped samples point; it must
  // cover the 2x2 footprint at the row stride of the widest staged level: (W + 2) + 2 rows.
  int nstaged = 0;
  int64_t total = 0;
  for (int pass = 0; pass < 2; ++pass) {
    int64_t maxW = 0;
    for (int l = 0; l < L; ++l)
      if (plan->staged & (1u << l)) maxW = plan->W[l] > maxW ? plan->W[l] : maxW;
    const int64_t null_bytes = pass == 0 ? 0 : (maxW + 4) * (int64_t)rowB;
    plan->staged = 0;
    nstaged = 0;
    total = null_bytes;
    for (int a = 0; a < L; ++a) {
      const int l = order[a];
      // pass 0 sizes the candidate set without the null block; pass 1 re-fits with it (may drop the largest)
      const int64_t reserve = pass == 0 ? (int64_t)(plan->W[l] + 4) * rowB : 0;
      // static shared memory of the kernel: the per-warp tap scratch, (nt / 32) warps x (32 / G) groups x (2G + 1) x 16 bytes
      const int64_t scratch = (int64_t)(nt / 32) * (32 / G) * (2 * G + 1) * 16 + 512;
      if (total + bytes[l] + reserve + scratch > (int64_t)kSmemBudget) break;
      plan->smem_off[l] = (unsigned)total;
      plan->staged |= 1u << l;
      total += bytes[l];
      ++nstaged;
    }
    if (nstaged == 0) return false;
  }
  plan->total_bytes = (unsigned)total;

  const int per_iter = (nt / 32) * (32 / G);
  const double bm = (double)d->batch * d->num_heads;
  const double g_smem = (double)d->num_query * nstaged * d->num_point * 4.0 * rowB;        // per (b,m), bytes
  const double g_l1 = (double)d->num_query * (L - nstaged) * d->num_point * 4.0 * rowB;
  const double t_l1_only = (g_smem + g_l1) / 62.0 * ceil(bm / (double)sm_count() / 4.0) ;  // rough; only the ratio below matters
  (void)t_l1_only;
  int best_c = 0;
  double best_t = 1e300;
  const int max_c = d->num_query / per_iter > 0 ? d->num_query / per_iter : 1;
  for (int c = 1; c <= 64 && c <= max_c; ++c) {
    const double waves = ceil(bm * c / (double)sm_count());
    const double per_cta = (g_smem / 245.0 + g_l1 / 62.0) / c + (double)total / 80.0;
    const double t = waves * per_cta;
    if (t < best_t) { best_t = t; best_c = c; }
  }
  const int forced = g_smem_chunks.load();
  if (forced > 0) best_c = forced < max_c ? forced : max_c;
  if (best_c == 0) return false;
  int qc = (d->num_query + best_c - 1) / best_c;
  qc = ((qc + per_iter - 1) / per_iter) * per_iter;
  *qc_out = qc;
  *nchunk_out = (d->num_query + qc - 1) / qc;
  return true;
}

// Cell-bucketed backward (msda_bwd_cell.cu): queries per chunk, histogram window and the shared-memory plan. The chunk is
// made as long as the shared memory of a CTA allows at 3 (else 2, else 1) resident CTAs per SM - longer chunks mean longer
// runs of points per bilinear cell - then shortened while the grid would leave SMs idle.
static bool plan_cell(const msda_dims* d, int dtype, Params& p, CellPlan* cp) {
  // MEASURED OUTCOME (profiles/r2_bwd_cell_*.{json,txt}): the cell-bucketed backward cuts the row atomics that reach the L2
  // 3.5x (58 M -> 17 M RED sectors at ViT-Adapter-B bs 16) but spends as many instructions per point on bucketing and
  // record handling as the query-order kernel spends on its gathers, at fewer eligible warps: 360 vs 320 us (Extractor),
  // 335 vs 240 us (Injector). So it is OPT-IN (tuning key "bwd_cell" = 2); 0 / 1 = off.
  const int mode = g_bwd_cell.load();
  if (mode != 2) return false;
  if (!(dtype == MSDA_F32 || dtype == MSDA_BF16 || dtype == MSDA_F16)) return false;
  if (!(d->channels == 32 || d->channels == 64)) return false;
  if (d->spatial_size >= (1 << 19)) return false;  // cell words keep the corner token in 20 bits
  const int LP = d->num_levels * d->num_point, es = (int)elem_size(dtype);
  const int max_qc = backward_cell_max_points() / LP;
  if (max_qc < 1) return false;
  // 228 KB per SM, 1 KB reserved per resident CTA, a few hundred bytes of static shared memory
  const unsigned budgets[3] = {74u * 1024u, 112u * 1024u, 226u * 1024u};
  const int per_cta[3] = {3, 2, 1};
  const int forced = g_bwd_cell_qc.load();
  const int hist_cap = d->spatial_size < 4096 ? d->spatial_size : 4096;  // one key window; larger bands take several
  for (int t = 0; t < 3; ++t) {
    int lo = forced > 0 ? forced : 1;
    if (lo > d->num_query) lo = d->num_query;
    if (lo > max_qc) lo = max_qc;
    CellPlan probe;
    if (!plan_backward_cell(d->channels, LP, es, lo, hist_cap, budgets[t], &probe)) continue;
    int qc = lo;
    if (forced <= 0) {
      const long long per_q = (long long)LP * 20 + (long long)d->channels * es;
      qc = (int)(lo + ((long long)budgets[t] - (long long)probe.total) / per_q);
      if (qc > d->num_query) qc = d->num_query;
      if (qc > max_qc) qc = max_qc;
      while (qc > lo && !plan_backward_cell(d->channels, LP, es, qc, hist_cap, budgets[t], &probe)) --qc;  // rounding slack
      // keep every SM busy for at least two rounds of resident CTAs when the problem is large enough
      const long long want = 2ll * sm_count() * per_cta[t];
      const long long bm = (long long)d->batch * d->num_heads;
      while (qc > 64 && bm * ((d->num_query + qc - 1) / qc) < want) qc = (qc + 1) / 2;
      const int nchunk = (d->num_query + qc - 1) / qc;
      qc = (d->num_query + nchunk - 1) / nchunk;  // equal chunks
    }
    if (!plan_backward_cell(d->channels, LP, es, qc, hist_cap, budgets[t], cp)) continue;
    p.qc = qc;
    p.nchunk = (d->num_query + qc - 1) / qc;
    return true;
  }
  return false;
}

// The dims and the inputs every entry point has (for the fused ones `loc` / `aw` are the raw offsets / logits)
static void fill_params(Params& p, const msda_dims* d, const void* value, const int64_t* shapes, const int64_t* lsi,
                        const void* loc, const void* aw) {
  memset(&p, 0, sizeof(p));
  p.N = d->batch; p.S = d->spatial_size; p.M = d->num_heads; p.D = d->channels;
  p.L = d->num_levels; p.Lq = d->num_query; p.P = d->num_point;
  p.value = value; p.shapes = shapes; p.lsi = lsi; p.loc = loc; p.aw = aw;
}

// Common tail of the forward entry points: chunk the queries for CTAs that serve `per_iter` of them per pass, then
// `launch()` (0 or a return code) and count it.
template <class Launch>
static int forward_tail(const msda_dims* d, Params& p, int per_iter, Launch&& launch) {
  p.qc = pick_chunk(d, per_iter, g_qc_fwd.load());
  p.nchunk = (p.Lq + p.qc - 1) / p.qc;
  if (int e = launch()) return e;
  g_launches.fetch_add(1);
  return 0;
}

// Where the scatter accumulates grad_value: grad_value itself for f32 / f64; for bf16 / f16 the fp32 scratch at the start of
// the workspace, converted into grad_value afterwards.
static void* backward_accum(int dtype, void* grad_value, void* workspace) {
  return dtype == MSDA_BF16 || dtype == MSDA_F16 ? workspace : grad_value;
}

// The backward after its argument checks, shared by both entry points: chunk the queries, zero-fill the accumulator, let
// `scatter(&launches)` accumulate into p.grad_value (0 or a return code; it sets `launches` if it issues more than one kernel),
// convert a 16-bit result, count the launches. `vec`: the 4-channel lane layout (G = D / 4) applies; the fused entry points
// (the ones that set p.ref) always meet it and the conditions of the packed 16-bit kernels.
template <class Scatter>
static int backward_body(const char* who, const msda_dims* dims, int dtype, Params& p, bool vec, void* grad_value,
                         void* workspace, cudaStream_t s, Scatter&& scatter) {
  const int G = p.D / 4;
  p.qc = pick_chunk(dims, vec ? kWarps * (32 / G) : kWarps, g_qc_bwd.load());
  p.nchunk = (p.Lq + p.qc - 1) / p.qc;
  const size_t nvalue = (size_t)p.N * p.S * p.M * p.D;
  const bool lowp = dtype == MSDA_BF16 || dtype == MSDA_F16;
  // packed 16-bit reductions straight into grad_value (no fp32 scratch, no convert; see msda_bwd.cu red_add_16x4)
  if (lowp && vec && g_bwd_packed16.load() == 2 && (G == 8 || G == 16) && ((p.L == 3 || p.L == 1) && p.P == 4) &&
      aligned(grad_value, 8)) {
    p.grad_value = grad_value;
    cudaError_t e = cudaMemsetAsync(grad_value, 0, nvalue * elem_size(dtype), s);
    if (e != cudaSuccess) return cuda_fail(e, "%s memset(grad_value)", who);
    e = launch_backward_packed16(p, dtype, G, p.ref != nullptr, s);
    if (e != cudaSuccess) return cuda_fail(e, "%s (packed 16-bit reductions) launch", who);
    g_launches.fetch_add(1);
    return 0;
  }
  p.grad_value = backward_accum(dtype, grad_value, workspace);
  cudaError_t e = cudaMemsetAsync(p.grad_value, 0, nvalue * (lowp ? sizeof(float) : elem_size(dtype)), s);
  if (e != cudaSuccess) return cuda_fail(e, "%s memset(grad_value)", who);
  int launches = 1;
  if (int rc = scatter(&launches)) return rc;
  g_launches.fetch_add(launches);
  if (lowp) {
    e = launch_cvt_f32_bf16(reinterpret_cast<const float*>(p.grad_value), grad_value, nvalue, dtype, s);
    if (e != cudaSuccess) return cuda_fail(e, "%s bf16 convert launch", who);
    g_launches.fetch_add(1);
  }
  return 0;
}

// ---- debug: per-point index dump (same point_geom the kernels use) -----------------------------
__global__ void msda_debug_index_kernel(const int64_t* shapes, const int64_t* lsi, const float* loc,
                                        int32_t* idx, int N, int M, int D, int L, int Lq, int P) {
  const size_t total = (size_t)N * Lq * M * L * P;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (size_t)gridDim.x * blockDim.x) {
    const int l = (int)((i / P) % L);
    const int m = (int)((i / ((size_t)P * L)) % M);
    const int H = (int)shapes[2 * l], W = (int)shapes[2 * l + 1];
    const PointGeom<float> g = point_geom<float>(loc[2 * i], loc[2 * i + 1], H, W);
    idx[4 * i + 0] = g.h_low;
    idx[4 * i + 1] = g.w_low;
    idx[4 * i + 2] = (int)g.mask;
    idx[4 * i + 3] = ((int)lsi[l] + g.h_low * W + g.w_low) * (M * D) + m * D;
  }
}
}  // namespace msda

using namespace msda;

extern "C" {

int msda_abi_version(void) { return MSDA_ABI_VERSION; }

const char* msda_last_error(void) { return g_err; }

uint64_t msda_launch_count(void) { return g_launches.load(); }

int msda_set_tuning(const char* key, int32_t value) {
  if (!key) return fail(MSDA_E_NULL, "msda_set_tuning: NULL key");
  std::atomic<int>* slot = nullptr;
  if (!strcmp(key, "fwd_chunk")) slot = &g_qc_fwd;
  else if (!strcmp(key, "bwd_chunk")) slot = &g_qc_bwd;
  else if (!strcmp(key, "fwd_min_ctas")) slot = &g_minb_fwd;
  else if (!strcmp(key, "bwd_min_ctas")) slot = &g_minb_bwd;
  else if (!strcmp(key, "fwd_smem")) slot = &g_smem_mode;
  else if (!strcmp(key, "fwd_smem_threads")) slot = &g_smem_nt;
  else if (!strcmp(key, "fwd_smem_chunks")) slot = &g_smem_chunks;
  else if (!strcmp(key, "fwd_wide")) slot = &g_fwd_wide;
  else if (!strcmp(key, "bwd_cell")) slot = &g_bwd_cell;
  else if (!strcmp(key, "bwd_cell_chunk")) slot = &g_bwd_cell_qc;
  else if (!strcmp(key, "bwd_packed16")) slot = &g_bwd_packed16;
  else if (!strcmp(key, "bwd_sorted")) slot = &g_bwd_sorted;
  if (!slot) return fail(MSDA_E_NULL, "msda_set_tuning: unknown key '%s'", key);
  slot->store(value);
  return 0;
}

int msda_check_im2col_step(int32_t batch, int32_t im2col_step) {
  if (batch <= 0 || im2col_step <= 0) return fail(MSDA_E_STEP, "batch(%d) / im2col_step(%d) must be positive", batch, im2col_step);
  const int step = batch < im2col_step ? batch : im2col_step;
  if (batch % step != 0) return fail(MSDA_E_STEP, "batch(%d) must divide im2col_step(%d)", batch, step);
  return 0;
}

int msda_forward(const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                 const int64_t* level_start_index, const void* sampling_loc, const void* attn_weight,
                 void* out, void* stream) {
  return msda_forward_ex(dims, dtype, value, spatial_shapes, level_start_index, sampling_loc, attn_weight, out,
                         nullptr, stream);
}

int msda_forward_ex(const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                    const int64_t* level_start_index, const void* sampling_loc, const void* attn_weight,
                    void* out, const int64_t* spatial_shapes_host, void* stream) {
  if (int e = check_dims(dims, dtype)) return e;
  if (!value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight || !out)
    return fail(MSDA_E_NULL, "msda_forward: NULL tensor pointer");
  const size_t es = elem_size(dtype), fs = dtype == MSDA_F64 ? 8 : 4;
  if (!aligned(value, es) || !aligned(out, es) || !aligned(sampling_loc, fs) || !aligned(attn_weight, fs) ||
      !aligned(spatial_shapes, 8) || !aligned(level_start_index, 8))
    return fail(MSDA_E_ALIGN, "msda_forward: pointer not aligned to its element size");

  Params p;
  fill_params(p, dims, value, spatial_shapes, level_start_index, sampling_loc, attn_weight);
  p.out = out;

  int G = 0;
  bool vec = vec_supported(dtype, p.D, &G) && aligned(value, 16) && aligned(out, 16) &&
             aligned(sampling_loc, 8);
  if (vec && spatial_shapes_host) {
    SmemPlan plan;
    const int nt = g_smem_nt.load() == 1024 ? 1024 : 512;
    if (plan_forward_smem(dims, dtype, G, spatial_shapes_host, nt, &plan, &p.qc, &p.nchunk)) {
      const cudaError_t es2 = launch_forward_smem(p, plan, dtype, G, nt, (cudaStream_t)stream);
      if (es2 == cudaSuccess) {
        g_launches.fetch_add(1);
        return 0;
      }
      if (es2 != cudaErrorNotSupported) return cuda_fail(es2, "msda_forward (shared-memory variant) launch");
    }
  }
  // fp32 with 32-byte lanes (LDG.256): 8 channels per lane, G = D/8
  const int wide_mode = g_fwd_wide.load();  // 0 auto, 1 off, 2 on
  if (vec && dtype == MSDA_F32 && wide_mode != 1 && p.D % 8 == 0 && aligned(value, 32) && aligned(out, 32)) {
    const int Gw = p.D / 8;
    if (Gw >= 2 && Gw <= 8 && (Gw & (Gw - 1)) == 0 && (wide_mode == 2 || kFwdWideDefault)) {
      p.qc = pick_chunk(dims, kWarps * (32 / Gw), g_qc_fwd.load());
      p.nchunk = (p.Lq + p.qc - 1) / p.qc;
      const cudaError_t ew = launch_forward_wide(p, Gw, g_minb_fwd.load(), (cudaStream_t)stream);
      if (ew == cudaSuccess) {
        g_launches.fetch_add(1);
        return 0;
      }
      if (ew != cudaErrorNotSupported) return cuda_fail(ew, "msda_forward (32-byte lanes) launch");
    }
  }
  return forward_tail(dims, p, vec ? kWarps * (32 / G) : kWarps, [&] {
    return launched(launch_forward(p, dtype, vec, G, g_minb_fwd.load(), (cudaStream_t)stream), "msda_forward launch");
  });
}

// fp32 accumulator of the 16-bit dtypes (first in the workspace), then the sort buffers of the slab-sorted backward
static size_t accum_workspace_bytes(const msda_dims* d, int dtype) {
  if (dtype != MSDA_BF16 && dtype != MSDA_F16) return 0;
  return (size_t)d->batch * d->spatial_size * d->num_heads * d->channels * sizeof(float);
}
// Slab-sorted backward (msda_bwd_sorted.cu). Tuning key "bwd_sorted": 0 = where it measured faster, 1 = off, 2 = wherever it
// applies. MEASURED (profiles/r2_bwd_sorted_vs_query_order.jsonl and r2_bwd_sorted_small_batches.jsonl, B200, L2 flushed,
// query order -> sorted): the sort costs ~45 us per 4 M samples plus four launches, the walker ~26 instructions per sample
// whatever the row length, so it pays where cell runs are long (one level, >= 16 samples per value token and head: the
// Extractor calls) and the call is large enough for the launches: from ~1 M samples at 128-byte rows (D = 32), ~0.25 M at
// 256-byte rows (D = 64), whose row atomics cost twice as much in query order:
//   ViT-Adapter-B Extractor bs 16  322 -> 267 us fp32 (1.21x), 337 -> 277 bf16     S bs 16  331 -> 241 (1.37x), 337 -> 230 bf16 (1.46x)
//   L 16x64 bs 1  196 -> 144 (1.35x), bf16 202 -> 136 (1.48x)     L 16x32 bs 1  105 -> 101, bf16 112 -> 105     T bs 16  1.09-1.11x
//   B bs 4 (1.0 M samples) 1.04-1.09x, bs 2 1.0-1.03x, bs 1 0.81-0.87x       S bs 4 (0.5 M) 1.19-1.32x, bs 2 (0.26 M) 1.11-1.19x, bs 1 0.90x
//   (small batches re-measured after the sort's scan became one kernel: profiles/r2_bwd_sorted_small_batches.jsonl)
// It loses on the Injectors (3 levels, ~2 samples per cell: 0.76-0.93x), which keep the query-order kernel.
static size_t sorted_workspace_bytes(const msda_dims* d, int dtype) {
  const int mode = g_bwd_sorted.load();
  if (mode == 1) return 0;
  if (!(dtype == MSDA_F32 || dtype == MSDA_BF16 || dtype == MSDA_F16)) return 0;
  if (g_bwd_cell.load() == 2 || g_bwd_packed16.load() == 2) return 0;  // an explicitly requested opt-in kernel wins
  if (mode != 2) {
    const long long samples_per_slab = (long long)d->num_query * d->num_levels * d->num_point;
    const long long samples = samples_per_slab * d->batch * d->num_heads;
    if (samples_per_slab < 16ll * d->spatial_size) return 0;
    if (samples < (d->channels == 64 ? 250000ll : 1000000ll)) return 0;
  }
  return backward_sorted_workspace_bytes(d->batch, d->spatial_size, d->num_heads, d->channels, d->num_levels, d->num_query,
                                         d->num_point, sm_count());
}

size_t msda_backward_workspace_bytes(const msda_dims* dims, int dtype) {
  if (!dims) return 0;
  return accum_workspace_bytes(dims, dtype) + sorted_workspace_bytes(dims, dtype);
}

int msda_backward(const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                  const int64_t* level_start_index, const void* sampling_loc, const void* attn_weight,
                  const void* grad_out, void* grad_value, void* grad_sampling_loc, void* grad_attn_weight,
                  void* workspace, size_t workspace_bytes, void* stream) {
  if (int e = check_dims(dims, dtype)) return e;
  if (!value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight || !grad_out ||
      !grad_value || !grad_sampling_loc || !grad_attn_weight)
    return fail(MSDA_E_NULL, "msda_backward: NULL tensor pointer");
  const size_t es = elem_size(dtype), fs = dtype == MSDA_F64 ? 8 : 4;
  if (!aligned(value, es) || !aligned(grad_out, es) || !aligned(grad_value, es) ||
      !aligned(sampling_loc, fs) || !aligned(attn_weight, fs) || !aligned(grad_sampling_loc, fs) ||
      !aligned(grad_attn_weight, fs) || !aligned(spatial_shapes, 8) || !aligned(level_start_index, 8))
    return fail(MSDA_E_ALIGN, "msda_backward: pointer not aligned to its element size");
  const size_t need = msda_backward_workspace_bytes(dims, dtype);
  if (need > 0 && (!workspace || workspace_bytes < need || !aligned(workspace, 16)))
    return fail(MSDA_E_WORKSPACE, "msda_backward: workspace of %zu bytes (16-byte aligned) required, got %zu",
                need, workspace ? workspace_bytes : (size_t)0);

  Params p;
  fill_params(p, dims, value, spatial_shapes, level_start_index, sampling_loc, attn_weight);
  p.grad_out = grad_out; p.grad_loc = grad_sampling_loc; p.grad_aw = grad_attn_weight;

  // backward lane layout: 4 channels per lane for every dtype (see VecB in msda_bwd.cu)
  const int G = p.D / 4;
  const bool vec = (dtype == MSDA_F32 || dtype == MSDA_BF16 || dtype == MSDA_F16) && p.D % 4 == 0 && G >= 2 && G <= 32 &&
                   (G & (G - 1)) == 0 && aligned(value, 16) && aligned(grad_out, 16) && aligned(sampling_loc, 8) &&
                   aligned(grad_sampling_loc, 8) && aligned(backward_accum(dtype, grad_value, workspace), 16);
  const cudaStream_t s = (cudaStream_t)stream;
  return backward_body("msda_backward", dims, dtype, p, vec, grad_value, workspace, s, [&](int* launches) {
    CellPlan cplan;
    if (vec && sorted_workspace_bytes(dims, dtype) > 0)
      return launched(launch_backward_sorted(p, dtype, reinterpret_cast<char*>(workspace) + accum_workspace_bytes(dims, dtype),
                                             sm_count(), launches, s),
                      "msda_backward (slab-sorted) launch");
    if (vec && plan_cell(dims, dtype, p, &cplan))
      return launched(launch_backward_cell(p, cplan, dtype, s), "msda_backward (cell-bucketed) launch");
    return launched(launch_backward(p, dtype, vec, G, g_minb_bwd.load(), s), "msda_backward launch");
  });
}

// (L, P) of the fused kernels
static bool fused_levels_points(const msda_dims* d) {
  return (d->num_levels == 3 || d->num_levels == 1 || d->num_levels == 4) && d->num_point == 4;
}

static int check_ref_dim(int32_t ref_dim) {
  if (ref_dim != 2 && ref_dim != 4) return fail(MSDA_E_DIMS, "fused entry: ref_dim=%d, expected 2 (points) or 4 (boxes)", ref_dim);
  return 0;
}

static bool ref_broadcasts(const msda_dims* d, int32_t ref_batch, int32_t ref_levels) {
  return (ref_batch == 1 || ref_batch == d->batch) && (ref_levels == 1 || ref_levels == d->num_levels);
}

static int check_ref_broadcast(const msda_dims* d, int32_t ref_batch, int32_t ref_levels, int32_t ref_dim) {
  if (!ref_broadcasts(d, ref_batch, ref_levels))
    return fail(MSDA_E_DIMS, "fused entry: reference_points [%d, Lq, %d, %d] does not broadcast to N=%d, L=%d", ref_batch,
                ref_levels, ref_dim, d->batch, d->num_levels);
  return 0;
}

static int fused_ref_params(Params& p, const msda_dims* d, const float* ref, int32_t ref_batch, int32_t ref_levels,
                            int32_t ref_dim, int64_t off_rowstride, int64_t logit_rowstride) {
  const int64_t mlp = (int64_t)d->num_heads * d->num_levels * d->num_point;
  p.off_rowstride = off_rowstride > 0 ? off_rowstride : mlp * 2;
  p.logit_rowstride = logit_rowstride > 0 ? logit_rowstride : mlp;
  if (p.off_rowstride < mlp * 2 || p.logit_rowstride < mlp || (p.off_rowstride & 1))
    return fail(MSDA_E_DIMS, "fused entry: row strides (%lld, %lld) smaller than a row or odd", (long long)p.off_rowstride,
                (long long)p.logit_rowstride);
  if (!ref) return fail(MSDA_E_NULL, "fused entry: reference_points is NULL");
  if (int e = check_ref_broadcast(d, ref_batch, ref_levels, ref_dim)) return e;
  if (!aligned(ref, 4 * (size_t)ref_dim))  // one 8-byte (point) or 16-byte (box) load per reference point
    return fail(MSDA_E_ALIGN, "fused entry: reference_points not %d-byte aligned", 4 * ref_dim);
  p.ref = ref;
  p.ref_dim = ref_dim;
  p.ref_qstride = ref_levels * ref_dim;
  p.ref_lstride = ref_levels == 1 ? 0 : ref_dim;
  p.ref_bstride = ref_batch == 1 ? 0 : (long long)d->num_query * ref_levels * ref_dim;
  return 0;
}

// Backward scratch of the fused entry: the fp32 accumulator of the 16-bit dtypes, then (16-byte aligned) the
// reference-point gradient partials [N, Lq, M, Lr, ref_dim] when that gradient is wanted.
static size_t ref_partial_offset(const msda_dims* d, int dtype) { return (accum_workspace_bytes(d, dtype) + 15) & ~(size_t)15; }
static size_t fused_workspace_bytes(const msda_dims* d, int dtype, int32_t ref_levels, int32_t ref_dim, bool with_ref_grad) {
  if (!with_ref_grad) return accum_workspace_bytes(d, dtype);
  return ref_partial_offset(d, dtype) +
         (size_t)d->batch * d->num_query * d->num_heads * ref_levels * ref_dim * sizeof(float);
}

// The fused forward of both entry points (msda_forward_fused is the ref_dim = 2 case).
static int forward_fused_body(const char* who, const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                              const int64_t* level_start_index, const float* reference_points, int32_t ref_batch,
                              int32_t ref_levels, int32_t ref_dim, const float* sampling_offsets, const float* attn_logits,
                              int64_t offsets_row_stride, int64_t logits_row_stride, void* out, void* stream) {
  if (int e = check_dims(dims, dtype)) return e;
  if (!value || !spatial_shapes || !level_start_index || !sampling_offsets || !attn_logits || !out)
    return fail(MSDA_E_NULL, "%s: NULL tensor pointer", who);
  int G = 0;
  if (!vec_supported(dtype, dims->channels, &G) || !fused_levels_points(dims))
    return fail(MSDA_E_UNSUPPORTED, "%s: no fused kernel for dtype=%d D=%d L=%d P=%d", who, dtype, dims->channels,
                dims->num_levels, dims->num_point);
  if (int e = check_ref_dim(ref_dim)) return e;
  if (!aligned(value, 16) || !aligned(out, 16) || !aligned(sampling_offsets, 8) || !aligned(attn_logits, 4) ||
      !aligned(spatial_shapes, 8) || !aligned(level_start_index, 8))
    return fail(MSDA_E_ALIGN, "%s: misaligned pointer", who);
  Params p;
  fill_params(p, dims, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits);
  p.out = out;
  if (int e = fused_ref_params(p, dims, reference_points, ref_batch, ref_levels, ref_dim, offsets_row_stride, logits_row_stride))
    return e;
  return forward_tail(dims, p, kWarps * (32 / G), [&] {
    return fused_launched(launch_forward_fused(p, dtype, G, (cudaStream_t)stream), who, G);
  });
}

int msda_forward_fused(const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                       const int64_t* level_start_index, const float* reference_points, int32_t ref_batch,
                       int32_t ref_levels, const float* sampling_offsets, const float* attn_logits,
                       int64_t offsets_row_stride, int64_t logits_row_stride, void* out, void* stream) {
  return forward_fused_body("msda_forward_fused", dims, dtype, value, spatial_shapes, level_start_index, reference_points,
                            ref_batch, ref_levels, 2, sampling_offsets, attn_logits, offsets_row_stride, logits_row_stride,
                            out, stream);
}

int msda_forward_fused_ref(const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                           const int64_t* level_start_index, const float* reference_points, int32_t ref_batch,
                           int32_t ref_levels, int32_t ref_dim, const float* sampling_offsets, const float* attn_logits,
                           int64_t offsets_row_stride, int64_t logits_row_stride, void* out, void* stream) {
  return forward_fused_body("msda_forward_fused_ref", dims, dtype, value, spatial_shapes, level_start_index, reference_points,
                            ref_batch, ref_levels, ref_dim, sampling_offsets, attn_logits, offsets_row_stride,
                            logits_row_stride, out, stream);
}

// The fused backward of both entry points (msda_backward_fused is the ref_dim = 2, grad_reference_points = NULL case).
static int backward_fused_body(const char* who, const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                               const int64_t* level_start_index, const float* reference_points, int32_t ref_batch,
                               int32_t ref_levels, int32_t ref_dim, const float* sampling_offsets, const float* attn_logits,
                               int64_t offsets_row_stride, int64_t logits_row_stride, const void* grad_out, void* grad_value,
                               float* grad_sampling_offsets, float* grad_attn_logits, float* grad_reference_points,
                               void* workspace, size_t workspace_bytes, void* stream) {
  if (int e = check_dims(dims, dtype)) return e;
  if (!value || !spatial_shapes || !level_start_index || !sampling_offsets || !attn_logits || !grad_out || !grad_value ||
      !grad_sampling_offsets || !grad_attn_logits)
    return fail(MSDA_E_NULL, "%s: NULL tensor pointer", who);
  const int G = dims->channels / 4;
  if (!(dtype == MSDA_F32 || dtype == MSDA_BF16 || dtype == MSDA_F16) || dims->channels % 4 != 0 || !(G == 8 || G == 16) ||
      !fused_levels_points(dims))
    return fail(MSDA_E_UNSUPPORTED, "%s: no fused kernel for dtype=%d D=%d L=%d P=%d", who, dtype, dims->channels,
                dims->num_levels, dims->num_point);
  if (int e = check_ref_dim(ref_dim)) return e;
  const bool ref_grad = grad_reference_points != nullptr;
  // the size of the gradient's partials depends on ref_levels: check it before sizing the workspace
  if (ref_grad)
    if (int e = check_ref_broadcast(dims, ref_batch, ref_levels, ref_dim)) return e;
  const size_t need = fused_workspace_bytes(dims, dtype, ref_levels, ref_dim, ref_grad);
  if (need > 0 && (!workspace || workspace_bytes < need || !aligned(workspace, 16)))
    return fail(MSDA_E_WORKSPACE, "%s: workspace of %zu bytes (16-byte aligned) required", who, need);
  Params p;
  fill_params(p, dims, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits);
  p.grad_out = grad_out; p.grad_loc = grad_sampling_offsets; p.grad_aw = grad_attn_logits;
  if (int e = fused_ref_params(p, dims, reference_points, ref_batch, ref_levels, ref_dim, offsets_row_stride, logits_row_stride))
    return e;
  // a 16-bit grad_value needs only its element size: the convert that writes it picks its stores from the alignment
  if (!aligned(value, 16) || !aligned(grad_out, 16) || !aligned(backward_accum(dtype, grad_value, workspace), 16) ||
      !aligned(grad_value, elem_size(dtype)) || !aligned(sampling_offsets, 8) || !aligned(grad_sampling_offsets, 8) ||
      (ref_grad && !aligned(grad_reference_points, 4)))
    return fail(MSDA_E_ALIGN, "%s: misaligned pointer", who);
  if (ref_grad) p.ref_partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + ref_partial_offset(dims, dtype));
  const cudaStream_t s = (cudaStream_t)stream;
  if (int rc = backward_body(who, dims, dtype, p, true, grad_value, workspace, s, [&](int*) {
        return fused_launched(launch_backward_fused(p, dtype, G, s), who, G);
      }))
    return rc;
  if (!ref_grad) return 0;
  // every partial was written by the scatter kernel above: sum them into grad_reference_points in a fixed order
  const cudaError_t e = launch_ref_grad_reduce(p, ref_batch, ref_levels, grad_reference_points, s);
  if (e != cudaSuccess) return cuda_fail(e, "%s reference-point gradient launch", who);
  g_launches.fetch_add(1);
  return 0;
}

int msda_backward_fused(const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                        const int64_t* level_start_index, const float* reference_points, int32_t ref_batch,
                        int32_t ref_levels, const float* sampling_offsets, const float* attn_logits,
                        int64_t offsets_row_stride, int64_t logits_row_stride,
                        const void* grad_out, void* grad_value, float* grad_sampling_offsets, float* grad_attn_logits,
                        void* workspace, size_t workspace_bytes, void* stream) {
  return backward_fused_body("msda_backward_fused", dims, dtype, value, spatial_shapes, level_start_index, reference_points,
                             ref_batch, ref_levels, 2, sampling_offsets, attn_logits, offsets_row_stride, logits_row_stride,
                             grad_out, grad_value, grad_sampling_offsets, grad_attn_logits, nullptr, workspace,
                             workspace_bytes, stream);
}

int msda_backward_fused_ref(const msda_dims* dims, int dtype, const void* value, const int64_t* spatial_shapes,
                            const int64_t* level_start_index, const float* reference_points, int32_t ref_batch,
                            int32_t ref_levels, int32_t ref_dim, const float* sampling_offsets, const float* attn_logits,
                            int64_t offsets_row_stride, int64_t logits_row_stride, const void* grad_out, void* grad_value,
                            float* grad_sampling_offsets, float* grad_attn_logits, float* grad_reference_points,
                            void* workspace, size_t workspace_bytes, void* stream) {
  return backward_fused_body("msda_backward_fused_ref", dims, dtype, value, spatial_shapes, level_start_index,
                             reference_points, ref_batch, ref_levels, ref_dim, sampling_offsets, attn_logits,
                             offsets_row_stride, logits_row_stride, grad_out, grad_value, grad_sampling_offsets,
                             grad_attn_logits, grad_reference_points, workspace, workspace_bytes, stream);
}

size_t msda_backward_fused_workspace_bytes(const msda_dims* dims, int dtype, int32_t ref_batch, int32_t ref_levels,
                                           int32_t ref_dim, int32_t with_ref_grad) {
  // the partials are per batch element whether or not the reference points broadcast over the batch
  if (!dims || elem_size(dtype) == 0 || (ref_dim != 2 && ref_dim != 4) || !ref_broadcasts(dims, ref_batch, ref_levels)) return 0;
  return fused_workspace_bytes(dims, dtype, ref_levels, ref_dim, with_ref_grad != 0);
}

static size_t adapter_elem_size(int dtype) { return elem_size(dtype); }

static int dw_check(int dtype, int32_t B, int32_t n_tokens, int32_t C, int32_t H, int32_t W) {
  if (adapter_elem_size(dtype) == 0) return fail(MSDA_E_DTYPE, "adapter_dwconv: unknown dtype %d", dtype);
  if (B <= 0 || n_tokens <= 0 || C <= 0 || H <= 0 || W <= 0 || (H & 1) || (W & 1) ||
      (int64_t)n_tokens != 21ll * (H / 2) * (W / 2) || C > 1024 || (int64_t)B * n_tokens * C >= (1ll << 40))
    return fail(MSDA_E_DIMS, "adapter_dwconv: need n_tokens == 21*H*W/4 with even H, W and C <= 1024 (B=%d n=%d C=%d H=%d W=%d)",
                B, n_tokens, C, H, W);
  return 0;
}

int adapter_dwconv_forward(int dtype, const void* x, const void* weight, const void* bias, void* y, int32_t batch,
                           int32_t n_tokens, int32_t channels, int32_t H, int32_t W, void* stream) {
  if (int e = dw_check(dtype, batch, n_tokens, channels, H, W)) return e;
  if (!x || !weight || !y) return fail(MSDA_E_NULL, "adapter_dwconv_forward: NULL tensor pointer");
  DwParams p{x, weight, bias, y, batch, n_tokens, channels, H, W};
  const cudaError_t e = launch_dwconv(p, dtype, false, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "adapter_dwconv_forward launch");
  g_launches.fetch_add(1);
  return 0;
}

int adapter_dwconv_backward_input(int dtype, const void* grad_y, const void* weight, void* grad_x, int32_t batch,
                                  int32_t n_tokens, int32_t channels, int32_t H, int32_t W, void* stream) {
  if (int e = dw_check(dtype, batch, n_tokens, channels, H, W)) return e;
  if (!grad_y || !weight || !grad_x) return fail(MSDA_E_NULL, "adapter_dwconv_backward_input: NULL tensor pointer");
  DwParams p{grad_y, weight, nullptr, grad_x, batch, n_tokens, channels, H, W};
  const cudaError_t e = launch_dwconv(p, dtype, true, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "adapter_dwconv_backward_input launch");
  g_launches.fetch_add(1);
  return 0;
}

size_t adapter_dwconv_backward_weight_workspace_bytes(int dtype, int32_t batch, int32_t n_tokens, int32_t channels, int32_t H,
                                                      int32_t W) {
  if (dw_check(dtype, batch, n_tokens, channels, H, W)) return 0;
  DwParams p{nullptr, nullptr, nullptr, nullptr, batch, n_tokens, channels, H, W};
  return dwconv_wgrad_workspace_bytes(p, dtype);
}

int adapter_dwconv_backward_weight(int dtype, const void* x, const void* grad_y, void* grad_weight, void* grad_bias,
                                   int32_t batch, int32_t n_tokens, int32_t channels, int32_t H, int32_t W, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  if (int e = dw_check(dtype, batch, n_tokens, channels, H, W)) return e;
  if (!x || !grad_y || !grad_weight || !grad_bias) return fail(MSDA_E_NULL, "adapter_dwconv_backward_weight: NULL tensor pointer");
  DwParams p{x, nullptr, nullptr, nullptr, batch, n_tokens, channels, H, W};
  const size_t need = dwconv_wgrad_workspace_bytes(p, dtype);
  if (need && (!workspace || workspace_bytes < need))
    return fail(MSDA_E_WORKSPACE, "adapter_dwconv_backward_weight: workspace of %zu bytes required, got %zu", need,
                workspace ? workspace_bytes : (size_t)0);
  int launches = 0;
  const cudaError_t e = launch_dwconv_wgrad(p, dtype, grad_y, grad_weight, grad_bias, workspace, workspace_bytes, &launches,
                                            (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "adapter_dwconv_backward_weight launch");
  g_launches.fetch_add(launches);
  return 0;
}

static int ln_check(const char* who, int in_dtype, int out_dtype, int64_t rows, int32_t C) {
  const bool combo = (in_dtype == MSDA_F32 && (out_dtype == MSDA_F32 || out_dtype == MSDA_BF16 || out_dtype == MSDA_F16)) ||
                     (in_dtype == MSDA_BF16 && out_dtype == MSDA_BF16) || (in_dtype == MSDA_F16 && out_dtype == MSDA_F16);
  if (!combo)
    return fail(MSDA_E_DTYPE, "%s: (x, y) dtypes must be (f32, f32), (f32, bf16), (bf16, bf16), (f32, f16) or (f16, f16), got (%d, %d)", who,
                in_dtype, out_dtype);
  if (rows <= 0 || C <= 0 || rows * (int64_t)C >= (1ll << 40)) return fail(MSDA_E_DIMS, "%s: bad dims rows=%lld C=%d", who, (long long)rows, C);
  if (!layernorm_supported(C)) return fail(MSDA_E_UNSUPPORTED, "%s: C=%d needs C %% 4 == 0 and C <= 1024", who, C);
  return 0;
}

static bool ln_misaligned(const void* p, int dtype) { return (reinterpret_cast<uintptr_t>(p) & (4 * adapter_elem_size(dtype) - 1)) != 0; }

int adapter_layernorm_forward(int in_dtype, int out_dtype, const void* x, const void* gamma, const void* beta, void* y,
                              float* mean, float* rstd, int64_t rows, int32_t channels, float eps, void* stream) {
  if (int e = ln_check("adapter_layernorm_forward", in_dtype, out_dtype, rows, channels)) return e;
  if (!x || !gamma || !y || !mean || !rstd) return fail(MSDA_E_NULL, "adapter_layernorm_forward: NULL tensor pointer");
  if (ln_misaligned(x, in_dtype) || ln_misaligned(y, out_dtype) || ln_misaligned(gamma, MSDA_F32) || (beta && ln_misaligned(beta, MSDA_F32)))
    return fail(MSDA_E_ALIGN, "adapter_layernorm_forward: x, y, gamma, beta must be aligned to 4 elements");
  LnParams p{x, gamma, beta, y, mean, rstd, nullptr, nullptr, nullptr, (long long)rows, channels, eps};
  const cudaError_t e = launch_layernorm_forward(p, in_dtype, out_dtype, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "adapter_layernorm_forward launch");
  g_launches.fetch_add(1);
  return 0;
}

size_t adapter_layernorm_backward_workspace_bytes(int64_t rows, int32_t channels) {
  if (rows <= 0 || !layernorm_supported(channels)) return 0;
  return layernorm_backward_workspace_bytes((long long)rows, channels);
}

int adapter_layernorm_backward(int in_dtype, int out_dtype, const void* grad_y, const void* x, const void* gamma,
                               const float* mean, const float* rstd, const void* grad_residual, void* grad_x,
                               float* grad_gamma, float* grad_beta, int64_t rows, int32_t channels, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (int e = ln_check("adapter_layernorm_backward", in_dtype, out_dtype, rows, channels)) return e;
  if (!grad_y || !x || !gamma || !mean || !rstd || !grad_x || !grad_gamma || !grad_beta)
    return fail(MSDA_E_NULL, "adapter_layernorm_backward: NULL tensor pointer");
  if (ln_misaligned(x, in_dtype) || ln_misaligned(grad_x, in_dtype) || ln_misaligned(grad_y, out_dtype) || ln_misaligned(gamma, MSDA_F32) ||
      (grad_residual && ln_misaligned(grad_residual, in_dtype)))
    return fail(MSDA_E_ALIGN, "adapter_layernorm_backward: x, grad_x, grad_y, grad_residual, gamma must be aligned to 4 elements");
  const size_t need = layernorm_backward_workspace_bytes((long long)rows, channels);
  if (!workspace || workspace_bytes < need || (reinterpret_cast<uintptr_t>(workspace) & 15))
    return fail(MSDA_E_WORKSPACE, "adapter_layernorm_backward: 16-byte aligned workspace of %zu bytes required, got %zu", need,
                workspace ? workspace_bytes : (size_t)0);
  LnParams p{x, gamma, nullptr, nullptr, const_cast<float*>(mean), const_cast<float*>(rstd), grad_y, grad_x,
             reinterpret_cast<float*>(workspace), (long long)rows, channels, 0.f, grad_residual};
  const cudaError_t e = launch_layernorm_backward(p, in_dtype, out_dtype, grad_gamma, grad_beta, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "adapter_layernorm_backward launch");
  g_launches.fetch_add(2);
  return 0;
}

int adapter_residual_add(int branch_dtype, const float* residual, const void* branch, float* out, int64_t n, void* stream) {
  if (branch_dtype != MSDA_F32 && branch_dtype != MSDA_BF16 && branch_dtype != MSDA_F16)
    return fail(MSDA_E_DTYPE, "adapter_residual_add: branch must be f32, bf16 or f16, got %d", branch_dtype);
  if (n <= 0 || n >= (1ll << 40)) return fail(MSDA_E_DIMS, "adapter_residual_add: bad element count %lld", (long long)n);
  if (n % 8) return fail(MSDA_E_UNSUPPORTED, "adapter_residual_add: element count %lld is not a multiple of 8", (long long)n);
  if (!residual || !branch || !out) return fail(MSDA_E_NULL, "adapter_residual_add: NULL tensor pointer");
  if ((reinterpret_cast<uintptr_t>(residual) | reinterpret_cast<uintptr_t>(branch) | reinterpret_cast<uintptr_t>(out)) & 15)
    return fail(MSDA_E_ALIGN, "adapter_residual_add: pointers must be 16-byte aligned");
  const cudaError_t e = launch_residual_add(branch_dtype, residual, branch, out, (long long)n, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "adapter_residual_add launch");
  g_launches.fetch_add(1);
  return 0;
}

size_t adapter_colsum_workspace_bytes(int dtype, int64_t rows, int32_t channels) {
  if (rows <= 0 || channels <= 0) return 0;
  return colsum_workspace_bytes(dtype, (long long)rows, channels);
}

int adapter_colsum(int dtype, const void* x, int64_t rows, int32_t channels, float* out, void* workspace,
                   size_t workspace_bytes, void* stream) {
  if (adapter_elem_size(dtype) == 0) return fail(MSDA_E_DTYPE, "adapter_colsum: unknown dtype %d", dtype);
  if (rows <= 0 || channels <= 0 || rows * (int64_t)channels >= (1ll << 40))
    return fail(MSDA_E_DIMS, "adapter_colsum: bad dims rows=%lld C=%d", (long long)rows, channels);
  if (!colsum_supported(dtype, channels))
    return fail(MSDA_E_UNSUPPORTED, "adapter_colsum: needs f32 (C %% 4 == 0, C <= 1024) or bf16 / f16 (C %% 8 == 0, C <= 2048), got dtype %d C=%d",
                dtype, channels);
  if (!x || !out) return fail(MSDA_E_NULL, "adapter_colsum: NULL tensor pointer");
  if (reinterpret_cast<uintptr_t>(x) & 15) return fail(MSDA_E_ALIGN, "adapter_colsum: x must be 16-byte aligned");
  const size_t need = colsum_workspace_bytes(dtype, (long long)rows, channels);
  if (!workspace || workspace_bytes < need)
    return fail(MSDA_E_WORKSPACE, "adapter_colsum: workspace of %zu bytes required, got %zu", need, workspace ? workspace_bytes : (size_t)0);
  const cudaError_t e = launch_colsum(dtype, x, (long long)rows, channels, out, reinterpret_cast<float*>(workspace), (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "adapter_colsum launch");
  g_launches.fetch_add(2);
  return 0;
}

int msda_debug_point_index(const msda_dims* dims, const int64_t* spatial_shapes,
                           const int64_t* level_start_index, const float* sampling_loc, int32_t* idx,
                           void* stream) {
  if (int e = check_dims(dims, MSDA_F32)) return e;
  if (!spatial_shapes || !level_start_index || !sampling_loc || !idx)
    return fail(MSDA_E_NULL, "msda_debug_point_index: NULL pointer");
  const size_t total = (size_t)dims->batch * dims->num_query * dims->num_heads * dims->num_levels * dims->num_point;
  size_t blocks = (total + 255) / 256;
  if (blocks > 148u * 8u) blocks = 148u * 8u;
  msda_debug_index_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      spatial_shapes, level_start_index, sampling_loc, idx, dims->batch, dims->num_heads, dims->channels,
      dims->num_levels, dims->num_query, dims->num_point);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "msda_debug_point_index launch");
  g_launches.fetch_add(1);
  return 0;
}

}  // extern "C"
