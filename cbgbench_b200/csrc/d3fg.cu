// D3FG sampler (repo/models/diffusion/difffg.py:174-246): one reverse step per C-ABI call = step-init (composed ligand
// FG rows of x / o / h) -> IPA encoder (ipa.cu) -> d3fg_reverse_kernel (position, rotation and FG-type updates in one
// launch).  Algebra and the multinomial definition: include/cbg_b200.h and DESIGN.md section 13.
#include <math.h>
#include "../../include/cbg_b200.h"
#include "cbg_kernels.cuh"

namespace {

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

struct D3fgWs {
  char* ipa;
  float *h, *eps, *o_pred, *r, *logits;
};

D3fgWs carve(void* base, long long n, int H, int K) {
  D3fgWs w;
  char* p = (char*)base;
  w.ipa = p; p += align256((size_t)cbg_ipa_workspace_bytes(n, H));
  w.h = (float*)p; p += align256((size_t)n * H * 4);
  w.eps = (float*)p; p += align256((size_t)n * 3 * 4);
  w.o_pred = (float*)p; p += align256((size_t)n * 3 * 4);
  w.r = (float*)p; p += align256((size_t)n * 9 * 4);
  w.logits = (float*)p; p += align256((size_t)n * K * 4);
  return w;
}

// ---- step-init: one CTA per composed row ---------------------------------------------------------------------------
__global__ void __launch_bounds__(64) d3fg_step_init_kernel(cbg_d3fg_plan p, const float* __restrict__ x_t,
                                                           const float* __restrict__ c_t, const float* __restrict__ o_t,
                                                           float* __restrict__ h) {
  __shared__ int s_a, s_v;
  const int i = blockIdx.x, H = p.hidden, K = p.num_classes;
  if (threadIdx.x == 0) {
    int lo = 0, hi = p.n_lig;                         // lig_node is increasing: lower bound of i
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (p.lig_node[mid] < i) lo = mid + 1; else hi = mid; }
    const int a = (lo < p.n_lig && p.lig_node[lo] == i) ? lo : -1;
    int v = 0;
    if (a >= 0) {
      float best = c_t[(size_t)a * K];
      for (int c = 1; c < K; ++c) { const float q = c_t[(size_t)a * K + c]; if (q > best) { best = q; v = c; } }
#pragma unroll
      for (int d = 0; d < 3; ++d) { p.x[3 * i + d] = x_t[3 * a + d]; p.o[3 * i + d] = o_t[3 * a + d]; }
    }
    s_a = a; s_v = v;
  }
  __syncthreads();
  const int a = s_a;
  float4* dst = reinterpret_cast<float4*>(h + (size_t)i * H);
  if (a < 0) {
    const float4* src = reinterpret_cast<const float4*>(p.h_static + (size_t)i * H);
    for (int f = threadIdx.x; f < H / 4; f += blockDim.x) dst[f] = src[f];
    return;
  }
  const float4* w = reinterpret_cast<const float4*>(p.fg_wt + (size_t)s_v * H);
  const float4* b = reinterpret_cast<const float4*>(p.fg_b);
  const float4* l = reinterpret_cast<const float4*>(p.lig_bias);
  for (int f = threadIdx.x; f < H / 4; f += blockDim.x) {
    const float4 wv = w[f], bv = b[f], lv = l[f];
    dst[f] = make_float4(__fadd_rn(__fadd_rn(wv.x, bv.x), lv.x), __fadd_rn(__fadd_rn(wv.y, bv.y), lv.y),
                         __fadd_rn(__fadd_rn(wv.z, bv.z), lv.z), __fadd_rn(__fadd_rn(wv.w, bv.w), lv.w));
  }
}

// ---- reverse step: one warp per FG, lane = class ---------------------------------------------------------------------
struct D3fgRevArgs {
  const float* eps; const float* logits; const float* o_pred;
  const int* row;                 // row of FG a in eps / logits / o_pred (nullptr: a)
  const float* x_t; const float* c_t; const float* o_t; const unsigned char* gen;
  const float* pos_noise; const float* rot_dir; const float* rot_bin_u; const float* rot_in_u; const float* rot_gauss;
  const float* type_u;
  const double* cdf; const float* X; int n_bins;
  cbg_d3fg_coef c;
  int n, K;
  float* x_next; float* c_next; float* o_next; long long* v_next; int* bin_out;
  float* eps_out; float* logits_out; float* o_pred_out;
};

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v = fmaxf(v, __shfl_xor_sync(CBG_FULL, v, m));
  return v;
}
// index of the largest value, first index on ties (torch.argmax)
__device__ __forceinline__ int warp_argmax(float v, int idx) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    const float ov = __shfl_xor_sync(CBG_FULL, v, m);
    const int oi = __shfl_xor_sync(CBG_FULL, idx, m);
    if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
  return idx;
}
__device__ __forceinline__ float log_add_exp(float a, float b) {
  const float m = fmaxf(a, b);
  return m + logf(expf(a - m) + expf(b - m));
}
__device__ __forceinline__ void mat3_mul(const float* A, const float* B, float* C) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c)
      C[3 * r + c] = __fadd_rn(__fadd_rn(__fmul_rn(A[3 * r], B[c]), __fmul_rn(A[3 * r + 1], B[3 + c])), __fmul_rn(A[3 * r + 2], B[6 + c]));
}
// so3vec_to_rotation (so3.py:33-57): I + b S + c S^2 with the reference's 1e-8 guards
__device__ __forceinline__ void so3_exp(float wx, float wy, float wz, float* R) {
  const float S[9] = {0.f, wz, -wy, -wz, 0.f, wx, wy, -wx, 0.f};
  const float xn = sqrtf(wx * wx + wy * wy + wz * wz);
  const float b = (sinf(xn) + 1e-8f) / (xn + 1e-8f);
  const float c = (1.f - cosf(xn) + 1e-8f) / (xn * xn + 2e-8f);
  float S2[9];
  mat3_mul(S, S, S2);
#pragma unroll
  for (int e = 0; e < 9; ++e) R[e] = ((e % 4 == 0) ? 1.f : 0.f) + b * S[e] + c * S2[e];
}
// rotation_to_so3vec (so3.py:10-31, 60-63), no-grad branch: min_cos = -1
__device__ __forceinline__ void so3_log(const float* R, float* w) {
  const float tr = R[0] + R[4] + R[8];
  const float cos_t = fmaxf((tr - 1.f) * 0.5f, -1.f);
  const float sin_t = sqrtf(1.f - cos_t * cos_t);
  const float theta = acosf(cos_t);
  const float coef = (theta + 1e-8f) / (2.f * sin_t + 2e-8f);
  w[0] = coef * (R[5] - R[7]); w[1] = coef * (R[6] - R[2]); w[2] = coef * (R[1] - R[3]);
}

__global__ void __launch_bounds__(128) d3fg_reverse_kernel(D3fgRevArgs p) {
  const int a = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (a >= p.n) return;                                       // whole warp
  const int row = p.row ? p.row[a] : a;
  const int K = p.K;
  const bool g = p.gen[a] != 0;
  const bool act = lane < K;
  // ---- FG type: TypeVPScheduler.backward_remove_noise (diffusion_scheduler.py:367-378, 407-441)
  const float lg = act ? p.logits[(size_t)row * K + lane] : -INFINITY;
  const float mx = warp_max(lg);
  const float lse = mx + logf(warp_sum(act ? expf(lg - mx) : 0.f));
  const float ctv = act ? p.c_t[(size_t)a * K + lane] : -INFINITY;
  const int arg_ct = warp_argmax(ctv, lane);
  const float logK = logf((float)K);
  const float A = log_add_exp((lg - lse) + p.c.log_alphas_cumprod_prev, p.c.log_one_minus_alphas_cumprod_prev - logK);
  const float B = log_add_exp(logf(ctv + 1e-8f) + p.c.log_alpha, p.c.log_one_minus_alpha - logK);
  const float un = act ? A + B : -INFINITY;
  const float m2 = warp_max(un);
  const float lse2 = m2 + logf(warp_sum(act ? expf(un - m2) : 0.f));
  float score = -INFINITY;
  if (act) {
    const float u = p.type_u[(size_t)a * K + lane];
    score = -logf(-logf(u + 1e-30f) + 1e-30f) + (un - lse2);
  }
  const int v = g ? warp_argmax(score, lane) : arg_ct;
  if (act) {
    p.c_next[(size_t)a * K + lane] = lane == v ? 1.f : 0.f;
    if (p.logits_out) p.logits_out[(size_t)a * K + lane] = lg;
  }
  // ---- position: CTNVPScheduler.backward_remove_noise, type='score' (:144-165)
  if (lane < 3) {
    const float xt = p.x_t[3 * a + lane], e = p.eps[3 * row + lane];
    const float sigma = __fsqrt_rn(__fsub_rn(1.f, p.c.alpha_cumprod));
    const float sc = -__fdiv_rn(e, sigma);
    float xs = __fdiv_rn(__fadd_rn(xt, __fmul_rn(p.c.beta, sc)), __fsqrt_rn(__fsub_rn(1.f, p.c.beta)));
    xs = __fadd_rn(xs, __fmul_rn(__fmul_rn(p.c.pos_nonzero, __fsqrt_rn(p.c.beta)), p.pos_noise[3 * a + lane]));
    p.x_next[3 * a + lane] = g ? xs : xt;
    if (p.eps_out) p.eps_out[3 * a + lane] = e;
  }
  if (lane != 0) return;
  p.v_next[a] = v;
  // ---- rotation: RotVPScheduler.backward_remove_noise (:558-574), random_normal_so3 / ApproxAngularDistribution.sample
  const float dx = p.rot_dir[3 * a], dy = p.rot_dir[3 * a + 1], dz = p.rot_dir[3 * a + 2];
  const float nrm = fmaxf(sqrtf(dx * dx + dy * dy + dz * dz), 1e-12f);          // F.normalize
  const double* cdf = p.cdf + (size_t)p.c.rot_row * p.n_bins;
  const double target = (double)p.rot_bin_u[a] * cdf[p.n_bins - 1];
  int lo = 0, hi = p.n_bins - 1;                 // first bin with cdf > target (the last bin if none)
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (cdf[mid] > target) hi = mid; else lo = mid + 1; }
  if (p.bin_out) p.bin_out[a] = lo;
  float theta;
  const float sd = p.c.rot_stddev;
  if (p.c.rot_approx) {
    theta = fmodf(fabsf(__fadd_rn(__fmul_rn(sd, 2.f), __fmul_rn(p.rot_gauss[a], sd))), 3.14159274101257324f);
  } else {
    const float* X = p.X + (size_t)p.c.rot_row * (p.n_bins + 1);
    theta = __fadd_rn(X[lo], __fmul_rn(p.rot_in_u[a], __fsub_rn(X[lo + 1], X[lo])));
  }
  float ex = 0.f, ey = 0.f, ez = 0.f;
  if (p.c.rot_nonzero != 0.f) { ex = __fmul_rn(dx / nrm, theta); ey = __fmul_rn(dy / nrm, theta); ez = __fmul_rn(dz / nrm, theta); }
  const float opx = p.o_pred[3 * row], opy = p.o_pred[3 * row + 1], opz = p.o_pred[3 * row + 2];
  float E[9], Rp[9], Rn[9], w[3];
  so3_exp(ex, ey, ez, E);
  so3_exp(opx, opy, opz, Rp);
  mat3_mul(E, Rp, Rn);
  so3_log(Rn, w);
  p.o_next[3 * a] = g ? w[0] : p.o_t[3 * a];
  p.o_next[3 * a + 1] = g ? w[1] : p.o_t[3 * a + 1];
  p.o_next[3 * a + 2] = g ? w[2] : p.o_t[3 * a + 2];
  if (p.o_pred_out) { p.o_pred_out[3 * a] = opx; p.o_pred_out[3 * a + 1] = opy; p.o_pred_out[3 * a + 2] = opz; }
}

int launch_reverse(const D3fgRevArgs& r, cudaStream_t st) {
  if (r.n <= 0) return 0;
  CBG_PROF_BEGIN(CBG_K_REVERSE, st);
  d3fg_reverse_kernel<<<(r.n + 3) / 4, 128, 0, st>>>(r);
  CBG_LAUNCHED(CBG_K_REVERSE, st);
  return 0;
}

bool bad_coef(const cbg_d3fg_coef* c, const double* cdf, const float* X, int n_bins) {
  if (!c || !cdf || !X) { cbg_set_error("null coef / rot_cdf / rot_x"); return true; }
  if (n_bins < 1 || c->rot_row < 0) { cbg_set_error("n_bins=%d rot_row=%d", n_bins, c->rot_row); return true; }
  return false;
}

}  // namespace

extern "C" {

int64_t cbg_d3fg_workspace_bytes(int64_t n_nodes, int32_t hidden, int32_t num_classes) {
  const size_t n = (size_t)n_nodes;
  return (int64_t)(align256((size_t)cbg_ipa_workspace_bytes(n_nodes, hidden)) + align256(n * hidden * 4) +
                   2 * align256(n * 3 * 4) + align256(n * 9 * 4) + align256(n * num_classes * 4));
}

int32_t cbg_d3fg_step_f32(const cbg_d3fg_plan* plan, const cbg_d3fg_coef* coef, const float* x_t, const float* c_t,
                          const float* o_t, const float* pos_noise, const float* rot_dir, const float* rot_bin_u,
                          const float* rot_in_u, const float* rot_gauss, const float* type_u, float* x_next, float* c_next,
                          float* o_next, int64_t* v_next, float* eps_pos_out, float* logits_out, float* o_pred_out,
                          void* stream) {
  if (!plan) { cbg_set_error("null plan"); return 1; }
  const int H = plan->hidden, K = plan->num_classes;
  const long long N = plan->n_nodes;
  if (H != 128 && H != 256) { cbg_set_error("cbg_d3fg_step_f32: hidden=%d (128 or 256)", H); return 1; }
  if (K < 1 || K > CBG_IPA_MAXCLS) { cbg_set_error("num_classes=%d outside [1,%d]", K, CBG_IPA_MAXCLS); return 1; }
  if (N <= 0 || N > 0x7fffffffLL / (5 * 256) || plan->n_lig < 0 || plan->n_lig > N) { cbg_set_error("n_nodes=%lld n_lig=%d out of range", N, plan->n_lig); return 1; }
  if (plan->num_blocks < 1 || plan->num_sublayers < 0 || plan->k < 1 || plan->k > CBG_KMAX) { cbg_set_error("num_blocks / num_sublayers / k"); return 1; }
  if (bad_coef(coef, plan->rot_cdf, plan->rot_x, plan->n_bins)) return 1;
  if (!plan->workspace || plan->workspace_bytes < cbg_d3fg_workspace_bytes(N, H, K)) { cbg_set_error("workspace too small"); return 1; }
  if (((uintptr_t)plan->workspace & 255) != 0) { cbg_set_error("workspace must be 256-byte aligned"); return 1; }
  if (!plan->x || !plan->o || !plan->h_static || !plan->fg_wt || !plan->fg_b || !plan->lig_bias) { cbg_set_error("null plan array"); return 1; }
  cudaStream_t st = (cudaStream_t)stream;
  const D3fgWs w = carve(plan->workspace, N, H, K);
  CBG_PROF_BEGIN(CBG_K_STEP_INIT, st);
  d3fg_step_init_kernel<<<(unsigned)N, 64, 0, st>>>(*plan, x_t, c_t, o_t, w.h);
  CBG_LAUNCHED(CBG_K_STEP_INIT, st);
  if (int rc = cbg_launch_ipa_forward(plan->blob, H, plan->num_sublayers, plan->num_blocks, K, plan->x, plan->o, w.h,
                                      plan->graph_ptr, plan->n_graphs, plan->max_graph_nodes, plan->lig_flag, plan->gen_flag,
                                      (int)N, plan->k, w.eps, w.h, w.o_pred, w.r, w.logits, w.ipa, st)) return rc;
  D3fgRevArgs r{};
  r.eps = w.eps; r.logits = w.logits; r.o_pred = w.o_pred; r.row = plan->lig_node;
  r.x_t = x_t; r.c_t = c_t; r.o_t = o_t; r.gen = plan->gen_lig;
  r.pos_noise = pos_noise; r.rot_dir = rot_dir; r.rot_bin_u = rot_bin_u; r.rot_in_u = rot_in_u; r.rot_gauss = rot_gauss;
  r.type_u = type_u; r.cdf = plan->rot_cdf; r.X = plan->rot_x; r.n_bins = plan->n_bins; r.c = *coef;
  r.n = plan->n_lig; r.K = K; r.x_next = x_next; r.c_next = c_next; r.o_next = o_next; r.v_next = (long long*)v_next;
  r.eps_out = eps_pos_out; r.logits_out = logits_out; r.o_pred_out = o_pred_out;
  return launch_reverse(r, st);
}

int32_t cbg_d3fg_reverse_f32(const cbg_d3fg_coef* coef, const double* rot_cdf, const float* rot_x, int32_t n_bins,
                             const float* eps, const float* logits, const float* o_pred, const float* x_t, const float* c_t,
                             const float* o_t, const uint8_t* gen, const float* pos_noise, const float* rot_dir,
                             const float* rot_bin_u, const float* rot_in_u, const float* rot_gauss, const float* type_u,
                             int32_t n, int32_t num_classes, float* x_next, float* c_next, float* o_next, int64_t* v_next,
                             int32_t* bin_out, void* stream) {
  if (bad_coef(coef, rot_cdf, rot_x, n_bins)) return 1;
  if (num_classes < 1 || num_classes > CBG_IPA_MAXCLS) { cbg_set_error("num_classes=%d outside [1,%d]", num_classes, CBG_IPA_MAXCLS); return 1; }
  if (n < 0) { cbg_set_error("n=%d", n); return 1; }
  D3fgRevArgs r{};
  r.eps = eps; r.logits = logits; r.o_pred = o_pred; r.row = nullptr;
  r.x_t = x_t; r.c_t = c_t; r.o_t = o_t; r.gen = gen;
  r.pos_noise = pos_noise; r.rot_dir = rot_dir; r.rot_bin_u = rot_bin_u; r.rot_in_u = rot_in_u; r.rot_gauss = rot_gauss;
  r.type_u = type_u; r.cdf = rot_cdf; r.X = rot_x; r.n_bins = n_bins; r.c = *coef;
  r.n = n; r.K = num_classes; r.x_next = x_next; r.c_next = c_next; r.o_next = o_next; r.v_next = (long long*)v_next;
  r.bin_out = bin_out;
  return launch_reverse(r, (cudaStream_t)stream);
}

}  // extern "C"
