// SURVEY.md section 8 row f4: the D3FG encoder, `IPATransformer` (repo/modules/e3nn/itatransformer.py:14-145) - an X2H-only
// stack (InvAttentionLayer :147-188 = num_x2h x X2HAttention, coordinates never move) at hidden width H = 128 or 256
// (the shipped config configs/denovo/train/d3fg_fg.yml:5 uses 256), followed by the rotation / translation / type heads
// (:54-66, :127-145) and the SO(3) update of the orientation vectors (repo/models/utils/so3.py, geometry.py:232-250).
//
// Same algebra as the 128-wide denoiser (DESIGN.md section 3): the first Linear of the edge MLPs is split into node planes
// (Pj, Pi), a type-dependent RBF mat-vec and a type bias, [E, 2H + 84] is never formed, the key bias cancels in the
// softmax.  The kernels here are width-generic fp32 SIMT kernels (one CTA per destination node, thread = feature): this
// row is built to the parity bar; the tcgen05 tile kernels (x2h_tc.cu) are specialised for H = 128 (TMEM budget).
// Graph construction (kNN) and the edge gate are the hot path's own kernels (graph.cu).
#include <math.h>
#include "cbg_kernels.cuh"

namespace {

// ---- blob layout (floats): [global block of cbg_layout.h | head block | num_sublayers x layer block] ----------------
enum IpaHeadField { IH_ROT_W0T, IH_ROT_B0, IH_ROT_W1T, IH_ROT_B1, IH_ROT_W2, IH_ROT_B2,
                    IH_CRD_W0T, IH_CRD_B0, IH_CRD_W1T, IH_CRD_B1, IH_CRD_W2, IH_CRD_B2,
                    IH_CLS_W0T, IH_CLS_B0, IH_CLS_W1, IH_CLS_B1, IH_COUNT };
enum IpaLayerField { IL_NODE_WT, IL_NODE_B, IL_Q_LN, IL_Q_W1T, IL_Q_B1,
                     IL_K_WRF, IL_K_C, IL_K_LN, IL_K_W1T,
                     IL_V_WRF, IL_V_C, IL_V_LN, IL_V_W1T, IL_V_B1, IL_RBF, IL_COUNT };

__host__ __device__ inline long long head_size(int H, int f) {
  switch (f) {
    case IH_ROT_W0T: case IH_CRD_W0T: return (long long)H * 2 * H;      // [k = H][n = 2H]
    case IH_ROT_B0: case IH_CRD_B0: return 2 * H;
    case IH_ROT_W1T: case IH_CRD_W1T: return (long long)2 * H * H;      // [k = 2H][n = H]
    case IH_ROT_B1: case IH_CRD_B1: return H;
    case IH_ROT_W2: case IH_CRD_W2: return 4 * H;                       // [3 (+1 zero)][H]
    case IH_ROT_B2: case IH_CRD_B2: return 4;
    case IH_CLS_W0T: return (long long)H * H;
    case IH_CLS_B0: return H;
    case IH_CLS_W1: return CBG_IPA_MAXCLS * H;
    case IH_CLS_B1: return CBG_IPA_MAXCLS;
  }
  return 0;
}
__host__ __device__ inline long long layer_size(int H, int f) {
  switch (f) {
    case IL_NODE_WT: return (long long)H * 5 * H;                       // [k = H][n = 5H]: Pj_k | Pj_v | Pi_k | Pi_v | q hidden
    case IL_NODE_B: return 5 * H;
    case IL_Q_LN: case IL_K_LN: case IL_V_LN: return 2 * H;
    case IL_Q_W1T: case IL_K_W1T: case IL_V_W1T: return (long long)H * H;   // [k][n]
    case IL_Q_B1: case IL_V_B1: return H;
    case IL_K_WRF: case IL_V_WRF: return (long long)CBG_NTYPE * CBG_NRBF * H;
    case IL_K_C: case IL_V_C: return CBG_NTYPE * H;
    case IL_RBF: return 32;
  }
  return 0;
}
__host__ __device__ inline long long head_off(int H, int f) { long long o = 0; for (int i = 0; i < f; ++i) o += head_size(H, i); return o; }
__host__ __device__ inline long long layer_off(int H, int f) { long long o = 0; for (int i = 0; i < f; ++i) o += layer_size(H, i); return o; }

// ---- C[N, M] = A[N, K] Wt[K, M] + bias[M]: 64 x 64 tiles, 256 threads, 4 x 4 outputs per thread -----------------------
__global__ void __launch_bounds__(256) ipa_linear_kernel(const float* __restrict__ A, int lda, const float* __restrict__ Wt,
                                                         int ldw, const float* __restrict__ bias, float* __restrict__ C,
                                                         int ldc, int N, int K, int M) {
  __shared__ float sa[16][64 + 4];      // [k][row]
  __shared__ float sw[16][64 + 4];      // [k][col]
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int row0 = blockIdx.y * 64, col0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int e = threadIdx.x; e < 64 * 16; e += 256) {
      const int r = e >> 4, kk = e & 15;
      sa[kk][r] = (row0 + r < N) ? A[(size_t)(row0 + r) * lda + k0 + kk] : 0.f;
      const int c = e & 63, k2 = e >> 6;
      sw[k2][c] = (col0 + c < M) ? Wt[(size_t)(k0 + k2) * ldw + col0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sa[kk][ty * 4 + i]; w[i] = sw[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = row0 + ty * 4 + i;
    if (r >= N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = col0 + tx * 4 + j;
      if (c < M) C[(size_t)r * ldc + c] = acc[i][j] + (bias ? bias[c] : 0.f);
    }
  }
}

// block-wide sum of one value per thread (blockDim.x = H, a multiple of 32); every thread gets the result
template <int H>
__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(CBG_FULL, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < H / 32; ++w) s += red[w];
  return s;
}

// rows: y = relu(LayerNorm(x)) in place (the hidden layer of the query MLP, common.py:151-171); one CTA per row
template <int H>
__global__ void __launch_bounds__(H) ipa_ln_relu_kernel(float* __restrict__ x, int ld, const float* __restrict__ ln, int N) {
  __shared__ float red[H / 32];
  const int r = blockIdx.x, f = threadIdx.x;
  if (r >= N) return;
  const float v = x[(size_t)r * ld + f];
  const float mean = block_sum<H>(v, red) * (1.f / H);
  const float d = v - mean;
  const float var = block_sum<H>(d * d, red) * (1.f / H);
  const float y = d * (1.f / sqrtf(var + 1e-5f)) * ln[f] + ln[H + f];
  x[(size_t)r * ld + f] = fmaxf(y, 0.f);
}

// ---- X2HAttention for one destination node per CTA (x2h_attention.py:43-97), thread = feature --------------------------
// planes: [N][5H] = Pj_k | Pj_v | Pi_k | Pi_v | (q hidden, unused here); q: [N][H] (already scaled by 1/sqrt(H/16)).
template <int H>
__global__ void __launch_bounds__(H) ipa_x2h_kernel(const float4* __restrict__ x4, const int* __restrict__ nbr,
                                                    const float* __restrict__ ew, const float* __restrict__ planes,
                                                    const float* __restrict__ q, const float* __restrict__ L,
                                                    float* __restrict__ h, int N) {
  constexpr int DH = H / CBG_HEADS;
  extern __shared__ __align__(16) float sm[];
  float* s_a = sm;                              // [32 edges][H]: pre -> activations
  float* s_g = s_a + 32 * H;                    // [20][32]
  float* s_lg = s_g + CBG_NRBF * 32;            // [32 edges][16 heads]: logits -> alpha * e_w
  float* s_stat = s_lg + 32 * CBG_HEADS;        // mean[32] | rstd[32]
  int* s_j = reinterpret_cast<int*>(s_stat + 64);
  int* s_t = s_j + 32;
  float* s_ew = reinterpret_cast<float*>(s_t + 32);
  const int i = blockIdx.x, f = threadIdx.x, warp = f >> 5, lane = f & 31;
  if (i >= N) return;
  const float* rbf = L + layer_off(H, IL_RBF);
  if (warp == 0) {      // edge setup: lane = neighbour slot (padded slots: j = i, e_w = 0, masked in the softmax)
    const float4 xi = x4[i];
    const int jn = nbr[(size_t)i * CBG_KMAX + lane];
    const int j = jn >= 0 ? jn : i;
    const float4 xj = x4[j];
    const float rx = xi.x - xj.x, ry = xi.y - xj.y, rz = xi.z - xj.z;
    const float d = sqrtf(rx * rx + ry * ry + rz * rz);
    const float coeff = rbf[20];
    for (int m = 0; m < CBG_NRBF; ++m) { const float u = d - rbf[m]; s_g[m * 32 + lane] = expf(coeff * u * u); }
    s_j[lane] = jn;
    // itatransformer.py:101-112: 0 lig->lig, 1 lig src / prot dst, 2 prot src / lig dst, 3 prot->prot
    s_t[lane] = ((node_flags(xj) & 1) ? 0 : 2) + ((node_flags(xi) & 1) ? 0 : 1);
    s_ew[lane] = jn >= 0 ? ew[(size_t)i * CBG_KMAX + lane] : 0.f;
  }
  __syncthreads();
  const float qf = q[(size_t)i * H + f];
  float out_acc = 0.f;
  for (int which = 0; which < 2; ++which) {          // 0: key MLP -> attention weights, 1: value MLP -> aggregation
    const float* wrf = L + layer_off(H, which ? IL_V_WRF : IL_K_WRF);
    const float* cc = L + layer_off(H, which ? IL_V_C : IL_K_C);
    const float* ln = L + layer_off(H, which ? IL_V_LN : IL_K_LN);
    const float* w1t = L + layer_off(H, which ? IL_V_W1T : IL_K_W1T);
    const float pi = planes[(size_t)i * 5 * H + (2 + which) * H + f];
    // first Linear: pre[e][f] = Pi[i] + Pj[j_e] + c[t_e] + Wrf[t_e] g_e
    for (int e = 0; e < 32; ++e) {
      const int jn = s_j[e], t = s_t[e];
      const int j = jn >= 0 ? jn : i;
      float a = pi + planes[(size_t)j * 5 * H + which * H + f] + cc[t * H + f];
      const float* w = wrf + (size_t)t * CBG_NRBF * H + f;
#pragma unroll 4
      for (int m = 0; m < CBG_NRBF; ++m) a = fmaf(w[(size_t)m * H], s_g[m * 32 + e], a);
      s_a[e * H + f] = a;
    }
    __syncthreads();
    // LayerNorm statistics per edge row: warp w handles edges w, w + H/32, ...
    for (int e = warp; e < 32; e += H / 32) {
      float s = 0.f;
      for (int c = lane; c < H; c += 32) s += s_a[e * H + c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(CBG_FULL, s, o);
      const float mean = s * (1.f / H);
      float v = 0.f;
      for (int c = lane; c < H; c += 32) { const float d = s_a[e * H + c] - mean; v = fmaf(d, d, v); }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(CBG_FULL, v, o);
      if (lane == 0) { s_stat[e] = mean; s_stat[32 + e] = 1.f / sqrtf(v * (1.f / H) + 1e-5f); }
    }
    __syncthreads();
    {
      const float ga = ln[f], be = ln[H + f];
      for (int e = 0; e < 32; ++e) s_a[e * H + f] = fmaxf((s_a[e * H + f] - s_stat[e]) * s_stat[32 + e] * ga + be, 0.f);
    }
    __syncthreads();
    // second Linear: thread f' accumulates its output for all 32 edges (W1T read once per node, coalesced)
    float acc[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) acc[e] = 0.f;
    for (int c = 0; c < H; c += 4) {
      const float w0 = w1t[(size_t)c * H + f], w1 = w1t[(size_t)(c + 1) * H + f], w2 = w1t[(size_t)(c + 2) * H + f],
                  w3 = w1t[(size_t)(c + 3) * H + f];
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const float4 a4 = *reinterpret_cast<const float4*>(s_a + e * H + c);
        acc[e] = fmaf(w3, a4.w, fmaf(w2, a4.z, fmaf(w1, a4.y, fmaf(w0, a4.x, acc[e]))));
      }
    }
    if (which == 0) {
      // logits[e][head] = sum over the head's DH features of q * k (the key bias is constant per (node, head): it
      // cancels in the softmax); DH consecutive threads = one head
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        float v = qf * acc[e];
#pragma unroll
        for (int o = DH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(CBG_FULL, v, o);
        if ((f & (DH - 1)) == 0) s_lg[e * CBG_HEADS + f / DH] = v;
      }
      __syncthreads();
      if (f < CBG_HEADS) {      // scatter_softmax over the node's valid in-edges, then * e_w (v = MLP_v(kv) * e_w)
        float mx = -INFINITY;
        for (int e = 0; e < 32; ++e) if (s_j[e] >= 0) mx = fmaxf(mx, s_lg[e * CBG_HEADS + f]);
        float sum = 0.f;
        for (int e = 0; e < 32; ++e) {
          const float p = s_j[e] >= 0 ? expf(s_lg[e * CBG_HEADS + f] - mx) : 0.f;
          s_lg[e * CBG_HEADS + f] = p;
          sum += p;
        }
        const float inv = sum > 0.f ? 1.f / sum : 0.f;
        for (int e = 0; e < 32; ++e) s_lg[e * CBG_HEADS + f] *= inv * s_ew[e];
      }
      __syncthreads();
    } else {
      const float b1 = (L + layer_off(H, IL_V_B1))[f];
      const int hd = f / DH;
#pragma unroll
      for (int e = 0; e < 32; ++e) out_acc = fmaf(s_lg[e * CBG_HEADS + hd], acc[e] + b1, out_acc);
    }
  }
  h[(size_t)i * H + f] += out_acc;          // output + h (x2h_attention.py:96); only this node's own row is touched
}

// ---- heads: eps_rot_net / eps_crd_net / classifier + the SO(3) update, one CTA per node ----------------------------------
template <int H>
__device__ __forceinline__ void head_mlp3(const float* s_h, float* s_t1, float* s_t2, const float* P, int base, float* out3) {
  // Linear(H, 2H) ReLU Linear(2H, H) ReLU Linear(H, 3)   (itatransformer.py:54-66)
  const float* w0t = P + head_off(H, base + 0);
  const float* b0 = P + head_off(H, base + 1);
  const float* w1t = P + head_off(H, base + 2);
  const float* b1 = P + head_off(H, base + 3);
  const float* w2 = P + head_off(H, base + 4);
  const float* b2 = P + head_off(H, base + 5);
  const int f = threadIdx.x;
  for (int n = f; n < 2 * H; n += H) {
    float a = b0[n];
    for (int c = 0; c < H; ++c) a = fmaf(w0t[(size_t)c * 2 * H + n], s_h[c], a);
    s_t1[n] = fmaxf(a, 0.f);
  }
  __syncthreads();
  {
    float a = b1[f];
    for (int c = 0; c < 2 * H; ++c) a = fmaf(w1t[(size_t)c * H + f], s_t1[c], a);
    s_t2[f] = fmaxf(a, 0.f);
  }
  __syncthreads();
  if (f < 96) {          // 3 outputs x 32 lanes
    const int o = f >> 5, lane = f & 31;
    float a = 0.f;
    for (int c = lane; c < H; c += 32) a = fmaf(w2[o * H + c], s_t2[c], a);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) a += __shfl_xor_sync(CBG_FULL, a, s);
    if (lane == 0) out3[o] = a + b2[o];
  }
  __syncthreads();
}

__device__ __forceinline__ void mat3_mul(const float* A, const float* B, float* C) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) C[3 * r + c] = A[3 * r] * B[c] + A[3 * r + 1] * B[3 + c] + A[3 * r + 2] * B[6 + c];
}

template <int H>
__global__ void __launch_bounds__(H) ipa_heads_kernel(const float* __restrict__ h, const float* __restrict__ o_in,
                                                      const unsigned char* __restrict__ gen, const float* __restrict__ P,
                                                      int num_classes, float* __restrict__ eps_pos, float* __restrict__ o_next,
                                                      float* __restrict__ R_next, float* __restrict__ logits, int N) {
  __shared__ float s_h[H], s_t1[2 * H], s_t2[H], s_rot[4], s_crd[4];
  const int i = blockIdx.x, f = threadIdx.x;
  if (i >= N) return;
  s_h[f] = h[(size_t)i * H + f];
  __syncthreads();
  head_mlp3<H>(s_h, s_t1, s_t2, P, IH_ROT_W0T, s_rot);
  head_mlp3<H>(s_h, s_t1, s_t2, P, IH_CRD_W0T, s_crd);
  // classifier: Linear(H, H) ShiftedSoftplus Linear(H, K)   (itatransformer.py:46-52, common.py:174-180)
  {
    const float* w0t = P + head_off(H, IH_CLS_W0T);
    float a = (P + head_off(H, IH_CLS_B0))[f];
    for (int c = 0; c < H; ++c) a = fmaf(w0t[(size_t)c * H + f], s_h[c], a);
    const float sp = (a > 20.f) ? a : log1pf(expf(a));              // F.softplus (beta = 1, threshold = 20)
    s_t2[f] = sp - 0.69314718055994530942f;
  }
  __syncthreads();
  for (int k = f >> 5; k < num_classes; k += H / 32) {
    const int lane = f & 31;
    const float* w1 = P + head_off(H, IH_CLS_W1) + (size_t)k * H;
    float a = 0.f;
    for (int c = lane; c < H; c += 32) a = fmaf(w1[c], s_t2[c], a);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) a += __shfl_xor_sync(CBG_FULL, a, s);
    if (lane == 0) logits[(size_t)i * num_classes + k] = a + (P + head_off(H, IH_CLS_B1))[k];
  }
  if (f == 0) {
    // U = quaternion_1ijk_to_rotation_matrix(eps_rot)      geometry.py:232-250
    float b = s_rot[0], c = s_rot[1], d = s_rot[2];
    const float s = sqrtf(1.f + b * b + c * c + d * d);
    const float a = 1.f / s;
    b /= s; c /= s; d /= s;
    const float U[9] = {a * a + b * b - c * c - d * d, 2 * b * c - 2 * a * d, 2 * b * d + 2 * a * c,
                        2 * b * c + 2 * a * d, a * a - b * b + c * c - d * d, 2 * c * d - 2 * a * b,
                        2 * b * d - 2 * a * c, 2 * c * d + 2 * a * b, a * a - b * b - c * c + d * d};
    // R_o = exp_skewsym(so3vec_to_skewsym(o))               so3.py:33-57
    const float wx = o_in[3 * i], wy = o_in[3 * i + 1], wz = o_in[3 * i + 2];
    const float S[9] = {0.f, wz, -wy, -wz, 0.f, wx, wy, -wx, 0.f};
    const float xn = sqrtf(wx * wx + wy * wy + wz * wz);
    const float bb = (sinf(xn) + 1e-8f) / (xn + 1e-8f);
    const float cb = (1.f - cosf(xn) + 1e-8f) / (xn * xn + 2e-8f);
    float S2[9], Ro[9], Rn[9];
    mat3_mul(S, S, S2);
#pragma unroll
    for (int e = 0; e < 9; ++e) Ro[e] = ((e % 4 == 0) ? 1.f : 0.f) + bb * S[e] + cb * S2[e];
    mat3_mul(Ro, U, Rn);                                      // R_next = R_o @ U_update   (itatransformer.py:131)
    // o_next = rotation_to_so3vec(R_next) = skewsym_to_so3vec(log_rotation(R_next))   so3.py:10-31, 60-63 (no-grad branch)
    const float tr = Rn[0] + Rn[4] + Rn[8];
    const float cos_t = fmaxf((tr - 1.f) * 0.5f, -1.f);
    const float sin_t = sqrtf(1.f - cos_t * cos_t);
    const float theta = acosf(cos_t);
    const float coef = (theta + 1e-8f) / (2.f * sin_t + 2e-8f);
    const float lx = coef * (Rn[5] - Rn[7]), ly = coef * (Rn[6] - Rn[2]), lz = coef * (Rn[1] - Rn[3]);
    const bool g = gen[i] != 0;
    o_next[3 * i] = g ? lx : wx; o_next[3 * i + 1] = g ? ly : wy; o_next[3 * i + 2] = g ? lz : wz;
#pragma unroll
    for (int e = 0; e < 9; ++e) R_next[9 * i + e] = Rn[e];
    // eps_pos = R_o eps_crd where gen_flag, else 0          (itatransformer.py:136-138)
#pragma unroll
    for (int r = 0; r < 3; ++r)
      eps_pos[3 * i + r] = g ? (Ro[3 * r] * s_crd[0] + Ro[3 * r + 1] * s_crd[1] + Ro[3 * r + 2] * s_crd[2]) : 0.f;
  }
}

template <int H>
int ipa_forward_t(const float* blob, int num_sublayers, int num_blocks, int num_classes, const float* x, const float* o,
                  const float* h_in, const int* graph_ptr, int n_graphs, int max_graph_nodes, const unsigned char* lig_flag,
                  const unsigned char* gen_flag, int N, int k, float* eps_pos, float* h_out, float* o_next, float* R_next,
                  float* logits, char* ws, cudaStream_t st) {
  // workspace: x4 [N] | nbr [N,32] | ew [N,32] | scratch [N,32] ints (gate compaction) | planes [N,5H] | q [N,H]
  size_t off = 0;
  auto take = [&](size_t nbytes) { char* p = ws + off; off += (nbytes + 255) & ~(size_t)255; return p; };
  float4* x4 = (float4*)take((size_t)N * 16);
  int* nbr = (int*)take((size_t)N * CBG_KMAX * 4);
  float* ew = (float*)take((size_t)N * CBG_KMAX * 4);
  float* planes = (float*)take((size_t)N * 5 * H * 4);
  float* q = (float*)take((size_t)N * H * 4);
  if (int rc = cbg_launch_pack_x4(x, lig_flag, gen_flag, N, x4, st)) return rc;
  if (int rc = cbg_launch_knn(x4, graph_ptr, n_graphs, max_graph_nodes, CBG_MODE_KNN, k, 0.f, 0, nullptr, nbr, st)) return rc;
  if (int rc = cbg_launch_edge_gate(blob, x4, nbr, N, nullptr, nullptr, ew, st)) return rc;
  if (h_out != h_in) CBG_CUDA_OK(cudaMemcpyAsync(h_out, h_in, (size_t)N * H * 4, cudaMemcpyDeviceToDevice, st));
  const float* head = blob + cbg_layout::kGlobalFloats;
  long long head_floats = 0, layer_floats = 0;
  for (int f = 0; f < IH_COUNT; ++f) head_floats += head_size(H, f);
  for (int f = 0; f < IL_COUNT; ++f) layer_floats += layer_size(H, f);
  const float* layers = head + head_floats;
  const size_t x2h_smem = (size_t)(32 * H + CBG_NRBF * 32 + 32 * CBG_HEADS + 64 + 96) * 4;
  static bool attr[CBG_MAX_DEVICES] = {};
  bool& attr_set = cbg_dev_flag(attr);
  if (!attr_set) {
    CBG_CUDA_OK(cudaFuncSetAttribute(ipa_x2h_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((32 * 128 + CBG_NRBF * 32 + 32 * CBG_HEADS + 64 + 96) * 4)));
    CBG_CUDA_OK(cudaFuncSetAttribute(ipa_x2h_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((32 * 256 + CBG_NRBF * 32 + 32 * CBG_HEADS + 64 + 96) * 4)));
    attr_set = true;
  }
  for (int b = 0; b < num_blocks; ++b) {      // shared blocks (itatransformer.py:115-125): x is constant, so the graph and the gate are too
    for (int l = 0; l < num_sublayers; ++l) {
      const float* L = layers + (size_t)l * layer_floats;
      dim3 g1((5 * H + 63) / 64, (N + 63) / 64);
      CBG_PROF_BEGIN(CBG_K_NODE_GEMM, st);
      ipa_linear_kernel<<<g1, 256, 0, st>>>(h_out, H, L + layer_off(H, IL_NODE_WT), 5 * H, L + layer_off(H, IL_NODE_B), planes, 5 * H, N, H, 5 * H);
      CBG_LAUNCHED(CBG_K_NODE_GEMM, st);
      CBG_PROF_BEGIN(CBG_K_MISC, st);
      ipa_ln_relu_kernel<H><<<N, H, 0, st>>>(planes + 4 * H, 5 * H, L + layer_off(H, IL_Q_LN), N);
      CBG_LAUNCHED(CBG_K_MISC, st);
      dim3 g2((H + 63) / 64, (N + 63) / 64);
      CBG_PROF_BEGIN(CBG_K_NODE_GEMM, st);
      ipa_linear_kernel<<<g2, 256, 0, st>>>(planes + 4 * H, 5 * H, L + layer_off(H, IL_Q_W1T), H, L + layer_off(H, IL_Q_B1), q, H, N, H, H);
      CBG_LAUNCHED(CBG_K_NODE_GEMM, st);
      CBG_PROF_BEGIN(CBG_K_X2H_K, st);
      ipa_x2h_kernel<H><<<N, H, x2h_smem, st>>>(x4, nbr, ew, planes, q, L, h_out, N);
      CBG_LAUNCHED(CBG_K_X2H_K, st);
    }
  }
  CBG_PROF_BEGIN(CBG_K_CLASSIFIER, st);
  ipa_heads_kernel<H><<<N, H, 0, st>>>(h_out, o, gen_flag, head, num_classes, eps_pos, o_next, R_next, logits, N);
  CBG_LAUNCHED(CBG_K_CLASSIFIER, st);
  CBG_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace

int cbg_launch_ipa_forward(const float* blob, int hidden, int num_sublayers, int num_blocks, int num_classes, const float* x,
                           const float* o, const float* h_in, const int* graph_ptr, int n_graphs, int max_graph_nodes,
                           const unsigned char* lig_flag, const unsigned char* gen_flag, int n_nodes, int k, float* eps_pos,
                           float* h_out, float* o_next, float* r_next, float* logits, char* ws, cudaStream_t st) {
  if (hidden == 128)
    return ipa_forward_t<128>(blob, num_sublayers, num_blocks, num_classes, x, o, h_in, graph_ptr, n_graphs, max_graph_nodes,
                              lig_flag, gen_flag, n_nodes, k, eps_pos, h_out, o_next, r_next, logits, ws, st);
  return ipa_forward_t<256>(blob, num_sublayers, num_blocks, num_classes, x, o, h_in, graph_ptr, n_graphs, max_graph_nodes,
                            lig_flag, gen_flag, n_nodes, k, eps_pos, h_out, o_next, r_next, logits, ws, st);
}

extern "C" {

int64_t cbg_ipa_head_floats(int32_t hidden) {
  long long s = 0;
  for (int f = 0; f < IH_COUNT; ++f) s += head_size(hidden, f);
  return s;
}
int64_t cbg_ipa_layer_floats(int32_t hidden) {
  long long s = 0;
  for (int f = 0; f < IL_COUNT; ++f) s += layer_size(hidden, f);
  return s;
}
int32_t cbg_ipa_head_fields(void) { return IH_COUNT; }
int32_t cbg_ipa_layer_fields(void) { return IL_COUNT; }
int64_t cbg_ipa_head_field_offset(int32_t hidden, int32_t field) { return head_off(hidden, field); }
int64_t cbg_ipa_head_field_size(int32_t hidden, int32_t field) { return head_size(hidden, field); }
int64_t cbg_ipa_layer_field_offset(int32_t hidden, int32_t field) { return layer_off(hidden, field); }
int64_t cbg_ipa_layer_field_size(int32_t hidden, int32_t field) { return layer_size(hidden, field); }
const char* cbg_ipa_head_field_name(int32_t f) {
  static const char* const n[IH_COUNT] = {"ROT_W0T", "ROT_B0", "ROT_W1T", "ROT_B1", "ROT_W2", "ROT_B2", "CRD_W0T", "CRD_B0",
                                          "CRD_W1T", "CRD_B1", "CRD_W2", "CRD_B2", "CLS_W0T", "CLS_B0", "CLS_W1", "CLS_B1"};
  return (f >= 0 && f < IH_COUNT) ? n[f] : nullptr;
}
const char* cbg_ipa_layer_field_name(int32_t f) {
  static const char* const n[IL_COUNT] = {"NODE_WT", "NODE_B", "Q_LN", "Q_W1T", "Q_B1", "K_WRF", "K_C", "K_LN", "K_W1T",
                                          "V_WRF", "V_C", "V_LN", "V_W1T", "V_B1", "RBF"};
  return (f >= 0 && f < IL_COUNT) ? n[f] : nullptr;
}
int64_t cbg_ipa_workspace_bytes(int64_t n_nodes, int32_t hidden) {
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  return (int64_t)(al((size_t)n_nodes * 16) + 2 * al((size_t)n_nodes * CBG_KMAX * 4) + al((size_t)n_nodes * 5 * hidden * 4) +
                   al((size_t)n_nodes * hidden * 4) + 256);
}

int32_t cbg_ipa_forward_f32(const float* blob, int32_t hidden, int32_t num_sublayers, int32_t num_blocks, int32_t num_classes,
                            const float* x, const float* o, const float* h, const int32_t* graph_ptr, int32_t n_graphs,
                            int32_t max_graph_nodes, const uint8_t* lig_flag, const uint8_t* gen_flag, int64_t n_nodes,
                            int32_t k, float* eps_pos, float* h_out, float* o_next, float* r_next, float* logits,
                            void* workspace, int64_t workspace_bytes, void* stream) {
  if (hidden != 128 && hidden != 256) { cbg_set_error("cbg_ipa_forward_f32: hidden=%d (128 or 256)", hidden); return 1; }
  if (num_classes < 1 || num_classes > CBG_IPA_MAXCLS) { cbg_set_error("num_classes=%d outside [1,%d]", num_classes, CBG_IPA_MAXCLS); return 1; }
  if (n_nodes <= 0 || n_nodes > 0x7fffffffLL / (5 * 256)) { cbg_set_error("n_nodes=%lld out of range", (long long)n_nodes); return 1; }
  if (!workspace || workspace_bytes < cbg_ipa_workspace_bytes(n_nodes, hidden)) { cbg_set_error("workspace too small"); return 1; }
  if (((uintptr_t)workspace & 255) != 0) { cbg_set_error("workspace must be 256-byte aligned"); return 1; }
  if (num_blocks < 1 || num_sublayers < 0) { cbg_set_error("num_blocks / num_sublayers"); return 1; }
  return cbg_launch_ipa_forward(blob, hidden, num_sublayers, num_blocks, num_classes, x, o, h, graph_ptr, n_graphs,
                                max_graph_nodes, lig_flag, gen_flag, (int)n_nodes, k, eps_pos, h_out, o_next, r_next, logits,
                                (char*)workspace, (cudaStream_t)stream);
}

}  // extern "C"
