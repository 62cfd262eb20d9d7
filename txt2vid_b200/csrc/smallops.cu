// Small fp32 kernels that take the last library calls off the training step:
//   * non-local block core as differentiable primitives (txt2vid/models/layers.py:23-36, 52-68): 1x2x2 max-pool with
//     recorded arg-max, batched small GEMM, row softmax with first- and second-order backward.  The discriminator's
//     block sits on the gradient-penalty path (gan/losses.py:169-178), so every primitive's backward is again one of
//     these primitives (ops.py) -- no ATen max_pool3d / cuBLAS bmm / softmax;
//   * the two Linear(.,1) heads of the discriminator (models/resnet3d.py:50-55) as row dot products with their
//     data / weight gradients (closed under the second differentiation of the penalty);
//   * relativistic / Wasserstein loss reduction over all pyramid levels and prediction pairs in ONE launch forward and
//     ONE backward (gan/losses.py:55-85, gan/cond_gan.py:51-61);
//   * gradient-penalty arithmetic: per-sample interpolation (gan/losses.py:140-145), the fp32 dot / scale kernels
//     behind sum ||g||^2 and its derivative, and mean_b (||g_b|| - 1)^2 with its derivative (losses.py:180-186).
#include "t2v_common.cuh"

namespace t2v {

static inline unsigned nblocks(long long n, int per) {
  long long b = (n + per - 1) / per;
  return (unsigned)(b < 1 ? 1 : b);
}

// ------------------------------------------------------------------------------------ 1x2x2 max-pool with arg-max
// x fp32 [maps][H][W][c] (maps = N*D) -> y [maps][H/2][W/2][c], idx u8 in 0..3 (first maximum, as ATen)
__global__ void maxpool122_fwd_kernel(const float* __restrict__ x, float* __restrict__ y,
                                      unsigned char* __restrict__ idx, int H, int W, int c, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int Hp = H / 2, Wp = W / 2;
  long long t = i;
  const int ch = (int)(t % c); t /= c;
  const int wp = (int)(t % Wp); t /= Wp;
  const int hp = (int)(t % Hp); t /= Hp;
  const long long m = t;
  const float* base = x + ((m * H + 2 * hp) * W + 2 * wp) * c + ch;
  const float v[4] = {base[0], base[c], base[(long long)W * c], base[(long long)W * c + c]};
  float best = v[0];
  int arg = 0;
#pragma unroll
  for (int j = 1; j < 4; ++j)
    if (v[j] > best || (v[j] != v[j] && best == best)) { best = v[j]; arg = j; }
  y[i] = best;
  idx[i] = (unsigned char)arg;
}
// gather: y[pooled] = x[window voxel idx]   (linear in x: the backward of scatter)
__global__ void pool122_gather_kernel(const float* __restrict__ x, const unsigned char* __restrict__ idx,
                                      float* __restrict__ y, int H, int W, int c, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int Hp = H / 2, Wp = W / 2;
  long long t = i;
  const int ch = (int)(t % c); t /= c;
  const int wp = (int)(t % Wp); t /= Wp;
  const int hp = (int)(t % Hp); t /= Hp;
  const int a = idx[i];
  y[i] = x[((t * H + 2 * hp + (a >> 1)) * W + 2 * wp + (a & 1)) * c + ch];
}
// scatter: dx[window voxel idx] = dy[pooled], zeros elsewhere (one thread per pooled element writes its 4 voxels)
__global__ void pool122_scatter_kernel(const float* __restrict__ dy, const unsigned char* __restrict__ idx,
                                       float* __restrict__ dx, int H, int W, int c, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int Hp = H / 2, Wp = W / 2;
  long long t = i;
  const int ch = (int)(t % c); t /= c;
  const int wp = (int)(t % Wp); t /= Wp;
  const int hp = (int)(t % Hp); t /= Hp;
  const int a = idx[i];
  const float g = dy[i];
  float* base = dx + ((t * H + 2 * hp) * W + 2 * wp) * c + ch;
  base[0] = a == 0 ? g : 0.f;
  base[c] = a == 1 ? g : 0.f;
  base[(long long)W * c] = a == 2 ? g : 0.f;
  base[(long long)W * c + c] = a == 3 ? g : 0.f;
}

// ------------------------------------------------------------------------------------ batched small GEMM (fp32)
// C[b] (M x N, row-major) = op(A[b]) * op(B[b]);  ta: A[b] stored (K x M);  tb: B[b] stored (N x K)
struct BmmParams {
  const float* A; const float* B; float* C;
  int M, N, K, ta, tb;
  long long sA, sB, sC;
};
__global__ void __launch_bounds__(256) bmm_kernel(const BmmParams p) {
  __shared__ float As[16][65], Bs[16][65];
  const int b = blockIdx.z;
  const float* A = p.A + b * p.sA;
  const float* B = p.B + b * p.sB;
  float* C = p.C + b * p.sC;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < p.K; k0 += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = threadIdx.x + 256 * i;
      // A tile: element (k, m)
      {
        const int k = p.ta ? e / 64 : e % 16, m = p.ta ? e % 64 : e / 16;
        float v = 0.f;
        if (k0 + k < p.K && m0 + m < p.M)
          v = p.ta ? A[(long long)(k0 + k) * p.M + m0 + m] : A[(long long)(m0 + m) * p.K + k0 + k];
        As[k][m] = v;
      }
      {
        const int k = p.tb ? e % 16 : e / 64, n = p.tb ? e / 16 : e % 64;
        float v = 0.f;
        if (k0 + k < p.K && n0 + n < p.N)
          v = p.tb ? B[(long long)(n0 + n) * p.K + k0 + k] : B[(long long)(k0 + k) * p.N + n0 + n];
        Bs[k][n] = v;
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], bb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; bb[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < p.N) C[(long long)m * p.N + n] = acc[i][j];
    }
  }
}

// ------------------------------------------------------------------------------------ row softmax (+ 1st / 2nd order bwd)
// one warp per row
__global__ void softmax_fwd_kernel(const float* __restrict__ S, float* __restrict__ out, long long rows, int cols) {
  const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* s = S + r * cols;
  float m = -INFINITY;
  for (int j = lane; j < cols; j += 32) m = fmaxf(m, s[j]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float l = 0.f;
  for (int j = lane; j < cols; j += 32) l += expf(s[j] - m);
  l = warp_sum(l);
  const float inv = 1.f / l;
  for (int j = lane; j < cols; j += 32) out[r * cols + j] = expf(s[j] - m) * inv;
}
// dS = beta * (dbeta - sum_j beta_j dbeta_j)
__global__ void softmax_bwd_kernel(const float* __restrict__ beta, const float* __restrict__ dbeta,
                                   float* __restrict__ dS, long long rows, int cols) {
  const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* b = beta + r * cols;
  const float* d = dbeta + r * cols;
  float s = 0.f;
  for (int j = lane; j < cols; j += 32) s = fmaf(b[j], d[j], s);
  s = warp_sum(s);
  for (int j = lane; j < cols; j += 32) dS[r * cols + j] = b[j] * (d[j] - s);
}
// derivative of dS = softmax_bwd(beta, dbeta) against a cotangent u:
//   g_dbeta = beta * (u - t),  g_beta = u * (dbeta - s) - dbeta * t,   s = sum beta dbeta, t = sum beta u
__global__ void softmax_bwd_bwd_kernel(const float* __restrict__ beta, const float* __restrict__ dbeta,
                                       const float* __restrict__ u, float* __restrict__ g_beta,
                                       float* __restrict__ g_dbeta, long long rows, int cols) {
  const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* b = beta + r * cols;
  const float* d = dbeta + r * cols;
  const float* uu = u + r * cols;
  float s = 0.f, t = 0.f;
  for (int j = lane; j < cols; j += 32) { s = fmaf(b[j], d[j], s); t = fmaf(b[j], uu[j], t); }
  s = warp_sum(s);
  t = warp_sum(t);
  for (int j = lane; j < cols; j += 32) {
    if (g_dbeta) g_dbeta[r * cols + j] = b[j] * (uu[j] - t);
    if (g_beta) g_beta[r * cols + j] = uu[j] * (d[j] - s) - d[j] * t;
  }
}

// ------------------------------------------------------------------------------------ Linear(., 1) heads
// out[b] = feat[b,:] . w[0:F] + cond[b,:] . w[F:F+E] + bias;  one warp per row
__global__ void head_fwd_kernel(const float* __restrict__ feat, const float* __restrict__ cond,
                                const float* __restrict__ w, const float* __restrict__ bias, float* __restrict__ out,
                                int B, int F, int E) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= B) return;
  float acc = 0.f;
  const float* f = feat + (long long)r * F;
  for (int j = lane; j < F; j += 32) acc = fmaf(f[j], w[j], acc);
  if (cond != nullptr) {
    const float* c = cond + (long long)r * E;
    for (int j = lane; j < E; j += 32) acc = fmaf(c[j], w[F + j], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) out[r] = acc + (bias ? bias[0] : 0.f);
}
// dfeat[b, j] = dpred[b] * w[j],  dcond[b, j] = dpred[b] * w[F + j]
__global__ void head_bwd_data_kernel(const float* __restrict__ dpred, const float* __restrict__ w,
                                     float* __restrict__ dfeat, float* __restrict__ dcond, int B, int F, int E) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int FE = F + (dcond ? E : 0);
  if (i >= (long long)B * FE) return;
  const int b = (int)(i / FE), j = (int)(i % FE);
  const float v = dpred[b] * w[j];
  if (j < F) dfeat[(long long)b * F + j] = v;
  else dcond[(long long)b * E + j - F] = v;
}
// dw[j] (+)= sum_b dpred[b] * [feat | cond][b, j];  db (+)= sum_b dpred[b].  One thread per column j, rows in chunks
// of 64 per block (grid.y) combined with one atomicAdd per column and block; dw / db zeroed by the host when not
// accumulating.
__global__ void head_bwd_weight_kernel(const float* __restrict__ dpred, const float* __restrict__ feat,
                                       const float* __restrict__ cond, float* __restrict__ dw, float* __restrict__ db,
                                       int B, int F, int E) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int FE = F + (cond ? E : 0);
  const int b0 = blockIdx.y * 64, b1 = min(B, b0 + 64);
  if (j < FE) {
    float acc = 0.f;
    for (int b = b0; b < b1; ++b)
      acc = fmaf(dpred[b], j < F ? feat[(long long)b * F + j] : cond[(long long)b * E + j - F], acc);
    atomicAdd(dw + j, acc);
  }
  if (db != nullptr && j == 0) {
    float s = 0.f;
    for (int b = b0; b < b1; ++b) s += dpred[b];
    atomicAdd(db, s);
  }
}

// ------------------------------------------------------------------------------------ fused loss reduction
// out = sum_e weight_e / n_e * sum_j f(b_e[j] - a_e[j]);  mode 0: f = softplus (RSGAN: BCE-with-logits of (a - b) against
// ones, gan/losses.py:74-85);  mode 1: f = identity (Wasserstein critic difference, losses.py:55-68)
struct LossEntries {
  static constexpr int kMax = 24;
  const float* a[kMax];
  const float* b[kMax];
  float* da[kMax];
  float* db[kMax];
  int n[kMax];
  float weight[kMax];
  int count;
};
T2V_DEVINL float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__global__ void __launch_bounds__(256) rel_loss_fwd_kernel(const LossEntries e, int mode, float* __restrict__ out) {
  __shared__ float red[8];
  float acc = 0.f;
  for (int k = 0; k < e.count; ++k) {
    const float sc = e.weight[k] / (float)e.n[k];
    float s = 0.f;
    for (int j = threadIdx.x; j < e.n[k]; j += blockDim.x) {
      const float d = e.b[k][j] - e.a[k][j];
      s += mode == 0 ? softplus_f(d) : d;
    }
    acc = fmaf(sc, s, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    out[0] = t;
  }
}
// da[j] (+)= -g * weight/n * f'(b - a),  db[j] (+)= +...  (several entries may share a tensor: the host zeroes the
// gradient buffers once and every entry accumulates; entries run sequentially inside one block, so no atomics)
__global__ void __launch_bounds__(256) rel_loss_bwd_kernel(const LossEntries e, int mode,
                                                           const float* __restrict__ gout) {
  const float g = gout[0];
  for (int k = 0; k < e.count; ++k) {
    const float sc = g * e.weight[k] / (float)e.n[k];
    for (int j = threadIdx.x; j < e.n[k]; j += blockDim.x) {
      const float d = e.b[k][j] - e.a[k][j];
      const float fp = mode == 0 ? 1.f / (1.f + expf(-d)) : 1.f;
      if (e.da[k]) e.da[k][j] -= sc * fp;
      if (e.db[k]) e.db[k][j] += sc * fp;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------ gradient-penalty arithmetic
// out[b, s] = alpha[b] * real[b, s] + (1 - alpha[b]) * fake[b, s]        (gan/losses.py:140-145)
__global__ void lerp_rows_kernel(const float* __restrict__ real, const float* __restrict__ fake,
                                 const float* __restrict__ alpha, float* __restrict__ out, long long S,
                                 long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float a = alpha[i / S];
  out[i] = a * real[i] + (1.f - a) * fake[i];
}

// Non-zero-centred penalty mean_b (||g_b||_2 - 1)^2 of g (B, S) (gan/losses.py:180-186, combine = torch.mean).
// Pass 1: block (sample b, split k) sums the squares of its contiguous chunk of row b with 16-byte loads into
// partials[b * splits + k].  Which thread reads which element and the in-block tree depend on S and splits only,
// so two calls give bit-identical sums (the fp32 mode relies on it, DESIGN §2).
__global__ void __launch_bounds__(256) gp_norm_partial_kernel(const float* __restrict__ g, float* __restrict__ partials,
                                                              long long S4, long long chunk4, int splits) {
  __shared__ float red[8];
  const long long blk = blockIdx.x;
  const long long b = blk / splits;
  const long long lo = (blk % splits) * chunk4, hi = min(S4, lo + chunk4);
  const float4* row = reinterpret_cast<const float4*>(g) + b * S4;
  float acc = 0.f;
#pragma unroll 8
  for (long long i = lo + threadIdx.x; i < hi; i += 256) {
    const float4 v = __ldg(row + i);
    acc = fmaf(v.x, v.x, acc);
    acc = fmaf(v.y, v.y, acc);
    acc = fmaf(v.z, v.z, acc);
    acc = fmaf(v.w, v.w, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    partials[blk] = t;
  }
}
// Pass 2 (one block): n_b = sqrt(sum of row b's partials, in split order); out = mean_b (n_b - 1)^2 over a fixed tree.
__global__ void __launch_bounds__(256) gp_norm_finish_kernel(const float* __restrict__ partials, float* __restrict__ norms,
                                                             float* __restrict__ out, long long B, int splits) {
  __shared__ float red[8];
  float acc = 0.f;
  for (long long b = threadIdx.x; b < B; b += 256) {
    const float* p = partials + b * splits;
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += p[k];
    const float n = sqrtf(s);
    norms[b] = n;
    const float d = n - 1.f;
    acc = fmaf(d, d, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    out[0] = t / (float)B;
  }
}
// dg[b, s] = gout * 2 (n_b - 1) / (n_b B) * g[b, s]; 0 on a row with n_b = 0 (the subgradient torch's norm takes)
__global__ void gp_norm_bwd_kernel(const float* __restrict__ g, const float* __restrict__ norms,
                                   const float* __restrict__ gout, float* __restrict__ dg, long long S4,
                                   long long total4, float B) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const float n = norms[i / S4];
  const float c = n > 0.f ? gout[0] * (2.f * (n - 1.f) / (n * B)) : 0.f;
  float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
  v.x *= c;
  v.y *= c;
  v.z *= c;
  v.w *= c;
  reinterpret_cast<float4*>(dg)[i] = v;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace t2v

using namespace t2v;
#define STREAM reinterpret_cast<cudaStream_t>(stream)

extern "C" {

int t2v_maxpool122_fwd(const float* x, float* y, void* idx, int64_t maps, int32_t H, int32_t W, int32_t c,
                       void* stream) {
  if (H % 2 || W % 2) return T2V_ERR_ARG;
  const long long total = maps * (H / 2) * (W / 2) * c;
  if (total == 0) return T2V_OK;
  maxpool122_fwd_kernel<<<nblocks(total, 256), 256, 0, STREAM>>>(x, y, reinterpret_cast<unsigned char*>(idx), H, W, c,
                                                                 total);
  count_launch();
  return check_last("maxpool122_fwd");
}
int t2v_pool122_gather(const float* x, const void* idx, float* y, int64_t maps, int32_t H, int32_t W, int32_t c,
                       void* stream) {
  if (H % 2 || W % 2) return T2V_ERR_ARG;
  const long long total = maps * (H / 2) * (W / 2) * c;
  if (total == 0) return T2V_OK;
  pool122_gather_kernel<<<nblocks(total, 256), 256, 0, STREAM>>>(x, reinterpret_cast<const unsigned char*>(idx), y, H,
                                                                 W, c, total);
  count_launch();
  return check_last("pool122_gather");
}
int t2v_pool122_scatter(const float* dy, const void* idx, float* dx, int64_t maps, int32_t H, int32_t W, int32_t c,
                        void* stream) {
  if (H % 2 || W % 2) return T2V_ERR_ARG;
  const long long total = maps * (H / 2) * (W / 2) * c;
  if (total == 0) return T2V_OK;
  pool122_scatter_kernel<<<nblocks(total, 256), 256, 0, STREAM>>>(dy, reinterpret_cast<const unsigned char*>(idx), dx,
                                                                  H, W, c, total);
  count_launch();
  return check_last("pool122_scatter");
}

int t2v_bmm_f32(const float* A, const float* B, float* C, int32_t batch, int32_t M, int32_t N, int32_t K,
                int32_t trans_a, int32_t trans_b, void* stream) {
  if (!A || !B || !C || batch < 0 || M < 0 || N < 0 || K < 0 || batch > 65535) return T2V_ERR_ARG;
  if (batch == 0 || M == 0 || N == 0) return T2V_OK;
  BmmParams p{A, B, C, M, N, K, trans_a ? 1 : 0, trans_b ? 1 : 0, (long long)M * K, (long long)K * N, (long long)M * N};
  dim3 grid((N + 63) / 64, (M + 63) / 64, batch);
  bmm_kernel<<<grid, 256, 0, STREAM>>>(p);
  count_launch();
  return check_last("bmm_f32");
}

int t2v_softmax_fwd(const float* S, float* out, int64_t rows, int32_t cols, void* stream) {
  if (rows == 0) return T2V_OK;
  softmax_fwd_kernel<<<nblocks(rows * 32, 256), 256, 0, STREAM>>>(S, out, rows, cols);
  count_launch();
  return check_last("softmax_fwd");
}
int t2v_softmax_bwd(const float* beta, const float* dbeta, float* dS, int64_t rows, int32_t cols, void* stream) {
  if (rows == 0) return T2V_OK;
  softmax_bwd_kernel<<<nblocks(rows * 32, 256), 256, 0, STREAM>>>(beta, dbeta, dS, rows, cols);
  count_launch();
  return check_last("softmax_bwd");
}
int t2v_softmax_bwd_bwd(const float* beta, const float* dbeta, const float* u, float* g_beta, float* g_dbeta,
                        int64_t rows, int32_t cols, void* stream) {
  if (rows == 0) return T2V_OK;
  softmax_bwd_bwd_kernel<<<nblocks(rows * 32, 256), 256, 0, STREAM>>>(beta, dbeta, u, g_beta, g_dbeta, rows, cols);
  count_launch();
  return check_last("softmax_bwd_bwd");
}

int t2v_head_fwd(const float* feat, const float* cond, const float* w, const float* bias, float* out, int32_t B,
                 int32_t F, int32_t E, void* stream) {
  if (!feat || !w || !out) return T2V_ERR_ARG;
  if (B == 0) return T2V_OK;
  head_fwd_kernel<<<nblocks((long long)B * 32, 256), 256, 0, STREAM>>>(feat, cond, w, bias, out, B, F, cond ? E : 0);
  count_launch();
  return check_last("head_fwd");
}
int t2v_head_bwd_data(const float* dpred, const float* w, float* dfeat, float* dcond, int32_t B, int32_t F, int32_t E,
                      void* stream) {
  if (!dpred || !w || !dfeat) return T2V_ERR_ARG;
  const long long total = (long long)B * (F + (dcond ? E : 0));
  if (total == 0) return T2V_OK;
  head_bwd_data_kernel<<<nblocks(total, 256), 256, 0, STREAM>>>(dpred, w, dfeat, dcond, B, F, E);
  count_launch();
  return check_last("head_bwd_data");
}
int t2v_head_bwd_weight(const float* dpred, const float* feat, const float* cond, float* dw, float* db, int32_t B,
                        int32_t F, int32_t E, int32_t accumulate, void* stream) {
  if (!dpred || !feat || !dw) return T2V_ERR_ARG;
  const int FE = F + (cond ? E : 0);
  if (!accumulate) {
    cudaMemsetAsync(dw, 0, sizeof(float) * FE, STREAM);
    if (db) cudaMemsetAsync(db, 0, sizeof(float), STREAM);
  }
  if (B == 0) return T2V_OK;
  dim3 grid((FE + 127) / 128, (B + 63) / 64, 1);
  head_bwd_weight_kernel<<<grid, 128, 0, STREAM>>>(dpred, feat, cond, dw, db, B, F, E);
  count_launch();
  return check_last("head_bwd_weight");
}

static int fill_entries(LossEntries& e, int32_t count, const float* const* a, const float* const* b, float* const* da,
                        float* const* db, const int32_t* n, const float* weight) {
  if (count < 0 || count > LossEntries::kMax) return T2V_ERR_ARG;
  e.count = count;
  for (int i = 0; i < count; ++i) {
    if (!a[i] || !b[i] || n[i] <= 0) return T2V_ERR_ARG;
    e.a[i] = a[i]; e.b[i] = b[i];
    e.da[i] = da ? da[i] : nullptr;
    e.db[i] = db ? db[i] : nullptr;
    e.n[i] = n[i]; e.weight[i] = weight[i];
  }
  return T2V_OK;
}
int t2v_rel_loss_fwd(int32_t count, const float* const* host_a, const float* const* host_b, const int32_t* host_n,
                     const float* host_weight, int32_t mode, float* out, void* stream) {
  LossEntries e;
  int rc = fill_entries(e, count, host_a, host_b, nullptr, nullptr, host_n, host_weight);
  if (rc) return rc;
  rel_loss_fwd_kernel<<<1, 256, 0, STREAM>>>(e, mode, out);
  count_launch();
  return check_last("rel_loss_fwd");
}
int t2v_rel_loss_bwd(int32_t count, const float* const* host_a, const float* const* host_b, float* const* host_da,
                     float* const* host_db, const int32_t* host_n, const float* host_weight, int32_t mode,
                     const float* gout, void* stream) {
  LossEntries e;
  int rc = fill_entries(e, count, host_a, host_b, host_da, host_db, host_n, host_weight);
  if (rc) return rc;
  rel_loss_bwd_kernel<<<1, 256, 0, STREAM>>>(e, mode, gout);
  count_launch();
  return check_last("rel_loss_bwd");
}

int t2v_lerp_rows(const float* real, const float* fake, const float* alpha, float* out, int64_t B, int64_t S,
                  void* stream) {
  const long long total = B * S;
  if (total == 0) return T2V_OK;
  lerp_rows_kernel<<<nblocks(total, 256), 256, 0, STREAM>>>(real, fake, alpha, out, S, total);
  count_launch();
  return check_last("lerp_rows");
}

int t2v_gp_norm_fwd(const float* g, float* partials, float* norms, float* out, int64_t B, int64_t S, int32_t splits,
                    void* stream) {
  if (B < 1 || S < 4 || S % 4 || splits < 1 || B * splits > 0x7fffffffLL) return T2V_ERR_ARG;
  if (!g || !partials || !norms || !out || !aligned16(g)) return T2V_ERR_ARG;
  const long long S4 = S / 4, chunk4 = (S4 + splits - 1) / splits;
  gp_norm_partial_kernel<<<(unsigned)(B * splits), 256, 0, STREAM>>>(g, partials, S4, chunk4, splits);
  gp_norm_finish_kernel<<<1, 256, 0, STREAM>>>(partials, norms, out, B, splits);
  count_launch(2);
  return check_last("gp_norm_fwd");
}
int t2v_gp_norm_bwd(const float* g, const float* norms, const float* gout, float* dg, int64_t B, int64_t S,
                    void* stream) {
  if (B < 1 || S < 4 || S % 4) return T2V_ERR_ARG;
  if (!g || !norms || !gout || !dg || !aligned16(g) || !aligned16(dg)) return T2V_ERR_ARG;
  const long long total4 = B * (S / 4);
  gp_norm_bwd_kernel<<<nblocks(total4, 256), 256, 0, STREAM>>>(g, norms, gout, dg, S / 4, total4, (float)B);
  count_launch();
  return check_last("gp_norm_bwd");
}

}  // extern "C"
