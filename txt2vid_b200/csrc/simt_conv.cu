// CUDA-core implicit-GEMM convolution (fp32 FMA; bf16 or fp32 channels-last I/O).
// Same contract as the tcgen05 engine in igemm_sm100.cu; used for shapes that engine does not take
// (channel counts that are not multiples of 16/64), as an on-GPU cross-check in the tests, and -- instantiated for
// fp32 operands (T2V_EPI_IN_F32 / T2V_ALGO_SIMT_F32) -- as the convolution of the fp32 PARITY mode: exact fp32
// products, fp32 accumulation flushed once per tap (chains of <= Cin FMAs), i.e. the reference's own numerics.  The
// tensor pipe cannot give that: its fp32 accumulator truncates on every MMA, which costs ~3e-5 relative on the
// K = 9216 layers however finely the operands are split (measured: profiles/r02_fp32_engine_accuracy.txt).
#include "t2v_common.cuh"

namespace t2v {

struct SimtParams {
  int N, D, H, W, Cin, Cout;
  int kd, kh, kw, pd, ph, pw;
  long long P;  // positions
  const void* x;
  const void* w;   // [Cout][taps][Cin]
  const float* bias;
  const void* residual;
  void* out;
  int out_f32, relu, relu_mask;
  // wgrad
  const void* dy;
  float* dw;
  int splits;
};

static constexpr int TM = 64, TN = 64, TK = 16;

// y[pos, co] tile 64x64, 256 threads, 4x4 per thread
template <typename T>
__global__ void __launch_bounds__(256) simt_fprop_kernel(const SimtParams p) {
  const T* __restrict__ px = reinterpret_cast<const T*>(p.x);
  const T* __restrict__ pw = reinterpret_cast<const T*>(p.w);
  const T* __restrict__ pres = reinterpret_cast<const T*>(p.residual);
  __shared__ float As[TK][TM + 1];
  __shared__ float Bs[TK][TN + 1];
  const int tid = threadIdx.x;
  const long long pos0 = (long long)blockIdx.x * TM;
  const int co0 = blockIdx.y * TN;
  const int tx = tid % 16, ty = tid / 16;  // tx -> cout, ty -> pos
  float acc[4][4] = {}, tot[4][4] = {};
  const int taps = p.kd * p.kh * p.kw;
  // each thread loads 4 elements of A and 4 of B per k-step: element e = tid + 256*i -> (row = e/16, k = e%16)
  for (int tap = 0; tap < taps; ++tap) {
    const int a_w = tap % p.kw, a_h = (tap / p.kw) % p.kh, a_d = tap / (p.kw * p.kh);
    for (int c0 = 0; c0 < p.Cin; c0 += TK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int e = tid + 256 * i;
        const int r = e / TK, k = e % TK;
        const long long pos = pos0 + r;
        float v = 0.f;
        if (pos < p.P && c0 + k < p.Cin) {
          long long t = pos;
          const int w = (int)(t % p.W); t /= p.W;
          const int h = (int)(t % p.H); t /= p.H;
          const int d = (int)(t % p.D); t /= p.D;
          const int n = (int)t;
          const int ww = w + a_w - p.pw, hh = h + a_h - p.ph, dd = d + a_d - p.pd;
          if (ww >= 0 && ww < p.W && hh >= 0 && hh < p.H && dd >= 0 && dd < p.D)
            v = bf2f(px[((((long long)n * p.D + dd) * p.H + hh) * p.W + ww) * p.Cin + c0 + k]);
        }
        As[k][r] = v;
        float wv = 0.f;
        const int co = co0 + r;
        if (co < p.Cout && c0 + k < p.Cin) wv = bf2f(pw[((long long)co * taps + tap) * p.Cin + c0 + k]);
        Bs[k][r] = wv;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < TK; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
    // one flush per tap: FMA chains stay <= Cin long (pairwise-like summation over the taps)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { tot[i][j] += acc[i][j]; acc[i][j] = 0.f; }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long pos = pos0 + ty * 4 + i;
    if (pos >= p.P) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = co0 + tx * 4 + j;
      if (co >= p.Cout) continue;
      float v = tot[i][j];
      if (p.bias) v += p.bias[co];
      if (p.residual) {
        const float r = bf2f(pres[pos * p.Cout + co]);
        if (p.relu_mask) v = r > 0.f ? v : 0.f;       // T2V_EPI_RELU_MASK: the pointer is the ReLU reference
        else v += r;
      }
      if (p.relu) v = fmaxf(v, 0.f);
      if (p.out_f32) reinterpret_cast<float*>(p.out)[pos * p.Cout + co] = v;
      else reinterpret_cast<__nv_bfloat16*>(p.out)[pos * p.Cout + co] = f2bf(v);
    }
  }
}

// dw[co, tap, ci] tile 64x64 for one tap, summed over a slice of positions
template <typename T>
__global__ void __launch_bounds__(256) simt_wgrad_kernel(const SimtParams p) {
  const T* __restrict__ pdy = reinterpret_cast<const T*>(p.dy);
  const T* __restrict__ px = reinterpret_cast<const T*>(p.x);
  __shared__ float As[TK][TM + 1];  // dy[pos k][co]
  __shared__ float Bs[TK][TN + 1];  // x[pos k + tap][ci]
  const int tid = threadIdx.x;
  const int co0 = blockIdx.x * TM, ci0 = blockIdx.y * TN;
  const int tap = blockIdx.z / p.splits, split = blockIdx.z % p.splits;
  const int taps = p.kd * p.kh * p.kw;
  const int a_w = tap % p.kw, a_h = (tap / p.kw) % p.kh, a_d = tap / (p.kw * p.kh);
  const int tx = tid % 16, ty = tid / 16;  // tx -> ci, ty -> co
  const long long chunks = (p.P + TK - 1) / TK;
  const long long per = (chunks + p.splits - 1) / p.splits;
  const long long cb = split * per, ce = min(chunks, cb + per);
  float acc[4][4] = {}, tot[4][4] = {};
  for (long long ch = cb; ch < ce; ++ch) {
    if (((ch - cb) & 63) == 63) {                 // flush every 1024 positions: bounded FMA chains
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { tot[i][j] += acc[i][j]; acc[i][j] = 0.f; }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + 256 * i;
      const int k = e / TM, c = e % TM;  // consecutive threads -> consecutive channels (coalesced)
      const long long pos = ch * TK + k;
      float av = 0.f, bv = 0.f;
      if (pos < p.P) {
        if (co0 + c < p.Cout) av = bf2f(pdy[pos * p.Cout + co0 + c]);
        if (ci0 + c < p.Cin) {
          long long t = pos;
          const int w = (int)(t % p.W); t /= p.W;
          const int h = (int)(t % p.H); t /= p.H;
          const int d = (int)(t % p.D); t /= p.D;
          const int n = (int)t;
          const int ww = w + a_w - p.pw, hh = h + a_h - p.ph, dd = d + a_d - p.pd;
          if (ww >= 0 && ww < p.W && hh >= 0 && hh < p.H && dd >= 0 && dd < p.D)
            bv = bf2f(px[((((long long)n * p.D + dd) * p.H + hh) * p.W + ww) * p.Cin + ci0 + c]);
        }
      }
      As[k][c] = av;
      Bs[k][c] = bv;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + ty * 4 + i;
    if (co >= p.Cout) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ci = ci0 + tx * 4 + j;
      if (ci >= p.Cin) continue;
      atomicAdd(p.dw + ((long long)co * taps + tap) * p.Cin + ci, tot[i][j] + acc[i][j]);
    }
  }
}

static void fill(SimtParams& p, const t2v_conv_geom* g) {
  p.N = g->N; p.D = g->D; p.H = g->H; p.W = g->W; p.Cin = g->Cin; p.Cout = g->Cout;
  p.kd = g->kd; p.kh = g->kh; p.kw = g->kw;
  p.pd = g->kd / 2; p.ph = g->kh / 2; p.pw = g->kw / 2;
  p.P = (long long)g->N * g->D * g->H * g->W;
}

int simt_fprop_launch(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                      const void* residual, void* y, uint32_t flags, cudaStream_t stream) {
  SimtParams p{};
  fill(p, g);
  p.x = x;
  p.w = w;
  p.bias = bias;
  p.residual = residual;
  p.out = y;
  p.out_f32 = (flags & (T2V_EPI_OUT_F32 | T2V_EPI_IN_F32)) ? 1 : 0;
  p.relu = (flags & T2V_EPI_RELU) ? 1 : 0;
  p.relu_mask = (flags & T2V_EPI_RELU_MASK) ? 1 : 0;
  dim3 grid((unsigned)((p.P + TM - 1) / TM), (g->Cout + TN - 1) / TN, 1);
  if (flags & T2V_EPI_IN_F32) simt_fprop_kernel<float><<<grid, 256, 0, stream>>>(p);
  else simt_fprop_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(p);
  count_launch();
  return check_last("simt_fprop");
}

int simt_wgrad_launch(const t2v_conv_geom* g, const void* dy, const void* x, float* dw, int accumulate,
                      cudaStream_t stream, int in_f32) {
  SimtParams p{};
  fill(p, g);
  p.dy = dy;
  p.x = x;
  p.dw = dw;
  const int taps = g->kd * g->kh * g->kw;
  const int base = ((g->Cout + TM - 1) / TM) * ((g->Cin + TN - 1) / TN) * taps;
  long long chunks = (p.P + TK - 1) / TK;
  int splits = (4 * 148 + base - 1) / base;
  if (splits > chunks / 8) splits = (int)(chunks / 8);
  if (splits < 1) splits = 1;
  p.splits = splits;
  if (!accumulate) cudaMemsetAsync(dw, 0, (size_t)g->Cout * taps * g->Cin * sizeof(float), stream);
  dim3 grid((g->Cout + TM - 1) / TM, (g->Cin + TN - 1) / TN, taps * splits);
  if (in_f32) simt_wgrad_kernel<float><<<grid, 256, 0, stream>>>(p);
  else simt_wgrad_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(p);
  count_launch();
  return check_last("simt_wgrad");
}

}  // namespace t2v
