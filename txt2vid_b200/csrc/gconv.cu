// CUDA-core implicit-GEMM convolution: any kernel / stride / zero padding, 1-D .. 3-D, fp32 FMA, channels-last bf16
// or fp32 storage.  One implementation behind two ABI routes:
//   * t2v_gconv_{fprop,dgrad,wgrad}[_f32]: the TGAN / TCWYT layers of any geometry --
//       Conv3d/Conv2d k4 s2 p1, k(1,3,3) s1|2 p0, k2 s2 p0    (txt2vid/models/tcwyt/video_discrim.py:12-46,
//       frame_discrim.py:8-22,49, motion_discrim.py:19)                       -> gconv_fprop
//       ConvTranspose1d/2d/3d k4 s2 p1, k(2,6,6) p0, k3 s1 p1, k1             (tgan/gen.py:21-25,
//       tgan/temporal_gen.py:16-20, tcwyt/gen.py:14-30)                       -> gconv_dgrad (a transposed
//       convolution IS the data gradient of the convolution with the same weight tensor)
//       their weight gradients                                                -> gconv_wgrad
//   * the CUDA-core branches of t2v_conv_fprop / t2v_conv_dgrad / t2v_conv_wgrad (api_conv.cu, stride 1, padding k/2):
//     T2V_ALGO_SIMT, shapes the tcgen05 engine does not take, and the fp32 parity mode (T2V_EPI_IN_F32 /
//     T2V_ALGO_SIMT_F32).
// Numerics of the fp32 parity mode, i.e. the reference's own: exact fp32 products, the per-thread accumulator is added
// into the running total once per tap (FMA chains of at most Cin terms, summed over the taps in ascending order), and
// the weight gradient flushes every 64 chunks of 16 positions.  The tensor pipe cannot give that: its fp32 accumulator
// truncates on every MMA, ~3e-5 relative on the K = 9216 layers however finely the operands are split (measured:
// profiles/r02_fp32_engine_accuracy.txt).
// Weight layout [Co][taps][Ci] where (Co, Ci) are the channel counts of the *convolution* whose input has Ci channels:
// for a ConvTranspose(Cin_t, Cout_t) that is Co = Cin_t, Ci = Cout_t, which is exactly the memory order of PyTorch's
// (Cin_t, Cout_t, k...) parameter in channels-last form.
#include "t2v_common.cuh"

namespace t2v {

static constexpr int GT = 64, GK = 16;

template <typename ST>
struct GconvParams {
  t2v_gconv_geom g;
  long long Pi, Po;            // input / output positions
  const ST* x;      // [N][Di][Hi][Wi][Ci]   (ST = bf16, or fp32 in the fp32 parity mode)
  const ST* w;      // [Co][taps][Ci]
  const ST* dy;     // [N][Do][Ho][Wo][Co]
  const float* bias;
  const ST* residual;          // fprop: output-shaped, added (or the ReLU reference under relu_mask)
  void* out;
  int out_f32, relu, relu_mask;
  float* dw;
  int splits;
};

template <typename I>
__device__ __forceinline__ void decode_pos(I pos, int D, int H, int W, int* n, int* d, int* h, int* w) {
  *w = (int)(pos % (I)W); pos /= (I)W;
  *h = (int)(pos % (I)H); pos /= (I)H;
  *d = (int)(pos % (I)D); pos /= (I)D;
  *n = (int)pos;
}

// acc[i][j] += As[k][ty*4 + i] * Bs[k][tx*4 + j] over the 16 k of one staged chunk, k ascending
__device__ __forceinline__ void chunk_fma(const float (&As)[GK][GT + 1], const float (&Bs)[GK][GT + 1], int ty, int tx,
                                          float (&acc)[4][4]) {
#pragma unroll
  for (int k = 0; k < GK; ++k) {
    float a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
}

__device__ __forceinline__ void flush(float (&tot)[4][4], float (&acc)[4][4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) { tot[i][j] += acc[i][j]; acc[i][j] = 0.f; }
}

// y[opos, co] = sum_{tap, ci} x[n, od*sd - pd + a_d, oh*sh - ph + a_h, ow*sw - pw + a_w, ci] * w[co, tap, ci]
//               (+ bias[co]) (+ residual | * (relu_ref > 0)) (ReLU)
template <typename ST>
__global__ void __launch_bounds__(256) gconv_fprop_kernel(const GconvParams<ST> p) {
  __shared__ float As[GK][GT + 1];
  __shared__ float Bs[GK][GT + 1];
  const t2v_gconv_geom& g = p.g;
  const int tid = threadIdx.x;
  const long long pos0 = (long long)blockIdx.x * GT;
  const int co0 = blockIdx.y * GT;
  const int tx = tid % 16, ty = tid / 16;   // tx -> co, ty -> position
  float acc[4][4] = {}, tot[4][4] = {};
  const int taps = g.kd * g.kh * g.kw;
  // this thread's 4 staging slots: element e = tid + 256*i -> (row = e / GK, k = e % GK)
  int rn[4], rd[4], rh[4], rw[4];
  bool rok[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long pos = pos0 + (tid + 256 * i) / GK;
    rok[i] = pos < p.Po;
    decode_pos(rok[i] ? pos : 0, g.Do, g.Ho, g.Wo, &rn[i], &rd[i], &rh[i], &rw[i]);
  }
  for (int tap = 0; tap < taps; ++tap) {
    const int a_w = tap % g.kw, a_h = (tap / g.kw) % g.kh, a_d = tap / (g.kw * g.kh);
    long long xrow[4];            // offset of the slot's input row for this tap, -1 where it reads zero padding
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int dd = rd[i] * g.sd - g.pd + a_d, hh = rh[i] * g.sh - g.ph + a_h, ww = rw[i] * g.sw - g.pw + a_w;
      xrow[i] = rok[i] && dd >= 0 && dd < g.Di && hh >= 0 && hh < g.Hi && ww >= 0 && ww < g.Wi
                    ? ((((long long)rn[i] * g.Di + dd) * g.Hi + hh) * g.Wi + ww) * g.Cin : -1;
    }
    for (int c0 = 0; c0 < g.Cin; c0 += GK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int e = tid + 256 * i;
        const int r = e / GK, k = e % GK;
        float v = 0.f;
        if (xrow[i] >= 0 && c0 + k < g.Cin) v = bf2f(p.x[xrow[i] + c0 + k]);
        As[k][r] = v;
        float wv = 0.f;
        const int co = co0 + r;
        if (co < g.Cout && c0 + k < g.Cin) wv = bf2f(p.w[((long long)co * taps + tap) * g.Cin + c0 + k]);
        Bs[k][r] = wv;
      }
      __syncthreads();
      chunk_fma(As, Bs, ty, tx, acc);
      __syncthreads();
    }
    flush(tot, acc);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long pos = pos0 + ty * 4 + i;
    if (pos >= p.Po) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = co0 + tx * 4 + j;
      if (co >= g.Cout) continue;
      float v = tot[i][j];
      if (p.bias != nullptr) v += p.bias[co];
      if (p.residual != nullptr) {
        const float r = bf2f(p.residual[pos * g.Cout + co]);
        if (p.relu_mask) v = r > 0.f ? v : 0.f;       // T2V_EPI_RELU_MASK: the pointer is the ReLU reference
        else v += r;
      }
      if (p.relu) v = fmaxf(v, 0.f);
      if (p.out_f32) reinterpret_cast<float*>(p.out)[pos * g.Cout + co] = v;
      else reinterpret_cast<__nv_bfloat16*>(p.out)[pos * g.Cout + co] = f2bf(v);
    }
  }
}

// dx[ipos, ci] = sum_{tap, co : (i + p - a) % s == 0} dy[n, (id+pd-a_d)/sd, ..., co] * w[co, tap, ci]   (+ bias[ci])
template <typename ST>
__global__ void __launch_bounds__(256) gconv_dgrad_kernel(const GconvParams<ST> p) {
  __shared__ float As[GK][GT + 1];
  __shared__ float Bs[GK][GT + 1];
  const t2v_gconv_geom& g = p.g;
  const int tid = threadIdx.x;
  const long long pos0 = (long long)blockIdx.x * GT;
  const int ci0 = blockIdx.y * GT;
  const int tx = tid % 16, ty = tid / 16;
  float acc[4][4] = {}, tot[4][4] = {};
  const int taps = g.kd * g.kh * g.kw;
  int rn[4], rd[4], rh[4], rw[4];
  bool rok[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long pos = pos0 + (tid + 256 * i) / GK;
    rok[i] = pos < p.Pi;
    decode_pos(rok[i] ? pos : 0, g.Di, g.Hi, g.Wi, &rn[i], &rd[i], &rh[i], &rw[i]);
  }
  for (int tap = 0; tap < taps; ++tap) {
    const int a_w = tap % g.kw, a_h = (tap / g.kw) % g.kh, a_d = tap / (g.kw * g.kh);
    long long dyrow[4];           // offset of the slot's dy row for this tap, -1 where no output position reads it
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      dyrow[i] = -1;
      const int td = rd[i] + g.pd - a_d, th = rh[i] + g.ph - a_h, tw = rw[i] + g.pw - a_w;
      if (rok[i] && td >= 0 && th >= 0 && tw >= 0 && td % g.sd == 0 && th % g.sh == 0 && tw % g.sw == 0) {
        const int od = td / g.sd, oh = th / g.sh, ow = tw / g.sw;
        if (od < g.Do && oh < g.Ho && ow < g.Wo)
          dyrow[i] = ((((long long)rn[i] * g.Do + od) * g.Ho + oh) * g.Wo + ow) * g.Cout;
      }
    }
    for (int c0 = 0; c0 < g.Cout; c0 += GK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int e = tid + 256 * i;
        const int r = e / GK, k = e % GK;
        float v = 0.f;
        if (dyrow[i] >= 0 && c0 + k < g.Cout) v = bf2f(p.dy[dyrow[i] + c0 + k]);
        As[k][r] = v;
        float wv = 0.f;
        const int ci = ci0 + r;
        if (ci < g.Cin && c0 + k < g.Cout) wv = bf2f(p.w[((long long)(c0 + k) * taps + tap) * g.Cin + ci]);
        Bs[k][r] = wv;
      }
      __syncthreads();
      chunk_fma(As, Bs, ty, tx, acc);
      __syncthreads();
    }
    flush(tot, acc);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long pos = pos0 + ty * 4 + i;
    if (pos >= p.Pi) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ci = ci0 + tx * 4 + j;
      if (ci >= g.Cin) continue;
      float v = tot[i][j];
      if (p.bias != nullptr) v += p.bias[ci];
      if (p.out_f32) reinterpret_cast<float*>(p.out)[pos * g.Cin + ci] = v;
      else reinterpret_cast<__nv_bfloat16*>(p.out)[pos * g.Cin + ci] = f2bf(v);
    }
  }
}

// dw[co, tap, ci] += sum_opos dy[opos, co] * x[ipos(opos, tap), ci];  grid = (co tiles, ci tiles, taps * splits).
// Three blocks per SM (80 registers): faster on the TGAN layers than two blocks with more registers (DESIGN §5).
template <typename ST>
__global__ void __launch_bounds__(256, 3) gconv_wgrad_kernel(const GconvParams<ST> p) {
  __shared__ float As[GK][GT + 1];   // [pos][co]
  __shared__ float Bs[GK][GT + 1];   // [pos][ci]
  const t2v_gconv_geom& g = p.g;
  const int tid = threadIdx.x;
  const int co0 = blockIdx.x * GT, ci0 = blockIdx.y * GT;
  const int taps = g.kd * g.kh * g.kw;
  const int tap = blockIdx.z % taps, split = blockIdx.z / taps;
  const int a_w = tap % g.kw, a_h = (tap / g.kw) % g.kh, a_d = tap / (g.kw * g.kh);
  const long long per = (p.Po + p.splits - 1) / p.splits;
  const long long pbeg = (long long)split * per, pend = min(p.Po, pbeg + per);
  const int tx = tid % 16, ty = tid / 16;   // tx -> ci, ty -> co
  float acc[4][4] = {}, tot[4][4] = {};
  for (long long q0 = pbeg; q0 < pend; q0 += GK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + 256 * i;
      const int k = e / GT, r = e % GT;         // k = position within the chunk, r = channel
      const long long pos = q0 + k;
      float av = 0.f, bv = 0.f;
      if (pos < pend) {
        int n, od, oh, ow;
        if (pos <= 0x7fffffff) decode_pos((unsigned)pos, g.Do, g.Ho, g.Wo, &n, &od, &oh, &ow);  // 32-bit: cheaper
        else decode_pos(pos, g.Do, g.Ho, g.Wo, &n, &od, &oh, &ow);
        if (co0 + r < g.Cout) av = bf2f(p.dy[pos * g.Cout + co0 + r]);
        const int dd = od * g.sd - g.pd + a_d, hh = oh * g.sh - g.ph + a_h, ww = ow * g.sw - g.pw + a_w;
        if (ci0 + r < g.Cin && dd >= 0 && dd < g.Di && hh >= 0 && hh < g.Hi && ww >= 0 && ww < g.Wi)
          bv = bf2f(p.x[((((long long)n * g.Di + dd) * g.Hi + hh) * g.Wi + ww) * g.Cin + ci0 + r]);
      }
      As[k][r] = av;
      Bs[k][r] = bv;
    }
    __syncthreads();
    chunk_fma(As, Bs, ty, tx, acc);
    __syncthreads();
    if (((q0 - pbeg) & (64 * GK - 1)) == 63 * GK) flush(tot, acc);     // every 64 chunks: bounded FMA chains
  }
  flush(tot, acc);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + ty * 4 + i;
    if (co >= g.Cout) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ci = ci0 + tx * 4 + j;
      if (ci >= g.Cin) continue;
      atomicAdd(p.dw + ((long long)co * taps + tap) * g.Cin + ci, tot[i][j]);
    }
  }
}

static bool gconv_ok(const t2v_gconv_geom* g) {
  if (!g || g->N <= 0 || g->Cin <= 0 || g->Cout <= 0) return false;
  if (g->kd <= 0 || g->kh <= 0 || g->kw <= 0 || g->sd <= 0 || g->sh <= 0 || g->sw <= 0) return false;
  if (g->pd < 0 || g->ph < 0 || g->pw < 0) return false;
  // output extents must be consistent with the convolution arithmetic
  auto oe = [](int i, int k, int s, int p) { return (i + 2 * p - k) / s + 1; };
  if (g->Di + 2 * g->pd < g->kd || g->Hi + 2 * g->ph < g->kh || g->Wi + 2 * g->pw < g->kw) return false;
  return g->Do == oe(g->Di, g->kd, g->sd, g->pd) && g->Ho == oe(g->Hi, g->kh, g->sh, g->ph) &&
         g->Wo == oe(g->Wi, g->kw, g->sw, g->pw);
}

template <typename ST>
static GconvParams<ST> gconv_params(const t2v_gconv_geom* g) {
  GconvParams<ST> p{};
  p.g = *g;
  p.Pi = (long long)g->N * g->Di * g->Hi * g->Wi;
  p.Po = (long long)g->N * g->Do * g->Ho * g->Wo;
  return p;
}

template <typename ST>
static void fprop_run(const t2v_gconv_geom* g, const void* x, const void* w, const float* bias, const void* residual,
                      void* y, uint32_t flags, int out_f32, cudaStream_t s) {
  GconvParams<ST> p = gconv_params<ST>(g);
  p.x = reinterpret_cast<const ST*>(x);
  p.w = reinterpret_cast<const ST*>(w);
  p.bias = bias;
  p.residual = reinterpret_cast<const ST*>(residual);
  p.out = y;
  p.out_f32 = out_f32;
  p.relu = (flags & T2V_EPI_RELU) ? 1 : 0;
  p.relu_mask = (flags & T2V_EPI_RELU_MASK) ? 1 : 0;
  dim3 grid((unsigned)((p.Po + GT - 1) / GT), (unsigned)((g->Cout + GT - 1) / GT), 1);
  gconv_fprop_kernel<ST><<<grid, 256, 0, s>>>(p);
}

template <typename ST>
static void dgrad_run(const t2v_gconv_geom* g, const void* dy, const void* w, const float* bias, void* dx, int out_f32,
                      cudaStream_t s) {
  GconvParams<ST> p = gconv_params<ST>(g);
  p.dy = reinterpret_cast<const ST*>(dy);
  p.w = reinterpret_cast<const ST*>(w);
  p.bias = bias;
  p.out = dx;
  p.out_f32 = out_f32;
  dim3 grid((unsigned)((p.Pi + GT - 1) / GT), (unsigned)((g->Cin + GT - 1) / GT), 1);
  gconv_dgrad_kernel<ST><<<grid, 256, 0, s>>>(p);
}

template <typename ST>
static void wgrad_run(const t2v_gconv_geom* g, const void* dy, const void* x, float* dw, cudaStream_t s) {
  GconvParams<ST> p = gconv_params<ST>(g);
  p.dy = reinterpret_cast<const ST*>(dy);
  p.x = reinterpret_cast<const ST*>(x);
  p.dw = dw;
  const int taps = g->kd * g->kh * g->kw;
  const int base = ((g->Cout + GT - 1) / GT) * ((g->Cin + GT - 1) / GT) * taps;
  long long splits = (4 * 148 + base - 1) / base;
  const long long max_splits = (p.Po + 4 * GK - 1) / (4 * GK);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if ((long long)taps * splits > 65535) splits = 65535 / taps;
  p.splits = (int)splits;
  dim3 grid((unsigned)((g->Cout + GT - 1) / GT), (unsigned)((g->Cin + GT - 1) / GT), (unsigned)(taps * splits));
  gconv_wgrad_kernel<ST><<<grid, 256, 0, s>>>(p);
}

// The launchers of the three directions.  f32 selects fp32 storage of every activation operand (x / w / dy /
// residual), whose output is always fp32; otherwise they are bf16 and T2V_EPI_OUT_F32 (fprop) or out_f32 (dgrad)
// selects an fp32 output.
int gconv_fprop_launch(const t2v_gconv_geom* g, const void* x, const void* w, const float* bias, const void* residual,
                       void* y, uint32_t flags, bool f32, cudaStream_t s) {
  if (!gconv_ok(g) || !x || !w || !y) return T2V_ERR_ARG;
  if (f32) fprop_run<float>(g, x, w, bias, residual, y, flags, 1, s);
  else fprop_run<__nv_bfloat16>(g, x, w, bias, residual, y, flags, (flags & T2V_EPI_OUT_F32) ? 1 : 0, s);
  count_launch();
  return check_last("gconv_fprop");
}

static int gconv_dgrad_launch(const t2v_gconv_geom* g, const void* dy, const void* w, const float* bias, void* dx,
                              int out_f32, bool f32, cudaStream_t s) {
  if (!gconv_ok(g) || !dy || !w || !dx) return T2V_ERR_ARG;
  if (f32) dgrad_run<float>(g, dy, w, bias, dx, 1, s);
  else dgrad_run<__nv_bfloat16>(g, dy, w, bias, dx, out_f32 ? 1 : 0, s);
  count_launch();
  return check_last("gconv_dgrad");
}

int gconv_wgrad_launch(const t2v_gconv_geom* g, const void* dy, const void* x, float* dw, int accumulate, bool f32,
                       cudaStream_t s) {
  if (!gconv_ok(g) || !dy || !x || !dw) return T2V_ERR_ARG;
  if (!accumulate) cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)g->Cout * g->kd * g->kh * g->kw * g->Cin, s);
  if (f32) wgrad_run<float>(g, dy, x, dw, s);
  else wgrad_run<__nv_bfloat16>(g, dy, x, dw, s);
  count_launch();
  return check_last("gconv_wgrad");
}

}  // namespace t2v

using namespace t2v;

static cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {
int t2v_gconv_fprop(const t2v_gconv_geom* g, const void* x, const void* w, const float* bias, void* y,
                    int32_t out_f32, void* stream) {
  return gconv_fprop_launch(g, x, w, bias, nullptr, y, out_f32 ? T2V_EPI_OUT_F32 : 0u, false, as_stream(stream));
}
int t2v_gconv_dgrad(const t2v_gconv_geom* g, const void* dy, const void* w, const float* bias, void* dx,
                    int32_t out_f32, void* stream) {
  return gconv_dgrad_launch(g, dy, w, bias, dx, out_f32, false, as_stream(stream));
}
int t2v_gconv_wgrad(const t2v_gconv_geom* g, const void* dy, const void* x, float* dw, int32_t accumulate,
                    void* stream) {
  return gconv_wgrad_launch(g, dy, x, dw, accumulate, false, as_stream(stream));
}
/* fp32 storage (the 1e-3 parity mode): x / w / dy fp32, output always fp32 */
int t2v_gconv_fprop_f32(const t2v_gconv_geom* g, const void* x, const void* w, const float* bias, void* y,
                        int32_t out_f32, void* stream) {
  (void)out_f32;
  return gconv_fprop_launch(g, x, w, bias, nullptr, y, 0u, true, as_stream(stream));
}
int t2v_gconv_dgrad_f32(const t2v_gconv_geom* g, const void* dy, const void* w, const float* bias, void* dx,
                        int32_t out_f32, void* stream) {
  (void)out_f32;
  return gconv_dgrad_launch(g, dy, w, bias, dx, 1, true, as_stream(stream));
}
int t2v_gconv_wgrad_f32(const t2v_gconv_geom* g, const void* dy, const void* x, float* dw, int32_t accumulate,
                        void* stream) {
  return gconv_wgrad_launch(g, dy, x, dw, accumulate, true, as_stream(stream));
}
}  // extern "C"
