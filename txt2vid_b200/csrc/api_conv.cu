// C-ABI entry points of the convolution engine (declared in include/t2v.h).
#include "t2v_common.cuh"

namespace t2v {
unsigned long long g_launch_count = 0;

bool igemm_fprop_supported(const t2v_conv_geom* g);
bool igemm_wgrad_supported(const t2v_conv_geom* g);
int igemm_fprop_launch(const t2v_conv_geom*, const void*, const void*, const float*, const void*, void*,
                       uint32_t, cudaStream_t);
int igemm_wgrad_launch(const t2v_conv_geom*, const void*, const void*, float*, int, cudaStream_t,
                       const ConvWindow* win = nullptr);
int igemm_fprop_launch_aux(const t2v_conv_geom*, const void*, const void*, const float*, const void*, void*, uint32_t,
                           cudaStream_t, const void*, const void*, int, const LstmEpi* lstm = nullptr,
                           const ConvWindow* win = nullptr);
bool halo_wgrad_supported(const t2v_conv_geom* g);
bool halo_fprop_supported(const t2v_conv_geom* g);
int halo_fprop_launch(const t2v_conv_geom*, const void*, const void*, const float*, const void*, void*,
                      uint32_t, cudaStream_t);
int halo_wgrad_launch(const t2v_conv_geom*, const void*, const void*, float*, int, cudaStream_t, int sd2);
bool halo_sd2_supported(const t2v_conv_geom* g);
int halo_fprop_sd2_launch(const t2v_conv_geom*, const void*, const void*, const float*, void*, uint32_t, cudaStream_t);
int halo_dgrad_sd2_launch(const t2v_conv_geom*, const void*, const void*, const void*, void*, uint32_t, cudaStream_t);
int gconv_fprop_launch(const t2v_gconv_geom*, const void*, const void*, const float*, const void*, void*, uint32_t,
                       bool f32, cudaStream_t);
int gconv_wgrad_launch(const t2v_gconv_geom*, const void*, const void*, float*, int, bool f32, cudaStream_t);
void prof_enable(int on);
void prof_read(double* out, int nkinds);
void prof_next_scale(double s);

__global__ void cast_f32_bf16_kernel(const float* __restrict__ s, __nv_bfloat16* __restrict__ d, long long n) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(s + i);
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(d + i) = o;
  } else {
    for (long long j = i; j < n; ++j) d[j] = f2bf(s[j]);
  }
}
__global__ void cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ s, float* __restrict__ d, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = bf2f(s[i]);
}
// wT[ci][taps-1-tap][co] = w[co][tap][ci]; destination is [CinP][taps][CoutP] (padding pre-zeroed by caller)
__global__ void pack_dgrad_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wT, int Cout,
                                  int taps, int Cin, int CoutP) {
  __shared__ float tile[32][33];
  const int tap = blockIdx.z;
  const int co0 = blockIdx.y * 32, ci0 = blockIdx.x * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int co = co0 + r, ci = ci0 + threadIdx.x;
    tile[r][threadIdx.x] = (co < Cout && ci < Cin) ? w[((long long)co * taps + tap) * Cin + ci] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int ci = ci0 + r, co = co0 + threadIdx.x;
    if (ci < Cin && co < Cout)
      wT[((long long)ci * taps + (taps - 1 - tap)) * CoutP + co] = f2bf(tile[threadIdx.x][r]);
  }
}
// dst bf16 [CoutP][taps][CinP] <- src fp32 [Cout][taps][Cin] (padding pre-zeroed by caller)
__global__ void pack_pad_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst, int taps, int Cin,
                                int CinP, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int ci = (int)(i % Cin);
  const long long r = i / Cin;  // co*taps + tap
  dst[r * CinP + ci] = f2bf(w[i]);
}
// dst fp32 [Cout][taps][Cin] <- src fp32 [CoutP][taps][CinP]
__global__ void unpack_pad_kernel(const float* __restrict__ src, float* __restrict__ dst, int taps, int Cin,
                                  int CinP, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int ci = (int)(i % Cin);
  const long long r = i / Cin;
  dst[i] = src[r * CinP + ci];
}
// Weight gradient of a (1,3,3) convolution computed on position PAIRS (two adjacent w voxels viewed as one voxel
// with twice the channels: 64-byte rows become 128-byte rows): dw2[(pw,co)][a_h*3 + s + 1][(qw,ci)] holds every
// product dy[w = 2u + pw] * x[w + 2s + qw - pw]; the real tap a_w (shift a_w - 1 = 2s + qw - pw) collects two of them.
__global__ void fold_pairs_kernel(const float* __restrict__ dw2, float* __restrict__ dw, int Co, int Ci, int ld2,
                                  int accumulate, int total) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int ci = i % Ci;
  int t = i / Ci;
  const int a_w = t % 3; t /= 3;
  const int a_h = t % 3;
  const int co = t / 3;
  // (s, pw, qw) pairs with 2s + qw - pw == a_w - 1
  const int s0 = 0, pw0 = a_w == 0 ? 1 : 0, qw0 = a_w == 2 ? 1 : (a_w == 1 ? 0 : 0);
  int s1, pw1, qw1;
  if (a_w == 1) { s1 = 0; pw1 = 1; qw1 = 1; }
  else if (a_w == 2) { s1 = 1; pw1 = 1; qw1 = 0; }
  else { s1 = -1; pw1 = 0; qw1 = 1; }
  const float v = dw2[((size_t)(pw0 * Co + co) * 9 + a_h * 3 + s0 + 1) * ld2 + qw0 * Ci + ci] +
                  dw2[((size_t)(pw1 * Co + co) * 9 + a_h * 3 + s1 + 1) * ld2 + qw1 * Ci + ci];
  dw[i] = accumulate ? dw[i] + v : v;
}
}  // namespace t2v

using namespace t2v;

// A stride-1 "same" convolution as a general geometry: the CUDA-core route of the t2v_conv_* entry points.
static t2v_gconv_geom same_geom(const t2v_conv_geom* g) {
  return t2v_gconv_geom{g->N, g->D, g->H, g->W, g->D, g->H, g->W, g->Cin, g->Cout,
                        g->kd, g->kh, g->kw, 1, 1, 1, g->kd / 2, g->kh / 2, g->kw / 2};
}

extern "C" {

int t2v_version(void) { return 100; }
unsigned long long t2v_launch_count(void) { return g_launch_count; }
int t2v_profile_enable(int on) { prof_enable(on); return T2V_OK; }
int t2v_profile_read(double* host_out6) { prof_read(host_out6, 2); return T2V_OK; }
int t2v_profile_read4(double* host_out12) { prof_read(host_out12, 4); return T2V_OK; }
int t2v_profile_read6(double* host_out18) { prof_read(host_out18, 6); return T2V_OK; }
int t2v_profile_next_scale(double real_fraction) { prof_next_scale(real_fraction); return T2V_OK; }

int t2v_conv_fprop(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                   const void* residual, void* y, uint32_t epi_flags, int algo, void* stream) {
  if (!g || !x || !w || !y) return T2V_ERR_ARG;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const t2v_gconv_geom gg = same_geom(g);
  if (epi_flags & T2V_EPI_IN_F32) {             // fp32 parity mode: fp32 operands on the CUDA-core FFMA kernel
    if (algo == T2V_ALGO_TC || algo == T2V_ALGO_TC_GENERIC) return T2V_ERR_ARG;
    if ((epi_flags & T2V_EPI_RELU_MASK) && !residual) return T2V_ERR_ARG;
    return gconv_fprop_launch(&gg, x, w, bias, residual, y, epi_flags, true, s);
  }
  const bool tc_ok = igemm_fprop_supported(g);
  if ((algo == T2V_ALGO_TC || algo == T2V_ALGO_TC_GENERIC) && !tc_ok) return T2V_ERR_ARG;
  if ((epi_flags & T2V_EPI_RELU_MASK) && (algo == T2V_ALGO_SIMT || !tc_ok || !residual)) return T2V_ERR_ARG;
  if (algo == T2V_ALGO_SIMT || !tc_ok) return gconv_fprop_launch(&gg, x, w, bias, residual, y, epi_flags, false, s);
  if (algo != T2V_ALGO_TC_GENERIC && halo_fprop_supported(g)) return halo_fprop_launch(g, x, w, bias, residual, y, epi_flags, s);
  return igemm_fprop_launch(g, x, w, bias, residual, y, epi_flags, s);
}

int t2v_conv_dgrad(const t2v_conv_geom* g, const void* dy, const void* wT, const void* residual,
                   void* dx, uint32_t epi_flags, int algo, void* stream) {
  if (!g) return T2V_ERR_ARG;
  t2v_conv_geom gt = *g;
  gt.Cin = g->Cout;
  gt.Cout = g->Cin;
  return t2v_conv_fprop(&gt, dy, wT, nullptr, residual, dx, epi_flags, algo, stream);
}

int t2v_conv_wgrad(const t2v_conv_geom* g, const void* dy, const void* x, float* dw, int accumulate,
                   int algo, void* stream) {
  if (!g || !dy || !x || !dw) return T2V_ERR_ARG;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const t2v_gconv_geom gg = same_geom(g);
  if (algo == T2V_ALGO_SIMT_F32) return gconv_wgrad_launch(&gg, dy, x, dw, accumulate, true, s);   // fp32 dy / x
  const bool tc_ok = igemm_wgrad_supported(g);
  if ((algo == T2V_ALGO_TC || algo == T2V_ALGO_TC_GENERIC) && !tc_ok) return T2V_ERR_ARG;
  if (algo == T2V_ALGO_SIMT || !tc_ok) return gconv_wgrad_launch(&gg, dy, x, dw, accumulate, false, s);
  if (algo != T2V_ALGO_TC_GENERIC && halo_wgrad_supported(g)) return halo_wgrad_launch(g, dy, x, dw, accumulate, s, 0);
  return igemm_wgrad_launch(g, dy, x, dw, accumulate, s);
}

static bool fill_window(ConvWindow* cw, const int32_t* w9) {
  if (!w9) return false;
  cw->iD = w9[0]; cw->iH = w9[1]; cw->iW = w9[2];
  cw->lo_d = w9[3]; cw->hi_d = w9[4]; cw->lo_h = w9[5]; cw->hi_h = w9[6]; cw->lo_w = w9[7]; cw->hi_w = w9[8];
  return cw->iD > 0 && cw->iH > 0 && cw->iW > 0;
}

int t2v_conv_fprop_win(const t2v_conv_geom* g, const int32_t* win9, const void* x, const void* w, const float* bias,
                       void* y, uint32_t epi_flags, void* stream) {
  ConvWindow cw;
  if (!g || !x || !w || !y || !fill_window(&cw, win9)) return T2V_ERR_ARG;
  if (epi_flags & ~(T2V_EPI_RELU | T2V_EPI_OUT_F32)) return T2V_ERR_ARG;
  return igemm_fprop_launch_aux(g, x, w, bias, nullptr, y, epi_flags, reinterpret_cast<cudaStream_t>(stream), nullptr,
                                nullptr, 0, nullptr, &cw);
}

int t2v_conv_wgrad_win(const t2v_conv_geom* g, const int32_t* win9, const void* dy, const void* x, float* dw,
                       int accumulate, void* stream) {
  ConvWindow cw;
  if (!g || !dy || !x || !dw || !fill_window(&cw, win9)) return T2V_ERR_ARG;
  return igemm_wgrad_launch(g, dy, x, dw, accumulate, reinterpret_cast<cudaStream_t>(stream), &cw);
}

int t2v_conv_fprop_skip(const t2v_conv_geom* g, const void* x, const void* w, const float* bias, const void* x2,
                        const void* w2, int32_t Cin2, void* y, uint32_t epi_flags, void* stream) {
  if (!g || !x || !w || !x2 || !w2 || !y) return T2V_ERR_ARG;
  if (!igemm_fprop_supported(g) || g->Cin % 64 || Cin2 % 64) return T2V_ERR_ARG;
  return igemm_fprop_launch_aux(g, x, w, bias, nullptr, y, epi_flags, reinterpret_cast<cudaStream_t>(stream), x2, w2,
                                Cin2);
}

int t2v_conv_lstm_step(const t2v_conv_geom* g, const void* x, const void* w_il, const float* bias_il,
                       const float* c_prev, float* gates, float* c_out, void* h_out, void* h_merged, int32_t t,
                       int32_t steps, void* stream) {
  if (!g || !x || !w_il || !bias_il || !gates || !c_out || !h_out || !h_merged) return T2V_ERR_ARG;
  LstmEpi e{c_prev, c_out, gates, h_out, h_merged, t, steps};
  return igemm_fprop_launch_aux(g, x, w_il, bias_il, nullptr, h_out, 0u, reinterpret_cast<cudaStream_t>(stream),
                                nullptr, nullptr, 0, &e);
}

int t2v_conv_sd2_supported(const t2v_conv_geom* g) { return (g && halo_sd2_supported(g)) ? 1 : 0; }

int t2v_conv_fprop_sd2(const t2v_conv_geom* g, const void* x, const void* w, const float* bias, void* y,
                       uint32_t epi_flags, void* stream) {
  if (!g || !x || !w || !y) return T2V_ERR_ARG;
  return halo_fprop_sd2_launch(g, x, w, bias, y, epi_flags, reinterpret_cast<cudaStream_t>(stream));
}

int t2v_conv_dgrad_sd2(const t2v_conv_geom* g, const void* dy, const void* wT, const void* relu_ref, void* dx,
                       uint32_t epi_flags, void* stream) {
  if (!g || !dy || !wT || !dx) return T2V_ERR_ARG;
  return halo_dgrad_sd2_launch(g, dy, wT, relu_ref, dx, epi_flags, reinterpret_cast<cudaStream_t>(stream));
}

int t2v_conv_wgrad_sd2(const t2v_conv_geom* g, const void* dy, const void* x, float* dw, int accumulate,
                       void* stream) {
  if (!g || !dy || !x || !dw) return T2V_ERR_ARG;
  return halo_wgrad_launch(g, dy, x, dw, accumulate, reinterpret_cast<cudaStream_t>(stream), 1);
}

int t2v_wgrad_fold_pairs(const float* dw2, float* dw, int32_t Cout, int32_t Cin, int32_t accumulate, void* stream) {
  if (!dw2 || !dw || Cout <= 0 || Cin <= 0) return T2V_ERR_ARG;
  const int total = Cout * 9 * Cin;
  fold_pairs_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      dw2, dw, Cout, Cin, 2 * Cin, accumulate ? 1 : 0, total);
  count_launch();
  return check_last("fold_pairs");
}

int t2v_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream) {
  if (n <= 0) return T2V_OK;
  const long long thr = (n + 3) / 4;
  cast_f32_bf16_kernel<<<(unsigned)((thr + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  count_launch();
  return check_last("cast");
}
int t2v_cast_bf16_to_f32(const void* src, float* dst, int64_t n, void* stream) {
  if (n <= 0) return T2V_OK;
  cast_bf16_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(src), dst, n);
  count_launch();
  return check_last("cast");
}
int t2v_pack_dgrad_weight(const float* w, void* wT, int32_t Cout, int32_t taps, int32_t Cin, int32_t CoutP,
                          void* stream) {
  dim3 grid((Cin + 31) / 32, (Cout + 31) / 32, taps), block(32, 8);
  pack_dgrad_kernel<<<grid, block, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      w, reinterpret_cast<__nv_bfloat16*>(wT), Cout, taps, Cin, CoutP);
  count_launch();
  return check_last("pack_dgrad");
}
int t2v_pack_weight_padded(const float* w, void* dst, int32_t Cout, int32_t taps, int32_t Cin, int32_t CinP,
                           void* stream) {
  const long long total = (long long)Cout * taps * Cin;
  if (total == 0) return T2V_OK;
  pack_pad_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      w, reinterpret_cast<__nv_bfloat16*>(dst), taps, Cin, CinP, total);
  count_launch();
  return check_last("pack_pad");
}
int t2v_unpack_wgrad_padded(const float* src, float* dst, int32_t Cout, int32_t taps, int32_t Cin, int32_t CinP,
                            void* stream) {
  const long long total = (long long)Cout * taps * Cin;
  if (total == 0) return T2V_OK;
  unpack_pad_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      src, dst, taps, Cin, CinP, total);
  count_launch();
  return check_last("unpack_pad");
}

}  // extern "C"
