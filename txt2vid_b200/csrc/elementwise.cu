// HBM-bound kernels of the TGANv2 training step: activation / pooling / normalisation / layout /
// index / reduction work on channels-last bf16 tensors.  One pass over the data each, 128-bit
// accesses where the channel count allows (C % 8 == 0), fp32 math.
//
// Reference call sites (txt2vid/...): ReLU models/layers.py:172,176,230,232,250; AvgPool
// layers.py:202-217 + resnet3d.py:16,18; nn.Upsample layers.py:168,180; BatchNorm2d(train)
// layers.py:171,175,249; tanh layers.py:252; torch.sum(x,[2,3,4]) resnet3d.py:48; Subsample
// layers.py:106-111; F.interpolate gan/trainer.py:149.
#include "t2v_common.cuh"

namespace t2v {

static inline unsigned blocks_for(long long n, int per_block) {
  long long b = (n + per_block - 1) / per_block;
  if (b < 1) b = 1;
  return (unsigned)b;
}

struct V8 { float f[8]; };
T2V_DEVINL V8 ld8(const __nv_bfloat16* p) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  V8 r;
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  r.f[0] = a.x; r.f[1] = a.y; r.f[2] = b.x; r.f[3] = b.y; r.f[4] = c.x; r.f[5] = c.y; r.f[6] = d.x; r.f[7] = d.y;
  return r;
}
T2V_DEVINL void st8(__nv_bfloat16* p, const V8& v) {
  *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(v.f[0], v.f[1]), pack_bf16x2(v.f[2], v.f[3]),
                                            pack_bf16x2(v.f[4], v.f[5]), pack_bf16x2(v.f[6], v.f[7]));
}

// fp32 storage overloads (the typed kernels of elementwise_typed.inc are instantiated for both)
template <typename T> T2V_DEVINL T cvt_store(float v);
template <> T2V_DEVINL __nv_bfloat16 cvt_store<__nv_bfloat16>(float v) { return f2bf(v); }
template <> T2V_DEVINL float cvt_store<float>(float v) { return v; }
T2V_DEVINL V8 ld8(const float* p) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  V8 r;
  r.f[0] = a.x; r.f[1] = a.y; r.f[2] = a.z; r.f[3] = a.w; r.f[4] = b.x; r.f[5] = b.y; r.f[6] = b.z; r.f[7] = b.w;
  return r;
}
T2V_DEVINL void st8(float* p, const V8& v) {
  *reinterpret_cast<float4*>(p) = make_float4(v.f[0], v.f[1], v.f[2], v.f[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v.f[4], v.f[5], v.f[6], v.f[7]);
}

// RGB clip fp32 (N, 3, S) -> bf16 (N, S, 16) and / or bf16 (N, S, 4) (zero padded), one thread per voxel:
// the discriminator's input conversion (16-channel rows for the TMA-fed skip path, 4-channel rows for the gather of
// the direct stem kernel); 12 B read, 8 + 32 B written per voxel in 8 / 16-byte stores
__global__ void rgb_to_cl_kernel(const float* __restrict__ x, uint4* __restrict__ y16, uint2* __restrict__ y4,
                                 long long S, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long n = i / S, s = i - n * S;
  const float* px = x + n * 3 * S + s;
  const uint2 v = make_uint2(pack_bf16x2(px[0], px[S]), pack_bf16x2(px[2 * S], 0.f));
  if (y4 != nullptr) y4[i] = v;
  if (y16 != nullptr) {
    y16[2 * i] = make_uint4(v.x, v.y, 0u, 0u);
    y16[2 * i + 1] = make_uint4(0u, 0u, 0u, 0u);
  }
}

// BatchNorm finalize (storage-type independent)
// mean / invstd / fused scale+shift, running-stat update (momentum, unbiased variance)
__global__ void bn_finalize_kernel(const float* __restrict__ stats, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float* __restrict__ mean_invstd,
                                   float* __restrict__ scale_shift, int C, float count, float eps, float momentum) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float mean = stats[c] / count;
  float var = stats[C + c] / count - mean * mean;
  var = fmaxf(var, 0.f);
  const float invstd = rsqrtf(var + eps);
  mean_invstd[c] = mean;
  mean_invstd[C + c] = invstd;
  const float sc = gamma[c] * invstd;
  scale_shift[c] = sc;
  scale_shift[C + c] = beta[c] - mean * sc;
  if (running_mean != nullptr) {
    const float unbiased = count > 1.f ? var * count / (count - 1.f) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * unbiased;
  }
}

// ------------------------------------------------------------------------------------ index kernels (bit-exact)
// Frame gather on merged-frame CL maps: out frame (b', t') <- in frame (sn*b', bt + st*t'); 16-byte units
__global__ void gather_frames_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int T, int To, int sn,
                                     int st, int bt_host, const int* __restrict__ bt_dev, long long frame_u4,
                                     long long total, int scatter) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int bt = bt_dev ? *bt_dev : bt_host;
  const long long e = i % frame_u4;
  const long long fo = i / frame_u4;
  const long long bo = fo / To, to = fo % To;
  const long long fi = (bo * sn) * T + bt + to * st;
  if (scatter) y[fi * frame_u4 + e] = x[i];       // x = grad of gathered, y = zero-filled grad of source
  else y[i] = x[fi * frame_u4 + e];
}
// x fp32 (B,C,T,H,W) -> y (Bo,C,To,Ho,Wo): y[b,c,t,h,w] = x[b*sn, c, bt + t*st, floor(h*H/Ho), floor(w*W/Wo)]
__global__ void pyramid_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int C, int T, int H, int W,
                               int Bo, int To, int Ho, int Wo, int sn, int st, int bt_host,
                               const int* __restrict__ bt_dev, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int bt = bt_dev ? *bt_dev : bt_host;
  long long t = i;
  const int w = (int)(t % Wo); t /= Wo;
  const int h = (int)(t % Ho); t /= Ho;
  const int f = (int)(t % To); t /= To;
  const int c = (int)(t % C); t /= C;
  const long long b = t;
  const int hs = (int)(((long long)h * H) / Ho), ws = (int)(((long long)w * W) / Wo);
  y[i] = x[((((b * sn) * C + c) * T + bt + (long long)f * st) * H + hs) * W + ws];
}

// ------------------------------------------------------------------------------------ Adam (multi-tensor)
struct AdamChunk {
  static constexpr int kMax = 48;
  float* p[kMax];
  const float* g[kMax];
  float* m[kMax];
  float* v[kMax];
  long long n[kMax];
  int count;
};
// dyn (optional, device): {lr / (1 - b1^t), 1 / sqrt(1 - b2^t)} for CUDA-graph replays, where the step
// count cannot be a baked-in kernel argument
__global__ void adam_kernel(const AdamChunk ch, float lr, float b1, float b2, float eps, float bc1, float bc2,
                            float grad_scale, const float* __restrict__ dyn) {
  const int t = blockIdx.y;
  if (t >= ch.count) return;
  float* p = ch.p[t];
  const float* g = ch.g[t];
  float* m = ch.m[t];
  float* v = ch.v[t];
  const long long n = ch.n[t];
  const float step = dyn ? dyn[0] : lr / bc1;
  const float inv_sqrt_bc2 = dyn ? dyn[1] : rsqrtf(bc2);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * grad_scale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= step * mi / (sqrtf(vi) * inv_sqrt_bc2 + eps);
  }
}

// ------------------------------------------------------------------------------------ multi-tensor copy
struct CopyChunk {
  static constexpr int kMax = 96;
  const float* src[kMax];
  float* dst[kMax];
  long long n[kMax];
  int count;
};
__global__ void multi_copy_kernel(const CopyChunk ch) {
  const int t = blockIdx.y;
  if (t >= ch.count) return;
  const float* s = ch.src[t];
  float* d = ch.dst[t];
  const long long n = ch.n[t];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = s[i];
}

}  // namespace t2v

#define ST __nv_bfloat16
#define NS ew_bf16
#define SFX(n) n
#include "elementwise_typed.inc"
#undef ST
#undef NS
#undef SFX
#define ST float
#define NS ew_f32
#define SFX(n) n##_f32
#include "elementwise_typed.inc"
#undef ST
#undef NS
#undef SFX

using namespace t2v;
#define STREAM reinterpret_cast<cudaStream_t>(stream)
extern "C" {
int t2v_rgb_to_cl(const float* x, void* y16, void* y4, int64_t N, int64_t S, void* stream) {
  const long long total = N * S;
  if (total == 0 || (!y16 && !y4)) return T2V_OK;
  rgb_to_cl_kernel<<<blocks_for(total, 256), 256, 0, STREAM>>>(x, reinterpret_cast<uint4*>(y16),
                                                               reinterpret_cast<uint2*>(y4), S, total);
  count_launch();
  return check_last("rgb_to_cl");
}
int t2v_bn_finalize(const float* stats, const float* gamma, const float* beta, float* running_mean,
                    float* running_var, float* mean_invstd, float* scale_shift, int32_t C, int64_t count,
                    float eps, float momentum, void* stream) {
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, STREAM>>>(stats, gamma, beta, running_mean, running_var, mean_invstd,
                                                          scale_shift, C, (float)count, eps, momentum);
  count_launch();
  return check_last("bn_finalize");
}
int t2v_gather_frames(const void* x, void* y, int32_t B, int32_t T, int64_t frame_bytes, int32_t sn, int32_t st,
                      int32_t bt, const int32_t* bt_dev, int32_t scatter, void* stream) {
  if (frame_bytes % 16 || bt < 0) return T2V_ERR_ARG;
  const int Bo = (B + sn - 1) / sn;
  const int To = T > bt ? (T - bt + st - 1) / st : 0;
  const long long fu4 = frame_bytes / 16;
  if (scatter) cudaMemsetAsync(y, 0, (size_t)B * T * frame_bytes, STREAM);
  const long long total = (long long)Bo * To * fu4;
  if (total == 0) return T2V_OK;
  gather_frames_kernel<<<blocks_for(total, 256), 256, 0, STREAM>>>(reinterpret_cast<const uint4*>(x),
                                                                   reinterpret_cast<uint4*>(y), T, To, sn, st, bt, bt_dev,
                                                                   fu4, total, scatter);
  count_launch();
  return check_last("gather_frames");
}
int t2v_pyramid_level(const float* x, float* y, const int32_t* in_shape, int32_t Ho, int32_t Wo, int32_t sn,
                      int32_t st, int32_t bt, const int32_t* bt_dev, void* stream) {
  const int B = in_shape[0], C = in_shape[1], T = in_shape[2], H = in_shape[3], W = in_shape[4];
  if (sn < 1 || st < 1 || bt < 0) return T2V_ERR_ARG;
  const int Bo = (B + sn - 1) / sn;
  const int To = T > bt ? (T - bt + st - 1) / st : 0;
  const long long total = (long long)Bo * C * To * Ho * Wo;
  if (total == 0) return T2V_OK;
  pyramid_kernel<<<blocks_for(total, 256), 256, 0, STREAM>>>(x, y, B, C, T, H, W, Bo, To, Ho, Wo, sn, st, bt, bt_dev,
                                                             total);
  count_launch();
  return check_last("pyramid_level");
}
int t2v_adam_step(int32_t count, float* const* host_params, const float* const* host_grads, float* const* host_m,
                  float* const* host_v, const int64_t* host_sizes, float lr, float beta1, float beta2, float eps,
                  int32_t step, float grad_scale, const float* dyn_dev, void* stream) {
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  for (int base = 0; base < count; base += AdamChunk::kMax) {
    AdamChunk ch;
    ch.count = count - base < AdamChunk::kMax ? count - base : AdamChunk::kMax;
    long long maxn = 0;
    for (int i = 0; i < ch.count; ++i) {
      ch.p[i] = host_params[base + i];
      ch.g[i] = host_grads[base + i];
      ch.m[i] = host_m[base + i];
      ch.v[i] = host_v[base + i];
      ch.n[i] = host_sizes[base + i];
      if (ch.n[i] > maxn) maxn = ch.n[i];
    }
    long long bx = (maxn + 256 * 4 - 1) / (256 * 4);
    if (bx > 2048) bx = 2048;
    if (bx < 1) bx = 1;
    dim3 grid((unsigned)bx, ch.count, 1);
    adam_kernel<<<grid, 256, 0, STREAM>>>(ch, lr, beta1, beta2, eps, bc1, bc2, grad_scale, dyn_dev);
    count_launch();
  }
  return check_last("adam_step");
}
int t2v_multi_copy(int32_t count, const float* const* host_src, float* const* host_dst, const int64_t* host_sizes,
                   void* stream) {
  for (int base = 0; base < count; base += CopyChunk::kMax) {
    CopyChunk ch;
    ch.count = count - base < CopyChunk::kMax ? count - base : CopyChunk::kMax;
    long long maxn = 0;
    for (int i = 0; i < ch.count; ++i) {
      ch.src[i] = host_src[base + i];
      ch.dst[i] = host_dst[base + i];
      ch.n[i] = host_sizes[base + i];
      if (ch.n[i] > maxn) maxn = ch.n[i];
    }
    long long bx = (maxn + 256 * 4 - 1) / (256 * 4);
    if (bx > 1024) bx = 1024;
    if (bx < 1) bx = 1;
    multi_copy_kernel<<<dim3((unsigned)bx, ch.count, 1), 256, 0, STREAM>>>(ch);
    count_launch();
  }
  return check_last("multi_copy");
}
}  // extern "C"
