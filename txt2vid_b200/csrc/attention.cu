// Fused core of the SA-GAN non-local block (txt2vid/models/layers.py:23-36 2-D, :52-68 3-D):
//     phi_p = maxpool_{1x2x2}(phi),  g_p = maxpool_{1x2x2}(g)
//     beta  = softmax_k(theta . phi_p^T)            (P queries x Kp keys per map, Kp = P/4)
//     o     = beta . g_p
// in ONE kernel per direction: the (P x Kp) attention matrix (1 MB fp32 per 32x32 map, 1 GB per step at batch
// 1024) never exists in memory.  The 1x1 convolutions around it (theta, phi, g, o) run on the tcgen05 engine.
// HBM-bound: algorithmic bytes = theta + phi + g + o rows (bf16, padded channels).
//
// Forward : thread = one query; pooled keys/values of the map live in shared memory (fp32).
// Backward: phase A (thread = query): softmax statistics, D_q = sum_j beta_j dbeta_j, d theta;
//           phase B (thread = key): d phi_p, d g_p summed over the queries, routed to the arg-max voxel of each
//           2x2 pooling window (the other three voxels get zeros).
// First-order only: the discriminator's block sits on the gradient-penalty path (double backward) and keeps the
// composite formulation of ops.nonlocal_block.
#include <cstdlib>

#include "t2v_common.cuh"

namespace t2v {

static constexpr int kMaxC8 = 8, kMaxC2 = 16;

struct AttnParams {
  int N, D, H, W, c8, c2, C8p, C2p;   // real and padded (memory) channel counts
  int P, Kp, Hp, Wp;
  const __nv_bfloat16* theta; const __nv_bfloat16* phi; const __nv_bfloat16* g;
  __nv_bfloat16* o;
  const __nv_bfloat16* dout;
  __nv_bfloat16* dtheta; __nv_bfloat16* dphi; __nv_bfloat16* dg;
};

// pooled key k of map n: window voxels and the max / arg-max over them, channel c
__device__ __forceinline__ void pooled_window(const AttnParams& p, int k, int* pos4) {
  const int wp = k % p.Wp, hp = (k / p.Wp) % p.Hp, d = k / (p.Wp * p.Hp);
  const int base = (d * p.H + 2 * hp) * p.W + 2 * wp;
  pos4[0] = base; pos4[1] = base + 1; pos4[2] = base + p.W; pos4[3] = base + p.W + 1;
}

__device__ __forceinline__ void build_keys(const AttnParams& p, long long map0, float* s_phi, float* s_g,
                                           unsigned char* s_aphi, unsigned char* s_ag) {
  for (int k = threadIdx.x; k < p.Kp; k += blockDim.x) {
    int pos4[4];
    pooled_window(p, k, pos4);
    for (int c = 0; c < p.c8; ++c) {
      float best = -INFINITY; int arg = 0;
      for (int j = 0; j < 4; ++j) {
        const float v = bf2f(p.phi[(map0 + pos4[j]) * p.C8p + c]);
        if (v > best) { best = v; arg = j; }
      }
      s_phi[k * p.c8 + c] = best;
      if (s_aphi) s_aphi[k * p.c8 + c] = (unsigned char)arg;
    }
    for (int c = 0; c < p.c2; ++c) {
      float best = -INFINITY; int arg = 0;
      for (int j = 0; j < 4; ++j) {
        const float v = bf2f(p.g[(map0 + pos4[j]) * p.C2p + c]);
        if (v > best) { best = v; arg = j; }
      }
      s_g[k * p.c2 + c] = best;
      if (s_ag) s_ag[k * p.c2 + c] = (unsigned char)arg;
    }
  }
}

__global__ void __launch_bounds__(256) attn_fwd_kernel(const AttnParams p) {
  extern __shared__ float smem_f[];
  float* s_phi = smem_f;                       // [Kp][c8]
  float* s_g = s_phi + p.Kp * p.c8;            // [Kp][c2]
  const long long map0 = (long long)blockIdx.x * p.P;
  build_keys(p, map0, s_phi, s_g, nullptr, nullptr);
  __syncthreads();
  const int q = blockIdx.y * blockDim.x + threadIdx.x;
  if (q >= p.P) return;
  float th[kMaxC8];
#pragma unroll
  for (int c = 0; c < kMaxC8; ++c) th[c] = c < p.c8 ? bf2f(p.theta[(map0 + q) * p.C8p + c]) : 0.f;
  float m = -INFINITY;
  for (int k = 0; k < p.Kp; ++k) {
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) s = fmaf(th[c], s_phi[k * p.c8 + c], s);
    m = fmaxf(m, s);
  }
  float l = 0.f, acc[kMaxC2];
#pragma unroll
  for (int c = 0; c < kMaxC2; ++c) acc[c] = 0.f;
  for (int k = 0; k < p.Kp; ++k) {
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) s = fmaf(th[c], s_phi[k * p.c8 + c], s);
    const float e = __expf(s - m);
    l += e;
#pragma unroll
    for (int c = 0; c < kMaxC2; ++c) if (c < p.c2) acc[c] = fmaf(e, s_g[k * p.c2 + c], acc[c]);
  }
  const float inv = 1.f / l;
  __nv_bfloat16* orow = p.o + (map0 + q) * p.C2p;
  for (int c = 0; c < p.C2p; ++c) orow[c] = f2bf(c < p.c2 ? acc[c < kMaxC2 ? c : 0] * inv : 0.f);
}

// one CTA per map
__global__ void __launch_bounds__(256) attn_bwd_kernel(const AttnParams p) {
  extern __shared__ float smem_f[];
  float* s_phi = smem_f;                              // [Kp][c8]
  float* s_g = s_phi + p.Kp * p.c8;                   // [Kp][c2]
  float* s_th = s_g + p.Kp * p.c2;                    // [P][c8]
  float* s_do = s_th + p.P * p.c8;                    // [P][c2]
  float* s_m = s_do + p.P * p.c2;                     // [P] row max
  float* s_il = s_m + p.P;                            // [P] 1 / row sum
  float* s_dq = s_il + p.P;                           // [P] D_q
  unsigned char* s_aphi = reinterpret_cast<unsigned char*>(s_dq + p.P);   // [Kp][c8]
  unsigned char* s_ag = s_aphi + p.Kp * p.c8;                              // [Kp][c2]
  const long long map0 = (long long)blockIdx.x * p.P;
  build_keys(p, map0, s_phi, s_g, s_aphi, s_ag);
  for (int i = threadIdx.x; i < p.P * p.c8; i += blockDim.x)
    s_th[i] = bf2f(p.theta[(map0 + i / p.c8) * p.C8p + i % p.c8]);
  for (int i = threadIdx.x; i < p.P * p.c2; i += blockDim.x)
    s_do[i] = bf2f(p.dout[(map0 + i / p.c2) * p.C2p + i % p.c2]);
  __syncthreads();
  // ---- phase A: per query
  for (int q = threadIdx.x; q < p.P; q += blockDim.x) {
    float th[kMaxC8], dy[kMaxC2];
#pragma unroll
    for (int c = 0; c < kMaxC8; ++c) th[c] = c < p.c8 ? s_th[q * p.c8 + c] : 0.f;
#pragma unroll
    for (int c = 0; c < kMaxC2; ++c) dy[c] = c < p.c2 ? s_do[q * p.c2 + c] : 0.f;
    float m = -INFINITY;
    for (int k = 0; k < p.Kp; ++k) {
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) s = fmaf(th[c], s_phi[k * p.c8 + c], s);
      m = fmaxf(m, s);
    }
    float l = 0.f, dq = 0.f;
    for (int k = 0; k < p.Kp; ++k) {
      float s = 0.f, db = 0.f;
#pragma unroll
      for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) s = fmaf(th[c], s_phi[k * p.c8 + c], s);
#pragma unroll
      for (int c = 0; c < kMaxC2; ++c) if (c < p.c2) db = fmaf(dy[c], s_g[k * p.c2 + c], db);
      const float e = __expf(s - m);
      l += e;
      dq = fmaf(e, db, dq);
    }
    const float il = 1.f / l;
    dq *= il;
    float dth[kMaxC8];
#pragma unroll
    for (int c = 0; c < kMaxC8; ++c) dth[c] = 0.f;
    for (int k = 0; k < p.Kp; ++k) {
      float s = 0.f, db = 0.f;
#pragma unroll
      for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) s = fmaf(th[c], s_phi[k * p.c8 + c], s);
#pragma unroll
      for (int c = 0; c < kMaxC2; ++c) if (c < p.c2) db = fmaf(dy[c], s_g[k * p.c2 + c], db);
      const float ds = __expf(s - m) * il * (db - dq);
#pragma unroll
      for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) dth[c] = fmaf(ds, s_phi[k * p.c8 + c], dth[c]);
    }
    s_m[q] = m; s_il[q] = il; s_dq[q] = dq;
    __nv_bfloat16* drow = p.dtheta + (map0 + q) * p.C8p;
    for (int c = 0; c < p.C8p; ++c) drow[c] = f2bf(c < p.c8 ? dth[c < kMaxC8 ? c : 0] : 0.f);
  }
  __syncthreads();
  // ---- phase B: per key
  for (int k = threadIdx.x; k < p.Kp; k += blockDim.x) {
    float ph[kMaxC8], gk[kMaxC2], dph[kMaxC8], dgk[kMaxC2];
#pragma unroll
    for (int c = 0; c < kMaxC8; ++c) { ph[c] = c < p.c8 ? s_phi[k * p.c8 + c] : 0.f; dph[c] = 0.f; }
#pragma unroll
    for (int c = 0; c < kMaxC2; ++c) { gk[c] = c < p.c2 ? s_g[k * p.c2 + c] : 0.f; dgk[c] = 0.f; }
    for (int q = 0; q < p.P; ++q) {
      float s = 0.f, db = 0.f;
#pragma unroll
      for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) s = fmaf(s_th[q * p.c8 + c], ph[c], s);
#pragma unroll
      for (int c = 0; c < kMaxC2; ++c) if (c < p.c2) db = fmaf(s_do[q * p.c2 + c], gk[c], db);
      const float beta = __expf(s - s_m[q]) * s_il[q];
      const float ds = beta * (db - s_dq[q]);
#pragma unroll
      for (int c = 0; c < kMaxC8; ++c) if (c < p.c8) dph[c] = fmaf(ds, s_th[q * p.c8 + c], dph[c]);
#pragma unroll
      for (int c = 0; c < kMaxC2; ++c) if (c < p.c2) dgk[c] = fmaf(beta, s_do[q * p.c2 + c], dgk[c]);
    }
    int pos4[4];
    pooled_window(p, k, pos4);
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat16* r1 = p.dphi + (map0 + pos4[j]) * p.C8p;
      for (int c = 0; c < p.C8p; ++c)
        r1[c] = f2bf((c < p.c8 && s_aphi[k * p.c8 + c] == j) ? dph[c < kMaxC8 ? c : 0] : 0.f);
      __nv_bfloat16* r2 = p.dg + (map0 + pos4[j]) * p.C2p;
      for (int c = 0; c < p.C2p; ++c)
        r2[c] = f2bf((c < p.c2 && s_ag[k * p.c2 + c] == j) ? dgk[c < kMaxC2 ? c : 0] : 0.f);
    }
  }
}


// ------------------------------------------------------------------------------------------------------------
// Fast path for the generator's block (C = 32: 4 query/key channels, 16 value channels, rows padded to 16 bf16):
// compile-time channel counts, keys / values in shared memory as float4 (every inner-loop load is one broadcast
// LDS.128), two queries per thread so that each key row feeds two dot products.  Same math as the generic kernels.
struct Key4 { float4 v; };

__device__ __forceinline__ float4 ld4_bf16(const __nv_bfloat16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void ld16_bf16(const __nv_bfloat16* p, float4* out) {
  const uint4 u0 = reinterpret_cast<const uint4*>(p)[0], u1 = reinterpret_cast<const uint4*>(p)[1];
  float2 a = unpack_bf16x2(u0.x), b = unpack_bf16x2(u0.y), c = unpack_bf16x2(u0.z), d = unpack_bf16x2(u0.w);
  out[0] = make_float4(a.x, a.y, b.x, b.y); out[1] = make_float4(c.x, c.y, d.x, d.y);
  a = unpack_bf16x2(u1.x); b = unpack_bf16x2(u1.y); c = unpack_bf16x2(u1.z); d = unpack_bf16x2(u1.w);
  out[2] = make_float4(a.x, a.y, b.x, b.y); out[3] = make_float4(c.x, c.y, d.x, d.y);
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}
__device__ __forceinline__ float dot16(const float4* a, const float4* b) {
  return dot4(a[0], b[0]) + dot4(a[1], b[1]) + dot4(a[2], b[2]) + dot4(a[3], b[3]);
}
__device__ __forceinline__ void fma4(float4& acc, float s, const float4& v) {
  acc.x = fmaf(s, v.x, acc.x); acc.y = fmaf(s, v.y, acc.y); acc.z = fmaf(s, v.z, acc.z); acc.w = fmaf(s, v.w, acc.w);
}
__device__ __forceinline__ void st16_bf16(__nv_bfloat16* p, const float4* v, float scale) {
  uint4 u0, u1;
  u0.x = pack_bf16x2(v[0].x * scale, v[0].y * scale); u0.y = pack_bf16x2(v[0].z * scale, v[0].w * scale);
  u0.z = pack_bf16x2(v[1].x * scale, v[1].y * scale); u0.w = pack_bf16x2(v[1].z * scale, v[1].w * scale);
  u1.x = pack_bf16x2(v[2].x * scale, v[2].y * scale); u1.y = pack_bf16x2(v[2].z * scale, v[2].w * scale);
  u1.z = pack_bf16x2(v[3].x * scale, v[3].y * scale); u1.w = pack_bf16x2(v[3].z * scale, v[3].w * scale);
  reinterpret_cast<uint4*>(p)[0] = u0; reinterpret_cast<uint4*>(p)[1] = u1;
}

// pooled keys / values of one map -> shared memory (+ arg-max of every channel for the backward pass)
// (k0, nk: the key range [k0, k0 + nk) of the map, stored at local index k - k0; default: all keys)
__device__ __forceinline__ void build_keys_fast(const AttnParams& p, long long map0, float4* s_phi, float4* s_g,
                                                unsigned char* s_aphi, unsigned char* s_ag, int k0 = 0, int nk = -1) {
  if (nk < 0) nk = p.Kp;
  for (int k = threadIdx.x; k < nk; k += blockDim.x) {
    int pos4[4];
    pooled_window(p, k0 + k, pos4);
    float4 bp = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    float4 bg[4];
    unsigned char ap[4] = {0, 0, 0, 0}, ag[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) bg[i] = bp;
#pragma unroll
    for (int i = 0; i < 16; ++i) ag[i] = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 v = ld4_bf16(p.phi + (map0 + pos4[j]) * 16);
      if (v.x > bp.x) { bp.x = v.x; ap[0] = j; }
      if (v.y > bp.y) { bp.y = v.y; ap[1] = j; }
      if (v.z > bp.z) { bp.z = v.z; ap[2] = j; }
      if (v.w > bp.w) { bp.w = v.w; ap[3] = j; }
      float4 gv[4];
      ld16_bf16(p.g + (map0 + pos4[j]) * 16, gv);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (gv[i].x > bg[i].x) { bg[i].x = gv[i].x; ag[4 * i + 0] = j; }
        if (gv[i].y > bg[i].y) { bg[i].y = gv[i].y; ag[4 * i + 1] = j; }
        if (gv[i].z > bg[i].z) { bg[i].z = gv[i].z; ag[4 * i + 2] = j; }
        if (gv[i].w > bg[i].w) { bg[i].w = gv[i].w; ag[4 * i + 3] = j; }
      }
    }
    s_phi[k] = bp;
#pragma unroll
    for (int i = 0; i < 4; ++i) s_g[k * 4 + i] = bg[i];
    if (s_aphi) {
#pragma unroll
      for (int i = 0; i < 4; ++i) s_aphi[k * 4 + i] = ap[i];
#pragma unroll
      for (int i = 0; i < 16; ++i) s_ag[k * 16 + i] = ag[i];
    }
  }
}

// grid (maps, ceil(P / 512)); 256 threads, two queries per thread
__global__ void __launch_bounds__(256) attn_fwd_fast_kernel(const AttnParams p) {
  extern __shared__ float4 smem_v[];
  float4* s_phi = smem_v;              // [Kp]
  float4* s_g = s_phi + p.Kp;          // [Kp][4]
  const long long map0 = (long long)blockIdx.x * p.P;
  build_keys_fast(p, map0, s_phi, s_g, nullptr, nullptr);
  __syncthreads();
  const int q0 = blockIdx.y * 512 + threadIdx.x, q1 = q0 + 256;
  const bool ok0 = q0 < p.P, ok1 = q1 < p.P;
  if (!ok0) return;
  const float4 t0 = ld4_bf16(p.theta + (map0 + q0) * 16);
  const float4 t1 = ok1 ? ld4_bf16(p.theta + (map0 + q1) * 16) : t0;
  float m0 = -INFINITY, m1 = -INFINITY;
  for (int k = 0; k < p.Kp; ++k) {
    const float4 ph = s_phi[k];
    m0 = fmaxf(m0, dot4(t0, ph));
    m1 = fmaxf(m1, dot4(t1, ph));
  }
  float l0 = 0.f, l1 = 0.f;
  float4 a0[4], a1[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) a0[i] = a1[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = 0; k < p.Kp; ++k) {
    const float4 ph = s_phi[k];
    const float e0 = __expf(dot4(t0, ph) - m0), e1 = __expf(dot4(t1, ph) - m1);
    l0 += e0; l1 += e1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 gv = s_g[k * 4 + i];
      fma4(a0[i], e0, gv);
      fma4(a1[i], e1, gv);
    }
  }
  st16_bf16(p.o + (map0 + q0) * 16, a0, 1.f / l0);
  if (ok1) st16_bf16(p.o + (map0 + q1) * 16, a1, 1.f / l1);
}

// one CTA (512 threads) per map
__global__ void __launch_bounds__(512) attn_bwd_fast_kernel(const AttnParams p) {
  extern __shared__ float4 smem_v[];
  float4* s_phi = smem_v;                         // [Kp]
  float4* s_g = s_phi + p.Kp;                     // [Kp][4]
  float4* s_th = s_g + 4 * p.Kp;                  // [P]
  float4* s_do = s_th + p.P;                      // [P][4]
  float4* s_part = s_do + 4 * p.P;                // [Kp][5] partial sums of the second query half
  float* s_m = reinterpret_cast<float*>(s_part + 5 * p.Kp);   // [P]
  float* s_il = s_m + p.P;                        // [P]
  float* s_dq = s_il + p.P;                       // [P]
  unsigned char* s_aphi = reinterpret_cast<unsigned char*>(s_dq + p.P);   // [Kp][4]
  unsigned char* s_ag = s_aphi + 4 * p.Kp;                                 // [Kp][16]
  const long long map0 = (long long)blockIdx.x * p.P;
  build_keys_fast(p, map0, s_phi, s_g, s_aphi, s_ag);
  for (int q = threadIdx.x; q < p.P; q += blockDim.x) {
    s_th[q] = ld4_bf16(p.theta + (map0 + q) * 16);
    ld16_bf16(p.dout + (map0 + q) * 16, s_do + 4 * q);
  }
  __syncthreads();
  // ---- phase A (thread = query): softmax statistics, D_q = sum_k beta_k (dy . g_k), d theta
  for (int q = threadIdx.x; q < p.P; q += blockDim.x) {
    const float4 th = s_th[q];
    float4 dy[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) dy[i] = s_do[4 * q + i];
    float m = -INFINITY;
    for (int k = 0; k < p.Kp; ++k) m = fmaxf(m, dot4(th, s_phi[k]));
    float l = 0.f, ws = 0.f;
    for (int k = 0; k < p.Kp; ++k) {
      const float e = __expf(dot4(th, s_phi[k]) - m);
      l += e;
      ws = fmaf(e, dot16(dy, s_g + 4 * k), ws);
    }
    const float il = 1.f / l, dq = ws * il;
    float4 dth = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < p.Kp; ++k) {
      const float4 ph = s_phi[k];
      const float ds = __expf(dot4(th, ph) - m) * il * (dot16(dy, s_g + 4 * k) - dq);
      fma4(dth, ds, ph);
    }
    s_m[q] = m; s_il[q] = il; s_dq[q] = dq;
    uint4 u0 = make_uint4(pack_bf16x2(dth.x, dth.y), pack_bf16x2(dth.z, dth.w), 0u, 0u);
    reinterpret_cast<uint4*>(p.dtheta + (map0 + q) * 16)[0] = u0;
    reinterpret_cast<uint4*>(p.dtheta + (map0 + q) * 16)[1] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();
  // ---- phase B (thread = key x query half): d phi_p, d g_p, routed to the arg-max voxel of the pooling window
  // (2 * Kp <= blockDim.x: every (key, half) item has its own thread, one sweep)
  const int nk = p.Kp;
  const int kk = threadIdx.x;
  const bool active = kk < 2 * nk;
  const int k = active ? kk % nk : 0, half = active ? kk / nk : 0;
  float4 dph = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 dgk[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) dgk[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (active) {
    const float4 ph = s_phi[k];
    float4 gk[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) gk[i] = s_g[4 * k + i];
    const int qh = (p.P + 1) / 2;
    const int qb = half * qh, qe = min(p.P, qb + qh);
    for (int q = qb; q < qe; ++q) {
      const float4 th = s_th[q];
      float4 dy[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) dy[i] = s_do[4 * q + i];
      const float beta = __expf(dot4(th, ph) - s_m[q]) * s_il[q];
      const float ds = beta * (dot16(dy, gk) - s_dq[q]);
      fma4(dph, ds, th);
#pragma unroll
      for (int i = 0; i < 4; ++i) fma4(dgk[i], beta, dy[i]);
    }
    if (half == 1) {
      s_part[5 * k] = dph;
#pragma unroll
      for (int i = 0; i < 4; ++i) s_part[5 * k + 1 + i] = dgk[i];
    }
  }
  __syncthreads();
  if (active && half == 0) {
    const float4 o = s_part[5 * k];
    dph.x += o.x; dph.y += o.y; dph.z += o.z; dph.w += o.w;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 t = s_part[5 * k + 1 + i];
      dgk[i].x += t.x; dgk[i].y += t.y; dgk[i].z += t.z; dgk[i].w += t.w;
    }
    int pos4[4];
    pooled_window(p, k, pos4);
    const float dp[4] = {dph.x, dph.y, dph.z, dph.w};
    const float* dgf = reinterpret_cast<const float*>(dgk);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v[16];
#pragma unroll
      for (int c = 0; c < 4; ++c) v[c] = s_aphi[4 * k + c] == j ? dp[c] : 0.f;
      uint4 u0 = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), 0u, 0u);
      reinterpret_cast<uint4*>(p.dphi + (map0 + pos4[j]) * 16)[0] = u0;
      reinterpret_cast<uint4*>(p.dphi + (map0 + pos4[j]) * 16)[1] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int c = 0; c < 16; ++c) v[c] = s_ag[16 * k + c] == j ? dgf[c] : 0.f;
      uint4 g0 = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                            pack_bf16x2(v[6], v[7]));
      uint4 g1 = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]),
                            pack_bf16x2(v[14], v[15]));
      reinterpret_cast<uint4*>(p.dg + (map0 + pos4[j]) * 16)[0] = g0;
      reinterpret_cast<uint4*>(p.dg + (map0 + pos4[j]) * 16)[1] = g1;
    }
  }
}

// ---- maps too large for one CTA (the 64 x 64 map of the 128 x 128 x 32 configuration: 4096 queries x 1024 keys) ----
// Same math in two launches.  A: grid (maps, query blocks of 256), thread = query, all keys in shared memory: softmax
// statistics, D_q and d theta; {m, 1/l, D_q} go to a workspace.  B: grid (maps, key blocks of 64), thread = (key, query
// quarter): the queries stream through shared memory in tiles of 256 (theta, dy and the statistics of A), every thread
// sums d phi_k / d g_k over its quarter of each tile, the four quarters are combined through shared memory and routed
// to the arg-max voxel of the pooling window.  No atomics: deterministic.
static constexpr int kLargeKeys = 64, kLargeTile = 256;

__global__ void __launch_bounds__(256) attn_bwd_large_a_kernel(const AttnParams p, float* __restrict__ stats) {
  extern __shared__ float4 smem_v[];
  float4* s_phi = smem_v;              // [Kp]
  float4* s_g = s_phi + p.Kp;          // [Kp][4]
  const long long map0 = (long long)blockIdx.x * p.P;
  build_keys_fast(p, map0, s_phi, s_g, nullptr, nullptr);
  __syncthreads();
  const int q = blockIdx.y * 256 + threadIdx.x;
  if (q >= p.P) return;
  const float4 th = ld4_bf16(p.theta + (map0 + q) * 16);
  float4 dy[4];
  ld16_bf16(p.dout + (map0 + q) * 16, dy);
  float m = -INFINITY;
  for (int k = 0; k < p.Kp; ++k) m = fmaxf(m, dot4(th, s_phi[k]));
  float l = 0.f, ws = 0.f;
  for (int k = 0; k < p.Kp; ++k) {
    const float e = __expf(dot4(th, s_phi[k]) - m);
    l += e;
    ws = fmaf(e, dot16(dy, s_g + 4 * k), ws);
  }
  const float il = 1.f / l, dq = ws * il;
  float4 dth = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = 0; k < p.Kp; ++k) {
    const float4 ph = s_phi[k];
    const float ds = __expf(dot4(th, ph) - m) * il * (dot16(dy, s_g + 4 * k) - dq);
    fma4(dth, ds, ph);
  }
  float* st = stats + (map0 + q) * 3;
  st[0] = m; st[1] = il; st[2] = dq;
  reinterpret_cast<uint4*>(p.dtheta + (map0 + q) * 16)[0] =
      make_uint4(pack_bf16x2(dth.x, dth.y), pack_bf16x2(dth.z, dth.w), 0u, 0u);
  reinterpret_cast<uint4*>(p.dtheta + (map0 + q) * 16)[1] = make_uint4(0u, 0u, 0u, 0u);
}

__global__ void __launch_bounds__(256) attn_bwd_large_b_kernel(const AttnParams p, const float* __restrict__ stats) {
  extern __shared__ float4 smem_v[];
  float4* s_phi = smem_v;                                   // [64]
  float4* s_g = s_phi + kLargeKeys;                         // [64][4]
  float4* s_th = s_g + 4 * kLargeKeys;                      // [256]
  float4* s_do = s_th + kLargeTile;                         // [256][4]
  float4* s_part = s_do + 4 * kLargeTile;                   // [3][64][5]
  float* s_st = reinterpret_cast<float*>(s_part + 3 * kLargeKeys * 5);     // [256][3]
  unsigned char* s_aphi = reinterpret_cast<unsigned char*>(s_st + 3 * kLargeTile);   // [64][4]
  unsigned char* s_ag = s_aphi + 4 * kLargeKeys;                                      // [64][16]
  const long long map0 = (long long)blockIdx.x * p.P;
  const int k0 = blockIdx.y * kLargeKeys;
  const int nk = min(kLargeKeys, p.Kp - k0);
  build_keys_fast(p, map0, s_phi, s_g, s_aphi, s_ag, k0, nk);
  const int kl = threadIdx.x % kLargeKeys, quarter = threadIdx.x / kLargeKeys;
  const bool active = kl < nk;
  float4 dph = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 dgk[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) dgk[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int t0 = 0; t0 < p.P; t0 += kLargeTile) {
    __syncthreads();                             // keys built / previous tile consumed
    {
      const int q = t0 + threadIdx.x;
      if (q < p.P) {
        s_th[threadIdx.x] = ld4_bf16(p.theta + (map0 + q) * 16);
        ld16_bf16(p.dout + (map0 + q) * 16, s_do + 4 * threadIdx.x);
        const float* st = stats + (map0 + q) * 3;
        s_st[3 * threadIdx.x] = st[0]; s_st[3 * threadIdx.x + 1] = st[1]; s_st[3 * threadIdx.x + 2] = st[2];
      } else {                                   // past the map: 1/l = 0 -> beta = 0, contributes nothing
        s_th[threadIdx.x] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 4; ++i) s_do[4 * threadIdx.x + i] = make_float4(0.f, 0.f, 0.f, 0.f);
        s_st[3 * threadIdx.x] = 0.f; s_st[3 * threadIdx.x + 1] = 0.f; s_st[3 * threadIdx.x + 2] = 0.f;
      }
    }
    __syncthreads();
    if (active) {
      const float4 ph = s_phi[kl];
      float4 gk[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) gk[i] = s_g[4 * kl + i];
      const int qb = quarter * (kLargeTile / 4);
      for (int qq = qb; qq < qb + kLargeTile / 4; ++qq) {
        const float4 th = s_th[qq];
        float4 dy[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) dy[i] = s_do[4 * qq + i];
        const float beta = __expf(dot4(th, ph) - s_st[3 * qq]) * s_st[3 * qq + 1];
        const float ds = beta * (dot16(dy, gk) - s_st[3 * qq + 2]);
        fma4(dph, ds, th);
#pragma unroll
        for (int i = 0; i < 4; ++i) fma4(dgk[i], beta, dy[i]);
      }
    }
  }
  if (active && quarter > 0) {
    float4* dst = s_part + ((quarter - 1) * kLargeKeys + kl) * 5;
    dst[0] = dph;
#pragma unroll
    for (int i = 0; i < 4; ++i) dst[1 + i] = dgk[i];
  }
  __syncthreads();
  if (active && quarter == 0) {
    for (int s = 0; s < 3; ++s) {
      const float4* src = s_part + (s * kLargeKeys + kl) * 5;
      dph.x += src[0].x; dph.y += src[0].y; dph.z += src[0].z; dph.w += src[0].w;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        dgk[i].x += src[1 + i].x; dgk[i].y += src[1 + i].y; dgk[i].z += src[1 + i].z; dgk[i].w += src[1 + i].w;
      }
    }
    int pos4[4];
    pooled_window(p, k0 + kl, pos4);
    const float dp[4] = {dph.x, dph.y, dph.z, dph.w};
    const float* dgf = reinterpret_cast<const float*>(dgk);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v[16];
#pragma unroll
      for (int c = 0; c < 4; ++c) v[c] = s_aphi[4 * kl + c] == j ? dp[c] : 0.f;
      reinterpret_cast<uint4*>(p.dphi + (map0 + pos4[j]) * 16)[0] =
          make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), 0u, 0u);
      reinterpret_cast<uint4*>(p.dphi + (map0 + pos4[j]) * 16)[1] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int c = 0; c < 16; ++c) v[c] = s_ag[16 * kl + c] == j ? dgf[c] : 0.f;
      reinterpret_cast<uint4*>(p.dg + (map0 + pos4[j]) * 16)[0] =
          make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      reinterpret_cast<uint4*>(p.dg + (map0 + pos4[j]) * 16)[1] =
          make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]),
                     pack_bf16x2(v[14], v[15]));
    }
  }
}

static bool attn_fast_cfg(const AttnParams& p) {
  return p.c8 == 4 && p.c2 == 16 && p.C8p == 16 && p.C2p == 16;
}

static bool attn_fast_ok(const AttnParams& p) {
  // phase B of the backward kernel needs both halves of a key in the same sweep (see the kernel)
  return p.c8 == 4 && p.c2 == 16 && p.C8p == 16 && p.C2p == 16 && 2 * p.Kp <= 512;
}

static int attn_fill(AttnParams& p, int64_t N, int D, int H, int W, int c8, int c2, int C8p, int C2p) {
  if (c8 < 1 || c8 > kMaxC8 || c2 < 1 || c2 > kMaxC2 || C8p < c8 || C2p < c2) return T2V_ERR_ARG;
  if ((H & 1) || (W & 1) || N <= 0 || N > 0x7fffffffLL) return T2V_ERR_ARG;
  p.N = (int)N; p.D = D; p.H = H; p.W = W; p.c8 = c8; p.c2 = c2; p.C8p = C8p; p.C2p = C2p;
  p.P = D * H * W; p.Hp = H / 2; p.Wp = W / 2; p.Kp = D * p.Hp * p.Wp;
  return T2V_OK;
}

}  // namespace t2v

using namespace t2v;

extern "C" {

int t2v_attention_fwd(const void* theta, const void* phi, const void* g, void* o, int64_t N, int32_t D, int32_t H,
                      int32_t W, int32_t c8, int32_t c2, int32_t C8p, int32_t C2p, void* stream) {
  AttnParams p{};
  int rc = attn_fill(p, N, D, H, W, c8, c2, C8p, C2p);
  if (rc) return rc;
  p.theta = reinterpret_cast<const __nv_bfloat16*>(theta);
  p.phi = reinterpret_cast<const __nv_bfloat16*>(phi);
  p.g = reinterpret_cast<const __nv_bfloat16*>(g);
  p.o = reinterpret_cast<__nv_bfloat16*>(o);
  if (attn_fast_cfg(p)) {          // (two queries per thread over grid.y: any number of queries)
    const size_t sm = sizeof(float4) * (size_t)p.Kp * 5;
    if (sm <= 200 * 1024) {
      cudaFuncSetAttribute(attn_fwd_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
      dim3 grid((unsigned)N, (unsigned)((p.P + 511) / 512), 1);
      attn_fwd_fast_kernel<<<grid, 256, sm, reinterpret_cast<cudaStream_t>(stream)>>>(p);
      count_launch();
      return check_last("attention_fwd_fast");
    }
  }
  const size_t smem = sizeof(float) * (size_t)p.Kp * (c8 + c2);
  if (smem > 200 * 1024) return T2V_ERR_ARG;
  cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  dim3 grid((unsigned)N, (unsigned)((p.P + 255) / 256), 1);
  attn_fwd_kernel<<<grid, 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  count_launch();
  return check_last("attention_fwd");
}

int t2v_attention_bwd(const void* theta, const void* phi, const void* g, const void* dout, void* dtheta, void* dphi,
                      void* dg, int64_t N, int32_t D, int32_t H, int32_t W, int32_t c8, int32_t c2, int32_t C8p,
                      int32_t C2p, void* stream) {
  AttnParams p{};
  int rc = attn_fill(p, N, D, H, W, c8, c2, C8p, C2p);
  if (rc) return rc;
  p.theta = reinterpret_cast<const __nv_bfloat16*>(theta);
  p.phi = reinterpret_cast<const __nv_bfloat16*>(phi);
  p.g = reinterpret_cast<const __nv_bfloat16*>(g);
  p.dout = reinterpret_cast<const __nv_bfloat16*>(dout);
  p.dtheta = reinterpret_cast<__nv_bfloat16*>(dtheta);
  p.dphi = reinterpret_cast<__nv_bfloat16*>(dphi);
  p.dg = reinterpret_cast<__nv_bfloat16*>(dg);
  if (attn_fast_ok(p)) {
    const size_t sm = sizeof(float4) * ((size_t)p.Kp * 10 + (size_t)p.P * 5) + sizeof(float) * 3 * (size_t)p.P +
                      (size_t)p.Kp * 20 + 16;
    if (sm <= 220 * 1024) {
      cudaFuncSetAttribute(attn_bwd_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
      attn_bwd_fast_kernel<<<(unsigned)N, 512, sm, reinterpret_cast<cudaStream_t>(stream)>>>(p);
      count_launch();
      return check_last("attention_bwd_fast");
    }
  }
  const size_t smem = sizeof(float) * ((size_t)p.Kp * (c8 + c2) + (size_t)p.P * (c8 + c2 + 3)) + (size_t)p.Kp * (c8 + c2);
  if (smem > 200 * 1024) return T2V_ERR_ARG;
  cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  attn_bwd_kernel<<<(unsigned)N, 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  count_launch();
  return check_last("attention_bwd");
}

/* t2v_attention_bwd for maps beyond one CTA (up to 2560 pooled keys): stats_ws = fp32 [N * D*H*W * 3] workspace */
int t2v_attention_bwd_large(const void* theta, const void* phi, const void* g, const void* dout, void* dtheta, void* dphi,
                            void* dg, float* stats_ws, int64_t N, int32_t D, int32_t H, int32_t W, int32_t c8, int32_t c2,
                            int32_t C8p, int32_t C2p, void* stream) {
  AttnParams p{};
  int rc = attn_fill(p, N, D, H, W, c8, c2, C8p, C2p);
  if (rc) return rc;
  if (!stats_ws || !attn_fast_cfg(p)) return T2V_ERR_ARG;
  const size_t sm_a = sizeof(float4) * (size_t)p.Kp * 5;
  if (sm_a > 200 * 1024) return T2V_ERR_ARG;
  p.theta = reinterpret_cast<const __nv_bfloat16*>(theta);
  p.phi = reinterpret_cast<const __nv_bfloat16*>(phi);
  p.g = reinterpret_cast<const __nv_bfloat16*>(g);
  p.dout = reinterpret_cast<const __nv_bfloat16*>(dout);
  p.dtheta = reinterpret_cast<__nv_bfloat16*>(dtheta);
  p.dphi = reinterpret_cast<__nv_bfloat16*>(dphi);
  p.dg = reinterpret_cast<__nv_bfloat16*>(dg);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  cudaFuncSetAttribute(attn_bwd_large_a_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_a);
  attn_bwd_large_a_kernel<<<dim3((unsigned)N, (unsigned)((p.P + 255) / 256), 1), 256, sm_a, s>>>(p, stats_ws);
  const size_t sm_b = sizeof(float4) * (5 * kLargeKeys + 5 * kLargeTile + 15 * kLargeKeys) + sizeof(float) * 3 * kLargeTile +
                      20 * kLargeKeys;
  cudaFuncSetAttribute(attn_bwd_large_b_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_b);
  attn_bwd_large_b_kernel<<<dim3((unsigned)N, (unsigned)((p.Kp + kLargeKeys - 1) / kLargeKeys), 1), 256, sm_b, s>>>(
      p, stats_ws);
  count_launch(2);
  return check_last("attention_bwd_large");
}

}  // extern "C"
