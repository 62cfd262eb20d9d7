// Length-masked (packed-sequence) LSTM recurrence for the caption encoder / decoder
// (txt2vid/models/txt/basic.py:18-19,49-70 nn.LSTM(256, 128, 4 layers, bidirectional) on a PackedSequence;
// :73-101 step-wise decoding), replacing cuDNN's RNN kernels.
//
// Split of the work per layer:
//   * input projection  gx[b,t,dir] = W_ih[dir] x[b,t] + b_ih + b_hh   -- ONE GEMM over all (b, t) and both
//     directions on the tcgen05 engine (t2v_conv_fprop, 1x1x1, fp32 output);
//   * THIS FILE: the sequential part.  One persistent CTA per (16 samples, direction) walks the time axis:
//     gates = gx + W_hh h (fp32 FMA, W_hh^T streamed from L2, h in shared memory), sigma / tanh cell update, length
//     masking exactly as cuDNN's packed sequences (sample b advances only while t < len_b; the reverse direction
//     starts at each sample's own last token; padded steps emit zeros), final (h_n, c_n);
//   * backward: the mirrored walk producing d(gates) for all steps (+ d h_0, d c_0); the weight / input gradients are
//     then three GEMMs on the engine (dX = dG W_ih, dW_ih = dG^T X, dW_hh = dG^T h_prev) and one column sum.
// Gate order i, f, g, o (PyTorch).  All state math is fp32; `ST` is the activation storage type of the sequence
// tensors that feed GEMMs (bf16, or fp32 in the fp32 parity mode).
#include <cstdlib>

#include "t2v_common.cuh"

namespace t2v {

static constexpr int kLstmBT = 16;   // samples per CTA

template <typename T> T2V_DEVINL T lstm_cvt(float v);
template <> T2V_DEVINL __nv_bfloat16 lstm_cvt<__nv_bfloat16>(float v) { return f2bf(v); }
template <> T2V_DEVINL float lstm_cvt<float>(float v) { return v; }

T2V_DEVINL float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

struct LstmSeq {
  int B, L, H, ndir;
  const float* gx;        // [B][L][ndir][4H]   input projection + both biases
  const float* whhT;      // [ndir][H][4H]      W_hh transposed (t2v_lstm_pack_whh)
  const float* whh;       // [ndir][4H][H]      (backward)
  const int* lengths;     // [B]
  const float* h0;        // [ndir][B][H] or null
  const float* c0;
  void* out;              // ST [B][L][ndir*H]    h_t (zeros at padded steps)
  void* hprev;            // ST [B][L][ndir*H]    h entering step t (zeros at padded steps), or null
  float* gates;           // [B][L][ndir][4H]   post-activation i, f, g, o (saved for backward), or null
  float* cells;           // [B][L][ndir][H]    c_t (saved for backward), or null
  float* hn;              // [ndir][B][H]
  float* cn;
  // backward
  const void* dout;       // ST [B][L][ndir*H] or null
  const float* dhn;       // [ndir][B][H] or null
  const float* dcn;
  void* dgates;           // ST [B][L][ndir*4H]  d(pre-activation gates) (zeros at padded steps)
  float* dh0;             // [ndir][B][H] or null
  float* dc0;
};

// grid (ceil(B / kLstmBT), ndir), block H threads (thread j = hidden unit j), dynamic smem kLstmBT * H floats
template <typename ST>
__global__ void lstm_seq_fwd_kernel(const LstmSeq p) {
  extern __shared__ float sh[];                 // [kLstmBT][H]
  const int H = p.H, j = threadIdx.x, dir = blockIdx.y;
  const int b0 = blockIdx.x * kLstmBT;
  const int nb = min(kLstmBT, p.B - b0);
  float c[kLstmBT], h[kLstmBT];
  int len[kLstmBT];
#pragma unroll
  for (int b = 0; b < kLstmBT; ++b) {
    const bool ok = b < nb;
    len[b] = ok ? p.lengths[b0 + b] : 0;
    h[b] = (ok && p.h0) ? p.h0[((size_t)dir * p.B + b0 + b) * H + j] : 0.f;
    c[b] = (ok && p.c0) ? p.c0[((size_t)dir * p.B + b0 + b) * H + j] : 0.f;
    sh[b * H + j] = h[b];
  }
  __syncthreads();
  const float* wT = p.whhT + (size_t)dir * H * 4 * H;
  ST* out = reinterpret_cast<ST*>(p.out);
  ST* hprev = reinterpret_cast<ST*>(p.hprev);
  for (int s = 0; s < p.L; ++s) {
    const int t = dir == 0 ? s : p.L - 1 - s;
    float acc[kLstmBT][4];
#pragma unroll
    for (int b = 0; b < kLstmBT; ++b) {
      if (b < nb && t < len[b]) {
        const float* g = p.gx + (((size_t)(b0 + b) * p.L + t) * p.ndir + dir) * 4 * H;
        acc[b][0] = g[j]; acc[b][1] = g[H + j]; acc[b][2] = g[2 * H + j]; acc[b][3] = g[3 * H + j];
      } else {
        acc[b][0] = acc[b][1] = acc[b][2] = acc[b][3] = 0.f;
      }
    }
    for (int k = 0; k < H; ++k) {
      const float w0 = wT[(size_t)k * 4 * H + j], w1 = wT[(size_t)k * 4 * H + H + j],
                  w2 = wT[(size_t)k * 4 * H + 2 * H + j], w3 = wT[(size_t)k * 4 * H + 3 * H + j];
#pragma unroll
      for (int b = 0; b < kLstmBT; ++b) {
        const float hv = sh[b * H + k];
        acc[b][0] = fmaf(hv, w0, acc[b][0]); acc[b][1] = fmaf(hv, w1, acc[b][1]);
        acc[b][2] = fmaf(hv, w2, acc[b][2]); acc[b][3] = fmaf(hv, w3, acc[b][3]);
      }
    }
    __syncthreads();                            // every thread has finished reading h_{t-1}
#pragma unroll
    for (int b = 0; b < kLstmBT; ++b) {
      if (b >= nb) continue;
      const size_t row = (size_t)(b0 + b) * p.L + t;
      const bool live = t < len[b];
      float hv = 0.f, hp = 0.f;
      if (live) {
        const float gi = sigmoidf_(acc[b][0]), gf = sigmoidf_(acc[b][1]), gg = tanhf(acc[b][2]),
                    go = sigmoidf_(acc[b][3]);
        hp = h[b];
        c[b] = gf * c[b] + gi * gg;
        h[b] = go * tanhf(c[b]);
        hv = h[b];
        sh[b * H + j] = hv;
        if (p.gates) {
          float* gs = p.gates + (row * p.ndir + dir) * 4 * H;
          gs[j] = gi; gs[H + j] = gf; gs[2 * H + j] = gg; gs[3 * H + j] = go;
        }
        if (p.cells) p.cells[(row * p.ndir + dir) * H + j] = c[b];
      }
      out[row * p.ndir * H + dir * H + j] = lstm_cvt<ST>(hv);
      if (hprev) hprev[row * p.ndir * H + dir * H + j] = lstm_cvt<ST>(hp);
    }
    __syncthreads();
  }
#pragma unroll
  for (int b = 0; b < kLstmBT; ++b) {
    if (b >= nb) continue;
    p.hn[((size_t)dir * p.B + b0 + b) * H + j] = h[b];
    p.cn[((size_t)dir * p.B + b0 + b) * H + j] = c[b];
  }
}

// Shared-memory-resident variant for the bf16 storage mode (H <= 128): W_hh^T lives in shared memory as bf16,
// gate-interleaved [k][j][i|f|g|o] (one 8-byte load per k and thread; H * 4H * 2 B = 128 KB at H = 128), instead of
// being streamed from L2 on every time step (the walk above is bound by the latency of those loads: 37 us per step at
// B = 1024).  256 threads: thread (j, half) owns hidden unit j of 8 of the CTA's 16 samples; h_{t-1} is kept
// k-major in shared memory so that the 8 samples of a thread are two broadcast 16-byte loads per k.  Same fp32 state
// math and masking as above; the recurrent weights carry the bf16 rounding every GEMM operand of this mode has.
static constexpr int kLstmSmemThreads = 256;
__global__ void __launch_bounds__(kLstmSmemThreads, 1) lstm_seq_fwd_smem_kernel(const LstmSeq p) {
  extern __shared__ __align__(16) uint8_t lsm[];
  const int H = p.H, tid = threadIdx.x, j = tid % H, half = tid / H, dir = blockIdx.y;
  const int per = kLstmBT / (kLstmSmemThreads / H);            // samples per thread (8 at H = 128)
  uint2* wsm = reinterpret_cast<uint2*>(lsm);                   // [H k][H j] x 4 bf16
  float* hsm = reinterpret_cast<float*>(lsm + (size_t)H * H * 8);   // [H k][kLstmBT]
  const int b0 = blockIdx.x * kLstmBT;
  const int nb = min(kLstmBT, p.B - b0);
  const float* wT = p.whhT + (size_t)dir * H * 4 * H;
  for (int i = tid; i < H * H; i += blockDim.x) {
    const int k = i / H, jj = i % H;
    const float* w = wT + (size_t)k * 4 * H + jj;
    wsm[i] = make_uint2(pack_bf16x2(w[0], w[H]), pack_bf16x2(w[2 * H], w[3 * H]));
  }
  float c[8], h[8];
  int len[8];
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const int bb = half * per + b;
    const bool ok = b < per && bb < nb;
    len[b] = ok ? p.lengths[b0 + bb] : 0;
    h[b] = (ok && p.h0) ? p.h0[((size_t)dir * p.B + b0 + bb) * H + j] : 0.f;
    c[b] = (ok && p.c0) ? p.c0[((size_t)dir * p.B + b0 + bb) * H + j] : 0.f;
    if (b < per) hsm[j * kLstmBT + bb] = h[b];
  }
  __syncthreads();
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(p.out);
  __nv_bfloat16* hprev = reinterpret_cast<__nv_bfloat16*>(p.hprev);
  for (int s = 0; s < p.L; ++s) {
    const int t = dir == 0 ? s : p.L - 1 - s;
    float acc[8][4];
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int bb = half * per + b;
      if (b < per && bb < nb && t < len[b]) {
        const float* g = p.gx + (((size_t)(b0 + bb) * p.L + t) * p.ndir + dir) * 4 * H;
        acc[b][0] = g[j]; acc[b][1] = g[H + j]; acc[b][2] = g[2 * H + j]; acc[b][3] = g[3 * H + j];
      } else {
        acc[b][0] = acc[b][1] = acc[b][2] = acc[b][3] = 0.f;
      }
    }
#pragma unroll 4
    for (int k = 0; k < H; ++k) {
      const uint2 wq = wsm[k * H + j];
      const float2 w01 = unpack_bf16x2(wq.x), w23 = unpack_bf16x2(wq.y);
      const float4 ha = *reinterpret_cast<const float4*>(hsm + k * kLstmBT + half * per);
      const float4 hb = *reinterpret_cast<const float4*>(hsm + k * kLstmBT + half * per + 4);
      const float hv[8] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        acc[b][0] = fmaf(hv[b], w01.x, acc[b][0]); acc[b][1] = fmaf(hv[b], w01.y, acc[b][1]);
        acc[b][2] = fmaf(hv[b], w23.x, acc[b][2]); acc[b][3] = fmaf(hv[b], w23.y, acc[b][3]);
      }
    }
    __syncthreads();                            // every thread has finished reading h_{t-1}
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int bb = half * per + b;
      if (b >= per || bb >= nb) continue;
      const size_t row = (size_t)(b0 + bb) * p.L + t;
      const bool live = t < len[b];
      float hv = 0.f, hp = 0.f;
      if (live) {
        const float gi = sigmoidf_(acc[b][0]), gf = sigmoidf_(acc[b][1]), gg = tanhf(acc[b][2]),
                    go = sigmoidf_(acc[b][3]);
        hp = h[b];
        c[b] = gf * c[b] + gi * gg;
        h[b] = go * tanhf(c[b]);
        hv = h[b];
        hsm[j * kLstmBT + bb] = hv;
        if (p.gates) {
          float* gs = p.gates + (row * p.ndir + dir) * 4 * H;
          gs[j] = gi; gs[H + j] = gf; gs[2 * H + j] = gg; gs[3 * H + j] = go;
        }
        if (p.cells) p.cells[(row * p.ndir + dir) * H + j] = c[b];
      }
      out[row * p.ndir * H + dir * H + j] = f2bf(hv);
      if (hprev) hprev[row * p.ndir * H + dir * H + j] = f2bf(hp);
    }
    __syncthreads();
  }
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const int bb = half * per + b;
    if (b >= per || bb >= nb) continue;
    p.hn[((size_t)dir * p.B + b0 + bb) * H + j] = h[b];
    p.cn[((size_t)dir * p.B + b0 + bb) * H + j] = c[b];
  }
}

// mirrored walk: d(pre-activation gates) for every step, d h_0 / d c_0.  smem: kLstmBT * 4H floats (dgates of a step)
template <typename ST>
__global__ void lstm_seq_bwd_kernel(const LstmSeq p) {
  extern __shared__ float sdg[];                // [kLstmBT][4H]
  const int H = p.H, j = threadIdx.x, dir = blockIdx.y;
  const int b0 = blockIdx.x * kLstmBT;
  const int nb = min(kLstmBT, p.B - b0);
  float dh[kLstmBT], dc[kLstmBT];
  int len[kLstmBT];
#pragma unroll
  for (int b = 0; b < kLstmBT; ++b) {
    const bool ok = b < nb;
    len[b] = ok ? p.lengths[b0 + b] : 0;
    dh[b] = (ok && p.dhn) ? p.dhn[((size_t)dir * p.B + b0 + b) * H + j] : 0.f;
    dc[b] = (ok && p.dcn) ? p.dcn[((size_t)dir * p.B + b0 + b) * H + j] : 0.f;
  }
  const float* W = p.whh + (size_t)dir * 4 * H * H;
  const ST* dout = reinterpret_cast<const ST*>(p.dout);
  ST* dgates = reinterpret_cast<ST*>(p.dgates);
  for (int s = p.L - 1; s >= 0; --s) {          // reverse of the forward order
    const int t = dir == 0 ? s : p.L - 1 - s;
#pragma unroll
    for (int b = 0; b < kLstmBT; ++b) {
      float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
      if (b < nb) {
        const size_t row = (size_t)(b0 + b) * p.L + t;
        if (t < len[b]) {
          const float* gs = p.gates + (row * p.ndir + dir) * 4 * H;
          const float gi = gs[j], gf = gs[H + j], gg = gs[2 * H + j], go = gs[3 * H + j];
          const float cv = p.cells[(row * p.ndir + dir) * H + j];
          // c entering this step: the previous step in walk order, or c_0 at the sample's first live step
          const int tp = dir == 0 ? t - 1 : t + 1;
          float cp;
          if (tp >= 0 && tp < len[b]) cp = p.cells[(((size_t)(b0 + b) * p.L + tp) * p.ndir + dir) * H + j];
          else cp = p.c0 ? p.c0[((size_t)dir * p.B + b0 + b) * H + j] : 0.f;
          const float tc = tanhf(cv);
          const float dhv = dh[b] + (dout ? bf2f(dout[row * p.ndir * H + dir * H + j]) : 0.f);
          const float dcv = dc[b] + dhv * go * (1.f - tc * tc);
          d0 = dcv * gg * gi * (1.f - gi);
          d1 = dcv * cp * gf * (1.f - gf);
          d2 = dcv * gi * (1.f - gg * gg);
          d3 = dhv * tc * go * (1.f - go);
          dc[b] = dcv * gf;
        }
        ST* dgr = dgates + row * p.ndir * 4 * H + (size_t)dir * 4 * H;
        dgr[j] = lstm_cvt<ST>(d0); dgr[H + j] = lstm_cvt<ST>(d1);
        dgr[2 * H + j] = lstm_cvt<ST>(d2); dgr[3 * H + j] = lstm_cvt<ST>(d3);
      }
      sdg[b * 4 * H + j] = d0; sdg[b * 4 * H + H + j] = d1; sdg[b * 4 * H + 2 * H + j] = d2;
      sdg[b * 4 * H + 3 * H + j] = d3;
    }
    __syncthreads();
    // dh_{prev}[j] = sum_r dgates[r] W[r][j]  (live samples; dead samples keep dh, dc unchanged: sdg row is zero and
    // dh must then carry over, so add instead of overwrite for them)
    float acc[kLstmBT];
#pragma unroll
    for (int b = 0; b < kLstmBT; ++b) acc[b] = 0.f;
    for (int r = 0; r < 4 * H; ++r) {
      const float w = W[(size_t)r * H + j];
#pragma unroll
      for (int b = 0; b < kLstmBT; ++b) acc[b] = fmaf(sdg[b * 4 * H + r], w, acc[b]);
    }
#pragma unroll
    for (int b = 0; b < kLstmBT; ++b)
      if (b < nb && t < len[b]) dh[b] = acc[b];
    __syncthreads();
  }
#pragma unroll
  for (int b = 0; b < kLstmBT; ++b) {
    if (b >= nb) continue;
    if (p.dh0) p.dh0[((size_t)dir * p.B + b0 + b) * H + j] = dh[b];
    if (p.dc0) p.dc0[((size_t)dir * p.B + b0 + b) * H + j] = dc[b];
  }
}

// whhT[dir][k][r] = whh[dir][r][k]
__global__ void lstm_pack_whh_kernel(const float* __restrict__ w, float* __restrict__ wT, int H, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int r = (int)(i % (4 * H));
  const long long t = i / (4 * H);
  const int k = (int)(t % H);
  const long long dir = t / H;
  wT[i] = w[(dir * 4 * H + r) * H + k];
}

// out[row, :] = weight[tokens[row], :]   (nn.Embedding, models/txt/basic.py:16,51); one thread per 4 elements
template <typename ST>
__global__ void embedding_fwd_kernel(const long long* __restrict__ tokens, const float* __restrict__ weight,
                                     ST* __restrict__ out, int E, long long total4) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int e4 = E / 4;
  const long long row = i / e4;
  const int c = (int)(i % e4) * 4;
  const float4 v = *reinterpret_cast<const float4*>(weight + tokens[row] * E + c);
  ST* o = out + row * E + c;
  o[0] = lstm_cvt<ST>(v.x); o[1] = lstm_cvt<ST>(v.y); o[2] = lstm_cvt<ST>(v.z); o[3] = lstm_cvt<ST>(v.w);
}
// dweight[tokens[row], :] += dout[row, :]   (dweight zeroed by the host call)
template <typename ST>
__global__ void embedding_bwd_kernel(const long long* __restrict__ tokens, const ST* __restrict__ dout,
                                     float* __restrict__ dweight, int E, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long row = i / E;
  atomicAdd(dweight + tokens[row] * E + (i % E), bf2f(dout[i]));
}

template <typename ST>
static int lstm_fwd_impl(LstmSeq p, cudaStream_t s) {
  if (p.H % 32 || p.H > 1024 || p.B <= 0 || p.L <= 0 || p.ndir < 1 || p.ndir > 2) return T2V_ERR_ARG;
  dim3 grid((p.B + kLstmBT - 1) / kLstmBT, p.ndir, 1);
  if (sizeof(ST) == 2 && p.H == 128) {            // bf16 storage mode: recurrent weights resident in smem
    const size_t smem = (size_t)p.H * p.H * 8 + sizeof(float) * kLstmBT * p.H;
    cudaFuncSetAttribute(lstm_seq_fwd_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    lstm_seq_fwd_smem_kernel<<<grid, kLstmSmemThreads, smem, s>>>(p);
    count_launch();
    return check_last("lstm_seq_fwd");
  }
  lstm_seq_fwd_kernel<ST><<<grid, p.H, sizeof(float) * kLstmBT * p.H, s>>>(p);
  count_launch();
  return check_last("lstm_seq_fwd");
}
template <typename ST>
static int lstm_bwd_impl(LstmSeq p, cudaStream_t s) {
  if (p.H % 32 || p.H > 512 || p.B <= 0 || p.L <= 0 || p.ndir < 1 || p.ndir > 2) return T2V_ERR_ARG;
  dim3 grid((p.B + kLstmBT - 1) / kLstmBT, p.ndir, 1);
  const size_t smem = sizeof(float) * kLstmBT * 4 * p.H;
  cudaFuncSetAttribute(lstm_seq_bwd_kernel<ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  lstm_seq_bwd_kernel<ST><<<grid, p.H, smem, s>>>(p);
  count_launch();
  return check_last("lstm_seq_bwd");
}

}  // namespace t2v

using namespace t2v;
#define STREAM reinterpret_cast<cudaStream_t>(stream)

extern "C" {

int t2v_lstm_pack_whh(const float* whh, float* whhT, int32_t ndir, int32_t H, void* stream) {
  const long long total = (long long)ndir * H * 4 * H;
  if (!whh || !whhT || total <= 0) return T2V_ERR_ARG;
  lstm_pack_whh_kernel<<<(unsigned)((total + 255) / 256), 256, 0, STREAM>>>(whh, whhT, H, total);
  count_launch();
  return check_last("lstm_pack_whh");
}

#define T2V_LSTM_FWD_ARGS                                                                                          \
  const float *gx, const float *whhT, const int32_t *lengths, const float *h0, const float *c0, void *out,       \
      void *hprev, float *gates, float *cells, float *hn, float *cn, int32_t B, int32_t L, int32_t H, int32_t ndir, \
      void *stream
static LstmSeq fwd_params(const float* gx, const float* whhT, const int32_t* lengths, const float* h0, const float* c0,
                          void* out, void* hprev, float* gates, float* cells, float* hn, float* cn, int32_t B,
                          int32_t L, int32_t H, int32_t ndir) {
  LstmSeq p{};
  p.B = B; p.L = L; p.H = H; p.ndir = ndir;
  p.gx = gx; p.whhT = whhT; p.lengths = lengths; p.h0 = h0; p.c0 = c0;
  p.out = out; p.hprev = hprev; p.gates = gates; p.cells = cells; p.hn = hn; p.cn = cn;
  return p;
}
int t2v_lstm_seq_fwd(T2V_LSTM_FWD_ARGS) {
  if (!gx || !whhT || !lengths || !out || !hn || !cn) return T2V_ERR_ARG;
  return lstm_fwd_impl<__nv_bfloat16>(fwd_params(gx, whhT, lengths, h0, c0, out, hprev, gates, cells, hn, cn, B, L, H,
                                                 ndir), STREAM);
}
int t2v_lstm_seq_fwd_f32(T2V_LSTM_FWD_ARGS) {
  if (!gx || !whhT || !lengths || !out || !hn || !cn) return T2V_ERR_ARG;
  return lstm_fwd_impl<float>(fwd_params(gx, whhT, lengths, h0, c0, out, hprev, gates, cells, hn, cn, B, L, H, ndir),
                              STREAM);
}

#define T2V_LSTM_BWD_ARGS                                                                                           \
  const float *whh, const int32_t *lengths, const float *c0, const float *gates, const float *cells,               \
      const void *dout, const float *dhn, const float *dcn, void *dgates, float *dh0, float *dc0, int32_t B,       \
      int32_t L, int32_t H, int32_t ndir, void *stream
static LstmSeq bwd_params(const float* whh, const int32_t* lengths, const float* c0, const float* gates,
                          const float* cells, const void* dout, const float* dhn, const float* dcn, void* dgates,
                          float* dh0, float* dc0, int32_t B, int32_t L, int32_t H, int32_t ndir) {
  LstmSeq p{};
  p.B = B; p.L = L; p.H = H; p.ndir = ndir;
  p.whh = whh; p.lengths = lengths; p.c0 = c0; p.gates = const_cast<float*>(gates); p.cells = const_cast<float*>(cells);
  p.dout = dout; p.dhn = dhn; p.dcn = dcn; p.dgates = dgates; p.dh0 = dh0; p.dc0 = dc0;
  return p;
}
int t2v_lstm_seq_bwd(T2V_LSTM_BWD_ARGS) {
  if (!whh || !lengths || !gates || !cells || !dgates) return T2V_ERR_ARG;
  return lstm_bwd_impl<__nv_bfloat16>(bwd_params(whh, lengths, c0, gates, cells, dout, dhn, dcn, dgates, dh0, dc0, B, L,
                                                 H, ndir), STREAM);
}
int t2v_lstm_seq_bwd_f32(T2V_LSTM_BWD_ARGS) {
  if (!whh || !lengths || !gates || !cells || !dgates) return T2V_ERR_ARG;
  return lstm_bwd_impl<float>(bwd_params(whh, lengths, c0, gates, cells, dout, dhn, dcn, dgates, dh0, dc0, B, L, H,
                                         ndir), STREAM);
}

int t2v_embedding_fwd(const int64_t* tokens, const float* weight, void* out, int64_t rows, int32_t E, void* stream) {
  if (!tokens || !weight || !out || E % 4) return T2V_ERR_ARG;
  const long long total4 = rows * E / 4;
  if (total4 == 0) return T2V_OK;
  embedding_fwd_kernel<__nv_bfloat16><<<(unsigned)((total4 + 255) / 256), 256, 0, STREAM>>>(
      reinterpret_cast<const long long*>(tokens), weight, reinterpret_cast<__nv_bfloat16*>(out), E, total4);
  count_launch();
  return check_last("embedding_fwd");
}
int t2v_embedding_fwd_f32(const int64_t* tokens, const float* weight, void* out, int64_t rows, int32_t E,
                          void* stream) {
  if (!tokens || !weight || !out || E % 4) return T2V_ERR_ARG;
  const long long total4 = rows * E / 4;
  if (total4 == 0) return T2V_OK;
  embedding_fwd_kernel<float><<<(unsigned)((total4 + 255) / 256), 256, 0, STREAM>>>(
      reinterpret_cast<const long long*>(tokens), weight, reinterpret_cast<float*>(out), E, total4);
  count_launch();
  return check_last("embedding_fwd");
}
int t2v_embedding_bwd(const int64_t* tokens, const void* dout, float* dweight, int64_t rows, int32_t E, int64_t V,
                      void* stream) {
  if (!tokens || !dout || !dweight) return T2V_ERR_ARG;
  cudaMemsetAsync(dweight, 0, sizeof(float) * (size_t)V * E, STREAM);
  const long long total = rows * E;
  if (total == 0) return T2V_OK;
  embedding_bwd_kernel<__nv_bfloat16><<<(unsigned)((total + 255) / 256), 256, 0, STREAM>>>(
      reinterpret_cast<const long long*>(tokens), reinterpret_cast<const __nv_bfloat16*>(dout), dweight, E, total);
  count_launch();
  return check_last("embedding_bwd");
}
int t2v_embedding_bwd_f32(const int64_t* tokens, const void* dout, float* dweight, int64_t rows, int32_t E, int64_t V,
                          void* stream) {
  if (!tokens || !dout || !dweight) return T2V_ERR_ARG;
  cudaMemsetAsync(dweight, 0, sizeof(float) * (size_t)V * E, STREAM);
  const long long total = rows * E;
  if (total == 0) return T2V_OK;
  embedding_bwd_kernel<float><<<(unsigned)((total + 255) / 256), 256, 0, STREAM>>>(
      reinterpret_cast<const long long*>(tokens), reinterpret_cast<const float*>(dout), dweight, E, total);
  count_launch();
  return check_last("embedding_bwd");
}

}  // extern "C"
