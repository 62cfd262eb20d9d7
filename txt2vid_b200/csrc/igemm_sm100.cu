// Implicit-GEMM convolution engine for sm_100a: TMA-fed tcgen05.mma with TMEM accumulators.
//
// Replaces every F.conv2d / F.conv3d / F.linear call site on the TGANv2 path of the reference
// (txt2vid/models/layers.py:174-183,231-237,251; resnet3d.py:12-17; conv_lstm.py:32-38 centre-tap
// GEMM; tganv2_cond/gen.py:39 Linear) -- all of them stride-1, "same"-padded, kernel 1 or 3.
//
// Layout trick: activations are channels-last [N][D][H][W][C] bf16.  A 5-D TMA box
// (C=BLOCK_K, bw, bh, bd, bn) with bw*bh*bd*bn = 128 lands in shared memory as 128 rows of
// BLOCK_K*2 bytes -- exactly the canonical K-major swizzled UMMA operand -- and a filter tap is just
// a coordinate offset; halo / padding comes from TMA out-of-bounds zero fill.  So im2col never
// exists in memory and the tensor core reads what TMA wrote.
//
//   fprop : D[128 pos x BN cout] += A[pos, (tap,ci)] * W[cout, (tap,ci)]      (both K-major)
//   dgrad : same kernel on dy with the flipped/transposed weight pack
//   wgrad : D[128 cout x BN cin]  += dy[pos, cout]^T * x[pos+tap, cin]        (both MN-major),
//           split over position tiles, fp32 atomics into dw[cout][tap][cin]
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2-5 = epilogue (TMEM -> registers -> global).
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "t2v_common.cuh"
#include "tmap.cuh"

namespace t2v {

struct IgemmParams {
  int N, D, H, W, Cin, Cout;
  int kd, kh, kw, pd, ph, pw;
  int bn, bd, bh, bw;          // position box (product = rows per k-block)
  int tn, td, th, tw;          // number of boxes per dim
  int BN;                      // GEMM-N tile (<= 256, multiple of 16)
  int lo_d, hi_d, lo_h, hi_h, lo_w, hi_w;  // live tap ranges (dead taps read only padding)
  int cblocks;                 // Cin / BLOCK_K
  int num_k_blocks;
  int aux_k_blocks;            // extra k-blocks of a fused 1x1x1 convolution of a second tensor (same positions)
  int stages;
  uint32_t stage_bytes, a_bytes, b_bytes;
  uint32_t idesc, tmem_cols;
  const float* bias;
  const __nv_bfloat16* residual;
  void* out;
  int out_f32, relu, relu_mask;
  // fused ConvLSTM cell epilogue (columns gate-interleaved per 32 hidden units: tile = [i | f | g | o] x 32)
  int lstm, lstm_t, lstm_steps, lstm_plane;
  const float* c_prev;
  float* c_out;
  float* gates_out;
  __nv_bfloat16* h_out;
  __nv_bfloat16* h_merged;
  // wgrad only
  float* dw;
  int taps_total, splits, tiles_total, atomic_out;
};

static constexpr int kThreads = 192;

template <int BLOCK_K>
struct SwizzleOf {
  static constexpr uint32_t layout = BLOCK_K == 64 ? 2u : (BLOCK_K == 32 ? 4u : 6u);
  static constexpr uint32_t sbo = 8u * BLOCK_K * 2u;
};

// ------------------------------------------------------------------------------------ fprop
// Epilogue of 16 accumulator columns of one output row: bias, residual / ReLU mask, ReLU, store.
T2V_DEVINL void fprop_epilogue16(const IgemmParams& p, const uint32_t (&v)[16], size_t pos, int col) {
  float f[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j]);
  if (p.bias != nullptr) {
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
      const float4 b = *reinterpret_cast<const float4*>(p.bias + col + j);
      f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
    }
  }
  if (p.residual != nullptr) {
    const uint4* rp = reinterpret_cast<const uint4*>(p.residual + pos * p.Cout + col);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const uint4 u = rp[j];
      const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), cc = unpack_bf16x2(u.z),
                   dd = unpack_bf16x2(u.w);
      if (p.relu_mask) {      // the pointer is a ReLU reference: dx = dgrad(dy) * (ref > 0)
        f[8 * j + 0] = a.x > 0.f ? f[8 * j + 0] : 0.f; f[8 * j + 1] = a.y > 0.f ? f[8 * j + 1] : 0.f;
        f[8 * j + 2] = b.x > 0.f ? f[8 * j + 2] : 0.f; f[8 * j + 3] = b.y > 0.f ? f[8 * j + 3] : 0.f;
        f[8 * j + 4] = cc.x > 0.f ? f[8 * j + 4] : 0.f; f[8 * j + 5] = cc.y > 0.f ? f[8 * j + 5] : 0.f;
        f[8 * j + 6] = dd.x > 0.f ? f[8 * j + 6] : 0.f; f[8 * j + 7] = dd.y > 0.f ? f[8 * j + 7] : 0.f;
      } else {
        f[8 * j + 0] += a.x; f[8 * j + 1] += a.y; f[8 * j + 2] += b.x; f[8 * j + 3] += b.y;
        f[8 * j + 4] += cc.x; f[8 * j + 5] += cc.y; f[8 * j + 6] += dd.x; f[8 * j + 7] += dd.y;
      }
    }
  }
  if (p.relu) {
#pragma unroll
    for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
  }
  if (p.out_f32) {
    float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + pos * p.Cout + col);
#pragma unroll
    for (int j = 0; j < 4; ++j) op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
  } else {
    st_global_v8(reinterpret_cast<__nv_bfloat16*>(p.out) + pos * p.Cout + col,
                 make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7])),
                 make_uint4(pack_bf16x2(f[8], f[9]), pack_bf16x2(f[10], f[11]), pack_bf16x2(f[12], f[13]), pack_bf16x2(f[14], f[15])));
  }
}

// ConvLSTM cell update on one accumulator row of a gate-interleaved 128-column tile (models/conv_lstm.py:32-38:
// ci = sigmoid(Wxi x + Whi h + b), cf, cc = cf c + ci tanh(.), co, ch = co tanh(cc); zero peepholes): the four gates
// of 32 hidden units sit in columns [0,32) [32,64) [64,96) [96,128) of the tile.  Writes the pre-activation gates
// (fp32, standard [i|f|g|o] layout, for the backward pass), the new cell state (fp32) and the new hidden state
// (bf16) twice: as the next step's GEMM operand and into its slot of the merged (b, t) frame map.
T2V_DEVINL void lstm_epilogue_row(const IgemmParams& p, uint32_t taddr, size_t pos, int col0, bool row_ok) {
  const int Hd = p.Cout >> 2;
  const int unit0 = (col0 >> 7) << 5;
  const size_t n = pos / (size_t)p.lstm_plane;
  const size_t pos2 = (n * p.lstm_steps + p.lstm_t) * p.lstm_plane + (pos - n * p.lstm_plane);
#pragma unroll 1
  for (int u = 0; u < 32; u += 8) {
    uint32_t vi[8], vf[8], vg[8], vo[8];
    tmem_ld8(taddr + (uint32_t)u, vi);
    tmem_ld8(taddr + (uint32_t)(32 + u), vf);
    tmem_ld8(taddr + (uint32_t)(64 + u), vg);
    tmem_ld8(taddr + (uint32_t)(96 + u), vo);
    tmem_ld_wait();                      // (the TMEM loads are warp-collective: rows outside the tensor only skip memory)
    if (!row_ok) continue;
    float gi[8], gf[8], gg[8], go[8], cn[8], hv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      gi[j] = __uint_as_float(vi[j]) + p.bias[col0 + u + j];
      gf[j] = __uint_as_float(vf[j]) + p.bias[col0 + 32 + u + j];
      gg[j] = __uint_as_float(vg[j]) + p.bias[col0 + 64 + u + j];
      go[j] = __uint_as_float(vo[j]) + p.bias[col0 + 96 + u + j];
    }
    const size_t hidx = pos * Hd + unit0 + u;
    float cp[8];
    if (p.c_prev != nullptr) {
      const float4 a = *reinterpret_cast<const float4*>(p.c_prev + hidx), b = *reinterpret_cast<const float4*>(p.c_prev + hidx + 4);
      cp[0] = a.x; cp[1] = a.y; cp[2] = a.z; cp[3] = a.w; cp[4] = b.x; cp[5] = b.y; cp[6] = b.z; cp[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) cp[j] = 0.f;
    }
    float* gp = p.gates_out + pos * (size_t)p.Cout + unit0 + u;
    *reinterpret_cast<float4*>(gp) = make_float4(gi[0], gi[1], gi[2], gi[3]);
    *reinterpret_cast<float4*>(gp + 4) = make_float4(gi[4], gi[5], gi[6], gi[7]);
    *reinterpret_cast<float4*>(gp + Hd) = make_float4(gf[0], gf[1], gf[2], gf[3]);
    *reinterpret_cast<float4*>(gp + Hd + 4) = make_float4(gf[4], gf[5], gf[6], gf[7]);
    *reinterpret_cast<float4*>(gp + 2 * Hd) = make_float4(gg[0], gg[1], gg[2], gg[3]);
    *reinterpret_cast<float4*>(gp + 2 * Hd + 4) = make_float4(gg[4], gg[5], gg[6], gg[7]);
    *reinterpret_cast<float4*>(gp + 3 * Hd) = make_float4(go[0], go[1], go[2], go[3]);
    *reinterpret_cast<float4*>(gp + 3 * Hd + 4) = make_float4(go[4], go[5], go[6], go[7]);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float si = 1.f / (1.f + __expf(-gi[j]));
      const float sf = 1.f / (1.f + __expf(-gf[j]));
      const float so = 1.f / (1.f + __expf(-go[j]));
      cn[j] = sf * cp[j] + si * tanhf(gg[j]);
      hv[j] = so * tanhf(cn[j]);
    }
    *reinterpret_cast<float4*>(p.c_out + hidx) = make_float4(cn[0], cn[1], cn[2], cn[3]);
    *reinterpret_cast<float4*>(p.c_out + hidx + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
    const uint4 hb = make_uint4(pack_bf16x2(hv[0], hv[1]), pack_bf16x2(hv[2], hv[3]), pack_bf16x2(hv[4], hv[5]),
                                pack_bf16x2(hv[6], hv[7]));
    *reinterpret_cast<uint4*>(p.h_out + hidx) = hb;
    *reinterpret_cast<uint4*>(p.h_merged + pos2 * Hd + unit0 + u) = hb;
  }
}

// PERSISTENT: gridDim.x CTAs (a multiple of the SM count, or every tile when there are few) walk the output tiles
// tile = blockIdx.x, + gridDim.x, ...  Column tile fastest: the CTAs running at the same time share the ACTIVATION
// tile, which is then read from DRAM once instead of once per column tile (the weights of a layer, <= 19 MB, stay in
// the 126 MB L2 either way).
// The TMA ring runs ahead ACROSS tiles (no pipeline fill / drain per tile), the accumulator is double buffered in
// TMEM (2 x BN columns): the MMA warp starts tile i+1 while the epilogue warps drain tile i, and barrier init /
// TMEM allocation / descriptor prefetch are paid once per CTA instead of once per 128-row tile.
template <int BLOCK_K>
__global__ void __launch_bounds__(kThreads, 3)
igemm_fprop_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
                   const IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tfull_bar = empty_bar + p.stages;       // [2] accumulator buffer b holds a finished tile
  uint64_t* tempty_bar = tfull_bar + 2;             // [2] accumulator buffer b has been drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total = p.tiles_total;                  // m tiles * column tiles
  const int ncols = total / (p.tn * p.td * p.th * p.tw);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.aux_k_blocks > 0) {
      tma_prefetch_desc(&tmA2);
      tma_prefetch_desc(&tmB2);
    }
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 4);                 // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t buf_cols = p.tmem_cols >> 1;       // column stride between the two accumulator buffers

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int nkw = p.hi_w - p.lo_w, nkh = p.hi_h - p.lo_h;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        int mt = tile / ncols;
        const int col0 = (tile % ncols) * p.BN;
        const int tw_i = mt % p.tw; mt /= p.tw;
        const int th_i = mt % p.th; mt /= p.th;
        const int td_i = mt % p.td; mt /= p.td;
        const int n0 = mt * p.bn, d0 = td_i * p.bd, h0 = th_i * p.bh, w0 = tw_i * p.bw;
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          int t = kb / p.cblocks;
          const int c0 = (kb - t * p.cblocks) * BLOCK_K;
          const int a_w = t % nkw + p.lo_w; t /= nkw;
          const int a_h = t % nkh + p.lo_h; t /= nkh;
          const int a_d = t + p.lo_d;
          const int tap = (a_d * p.kh + a_h) * p.kw + a_w;
          uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
          uint8_t* sb = sa + p.a_bytes;
          mbar_expect_tx(&full_bar[stage], p.a_bytes + p.b_bytes);
          tma_load_5d(sa, &tmA, &full_bar[stage], c0, w0 + a_w - p.pw, h0 + a_h - p.ph,
                      d0 + a_d - p.pd, n0);
          tma_load_2d(sb, &tmB, &full_bar[stage], tap * p.Cin + c0, col0);
          if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
        // fused skip connection: y += conv1x1x1(x2, w2), accumulated into the same TMEM tile (layers.py:224-243:
        // DownBlock's identity_map convolution is added to the main path; here it is extra K of the same GEMM)
        for (int kb = 0; kb < p.aux_k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
          uint8_t* sb = sa + p.a_bytes;
          mbar_expect_tx(&full_bar[stage], p.a_bytes + p.b_bytes);
          tma_load_5d(sa, &tmA2, &full_bar[stage], kb * BLOCK_K, w0, h0, d0, n0);
          tma_load_2d(sb, &tmB2, &full_bar[stage], kb * BLOCK_K, col0);
          if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    // operands are computed warp-uniformly, only the tcgen05 instructions are predicated on the elected lane
    // (descriptors then stay in uniform registers: no ELECT/R2UR waterfall in front of every UTCHMMA)
    const uint32_t d_hi = desc_hi(SwizzleOf<BLOCK_K>::sbo, SwizzleOf<BLOCK_K>::layout);
    const uint32_t leader = elect_one();
    const int nkb = p.num_k_blocks + p.aux_k_blocks;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      mbar_wait(&tempty_bar[buf], ((uint32_t)(it >> 1) & 1u) ^ 1u);      // the epilogue drained this buffer
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)buf * buf_cols;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa16 = smem_u32(smem + (size_t)stage * p.stage_bytes) >> 4;
        const uint32_t sb16 = sa16 + (p.a_bytes >> 4);
#pragma unroll
        for (int k = 0; k < BLOCK_K / 16; ++k) {
          // advance 16 bf16 = 32 bytes along K inside the swizzle atom: +2 in the (addr>>4) field
          if (leader)
            umma_bf16_ss2(tmem_d, desc_lo(sa16 + 2u * k, 0), d_hi, desc_lo(sb16 + 2u * k, 0), d_hi, p.idesc,
                          (kb | k) != 0 ? 1u : 0u);
        }
        if (leader) {
          umma_commit(&empty_bar[stage]);
          if (kb == nkb - 1) umma_commit(&tfull_bar[buf]);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else {
    // epilogue: warp w owns TMEM lanes [32*(w%4), +32) = accumulator rows
    const int q = warp & 3;
    const int row = q * 32 + lane;
    int r = row;
    const int iw = r % p.bw; r /= p.bw;
    const int ih = r % p.bh; r /= p.bh;
    const int id = r % p.bd; r /= p.bd;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
      int mt = tile / ncols;
      const int col0 = (tile % ncols) * p.BN;
      const int tw_i = mt % p.tw; mt /= p.tw;
      const int th_i = mt % p.th; mt /= p.th;
      const int td_i = mt % p.td; mt /= p.td;
      const int n = mt * p.bn + r, d = td_i * p.bd + id, h = th_i * p.bh + ih, w = tw_i * p.bw + iw;
      const bool row_ok = (n < p.N) && (d < p.D) && (h < p.H) && (w < p.W);
      const size_t pos = (((size_t)n * p.D + d) * p.H + h) * p.W + w;
      const int buf = it & 1;
      mbar_wait(&tfull_bar[buf], (uint32_t)(it >> 1) & 1u);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)buf * buf_cols;
      if (p.lstm) {                                   // warp-uniform: the TMEM loads inside are .sync.aligned
        lstm_epilogue_row(p, taddr, pos, col0, row_ok);
        __syncwarp();
      } else {
      // software pipeline over 16-column chunks: the TMEM load of chunk c+1 is in flight while chunk c is
      // converted and stored
      uint32_t va[16], vb[16];
      tmem_ld16(taddr, va);
      for (int c = 0; c < p.BN; c += 32) {
        tmem_ld_wait();
        const bool more1 = c + 16 < p.BN;
        if (more1) tmem_ld16(taddr + (uint32_t)(c + 16), vb);
        if (row_ok && col0 + c < p.Cout) fprop_epilogue16(p, va, pos, col0 + c);
        if (more1) {
          tmem_ld_wait();
          if (c + 32 < p.BN) tmem_ld16(taddr + (uint32_t)(c + 32), va);
          if (row_ok && col0 + c + 16 < p.Cout) fprop_epilogue16(p, vb, pos, col0 + c + 16);
        }
      }
      }
      // all TMEM reads of this buffer have completed (tcgen05.wait::ld): hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------ fprop, one tile per CTA
// (short K loops / small problems: 56 registers and one accumulator buffer keep up to 6 CTAs resident per SM, which
// is what hides the load latency there; the persistent kernel below wins once a tile carries >= 8 k-blocks)
template <int BLOCK_K>
__global__ void __launch_bounds__(kThreads, 2)
igemm_fprop_simple_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
                   const IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* accum_bar = empty_bar + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // tile coordinates (1-D grid; same order as the persistent kernel)
  const int ncols = p.tiles_total / (p.tn * p.td * p.th * p.tw);
  int mt = (int)blockIdx.x / ncols;
  const int col0 = ((int)blockIdx.x % ncols) * p.BN;
  const int tw_i = mt % p.tw; mt /= p.tw;
  const int th_i = mt % p.th; mt /= p.th;
  const int td_i = mt % p.td; mt /= p.td;
  const int n0 = mt * p.bn, d0 = td_i * p.bd, h0 = th_i * p.bh, w0 = tw_i * p.bw;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.aux_k_blocks > 0) {
      tma_prefetch_desc(&tmA2);
      tma_prefetch_desc(&tmB2);
    }
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int nkw = p.hi_w - p.lo_w, nkh = p.hi_h - p.lo_h;
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        int t = kb / p.cblocks;
        const int c0 = (kb - t * p.cblocks) * BLOCK_K;
        const int a_w = t % nkw + p.lo_w; t /= nkw;
        const int a_h = t % nkh + p.lo_h; t /= nkh;
        const int a_d = t + p.lo_d;
        const int tap = (a_d * p.kh + a_h) * p.kw + a_w;
        uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
        uint8_t* sb = sa + p.a_bytes;
        mbar_expect_tx(&full_bar[stage], p.a_bytes + p.b_bytes);
        tma_load_5d(sa, &tmA, &full_bar[stage], c0, w0 + a_w - p.pw, h0 + a_h - p.ph,
                    d0 + a_d - p.pd, n0);
        tma_load_2d(sb, &tmB, &full_bar[stage], tap * p.Cin + c0, col0);
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
      // fused skip connection: y += conv1x1x1(x2, w2), accumulated into the same TMEM tile (layers.py:224-243:
      // DownBlock's identity_map convolution is added to the main path; here it is extra K of the same GEMM)
      for (int kb = 0; kb < p.aux_k_blocks; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
        uint8_t* sb = sa + p.a_bytes;
        mbar_expect_tx(&full_bar[stage], p.a_bytes + p.b_bytes);
        tma_load_5d(sa, &tmA2, &full_bar[stage], kb * BLOCK_K, w0, h0, d0, n0);
        tma_load_2d(sb, &tmB2, &full_bar[stage], kb * BLOCK_K, col0);
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    // operands are computed warp-uniformly, only the tcgen05 instructions are predicated on the elected lane
    // (descriptors then stay in uniform registers: no ELECT/R2UR waterfall in front of every UTCHMMA)
    const uint32_t d_hi = desc_hi(SwizzleOf<BLOCK_K>::sbo, SwizzleOf<BLOCK_K>::layout);
    const uint32_t leader = elect_one();
    const int nkb = p.num_k_blocks + p.aux_k_blocks;
    for (int kb = 0; kb < nkb; ++kb) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint32_t sa16 = smem_u32(smem + (size_t)stage * p.stage_bytes) >> 4;
      const uint32_t sb16 = sa16 + (p.a_bytes >> 4);
#pragma unroll
      for (int k = 0; k < BLOCK_K / 16; ++k) {
        // advance 16 bf16 = 32 bytes along K inside the swizzle atom: +2 in the (addr>>4) field
        if (leader)
          umma_bf16_ss2(tmem_base, desc_lo(sa16 + 2u * k, 0), d_hi, desc_lo(sb16 + 2u * k, 0), d_hi, p.idesc,
                        (kb | k) != 0 ? 1u : 0u);
      }
      if (leader) {
        umma_commit(&empty_bar[stage]);
        if (kb == nkb - 1) umma_commit(accum_bar);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1u; }
    }
  } else {
    // epilogue: warp w owns TMEM lanes [32*(w%4), +32) = accumulator rows
    const int q = warp & 3;
    const int row = q * 32 + lane;
    int r = row;
    const int iw = r % p.bw; r /= p.bw;
    const int ih = r % p.bh; r /= p.bh;
    const int id = r % p.bd; r /= p.bd;
    const int n = n0 + r, d = d0 + id, h = h0 + ih, w = w0 + iw;
    const bool row_ok = (n < p.N) && (d < p.D) && (h < p.H) && (w < p.W);
    const size_t pos = (((size_t)n * p.D + d) * p.H + h) * p.W + w;
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    for (int c = 0; c < p.BN; c += 16) {
      uint32_t v[16];
      tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, v);
      tmem_ld_wait();
      const int col = col0 + c;
      if (row_ok && col < p.Cout) {
        float f[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j]);
        if (p.bias != nullptr) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 b = *reinterpret_cast<const float4*>(p.bias + col + j);
            f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
          }
        }
        if (p.residual != nullptr) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.residual + pos * p.Cout + col);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint4 u = rp[j];
            const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), cc = unpack_bf16x2(u.z),
                         dd = unpack_bf16x2(u.w);
            if (p.relu_mask) {      // the pointer is a ReLU reference: dx = dgrad(dy) * (ref > 0)
              f[8 * j + 0] = a.x > 0.f ? f[8 * j + 0] : 0.f; f[8 * j + 1] = a.y > 0.f ? f[8 * j + 1] : 0.f;
              f[8 * j + 2] = b.x > 0.f ? f[8 * j + 2] : 0.f; f[8 * j + 3] = b.y > 0.f ? f[8 * j + 3] : 0.f;
              f[8 * j + 4] = cc.x > 0.f ? f[8 * j + 4] : 0.f; f[8 * j + 5] = cc.y > 0.f ? f[8 * j + 5] : 0.f;
              f[8 * j + 6] = dd.x > 0.f ? f[8 * j + 6] : 0.f; f[8 * j + 7] = dd.y > 0.f ? f[8 * j + 7] : 0.f;
            } else {
              f[8 * j + 0] += a.x; f[8 * j + 1] += a.y; f[8 * j + 2] += b.x; f[8 * j + 3] += b.y;
              f[8 * j + 4] += cc.x; f[8 * j + 5] += cc.y; f[8 * j + 6] += dd.x; f[8 * j + 7] += dd.y;
            }
          }
        }
        if (p.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
        }
        if (p.out_f32) {
          float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + pos * p.Cout + col);
#pragma unroll
          for (int j = 0; j < 4; ++j) op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        } else {
          st_global_v8(reinterpret_cast<__nv_bfloat16*>(p.out) + pos * p.Cout + col,
                       make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7])),
                       make_uint4(pack_bf16x2(f[8], f[9]), pack_bf16x2(f[10], f[11]), pack_bf16x2(f[12], f[13]), pack_bf16x2(f[14], f[15])));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------ wgrad
// One CTA: output tile dW[co0:co0+128, tap, ci0:ci0+BN] partial-summed over a range of position
// boxes (64 positions per k-block).  dy box -> A (MN-major, two 64-channel atoms), shifted x box -> B.
static constexpr int kWgradPos = 64;

__global__ void __launch_bounds__(kThreads, 2)
igemm_wgrad_kernel(const __grid_constant__ CUtensorMap tmDy, const __grid_constant__ CUtensorMap tmX,
                   const IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* accum_bar = empty_bar + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int co0 = blockIdx.x * 128;
  const int ci0 = blockIdx.y * p.BN;
  // blockIdx.z = split * ntaps + tap (tap fastest): the CTAs that share a position range (all taps and column tiles of
  // one split) are launched together and walk it at the same pace, so the range is read from DRAM once and served to
  // the others from L2.  With the split fastest (round 1) the taps of a range ran in different waves: ncu showed
  // dram__bytes_read = 2-3x the operand bytes.
  const int nkw = p.hi_w - p.lo_w, nkh = p.hi_h - p.lo_h;
  const int ntaps_live = nkw * nkh * (p.hi_d - p.lo_d);
  const int split = (int)blockIdx.z / ntaps_live;
  int t = (int)blockIdx.z % ntaps_live;
  const int a_w = t % nkw + p.lo_w; t /= nkw;
  const int a_h = t % nkh + p.lo_h; t /= nkh;
  const int a_d = t + p.lo_d;
  const int tap = (a_d * p.kh + a_h) * p.kw + a_w;
  // position boxes handled by this split
  const int per = (p.tiles_total + p.splits - 1) / p.splits;
  const int t_begin = split * per;
  const int t_end = min(p.tiles_total, t_begin + per);
  const int nkb = max(0, t_end - t_begin);
  constexpr uint32_t kBoxBytes = kWgradPos * 128;  // 64 positions x 64 channels x bf16

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmDy);
    tma_prefetch_desc(&tmX);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (nkb > 0) {
    if (warp == 0) {
      if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        const int nb_boxes = p.BN / 64;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          int mt = t_begin + kb;
          const int tw_i = mt % p.tw; mt /= p.tw;
          const int th_i = mt % p.th; mt /= p.th;
          const int td_i = mt % p.td; mt /= p.td;
          const int n0 = mt * p.bn, d0 = td_i * p.bd, h0 = th_i * p.bh, w0 = tw_i * p.bw;
          uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
          uint8_t* sb = sa + 2 * kBoxBytes;
          mbar_expect_tx(&full_bar[stage], (2 + nb_boxes) * kBoxBytes);
          tma_load_5d(sa, &tmDy, &full_bar[stage], co0, w0, h0, d0, n0);
          tma_load_5d(sa + kBoxBytes, &tmDy, &full_bar[stage], co0 + 64, w0, h0, d0, n0);
          for (int j = 0; j < nb_boxes; ++j)
            tma_load_5d(sb + j * kBoxBytes, &tmX, &full_bar[stage], ci0 + 64 * j, w0 + a_w - p.pw,
                        h0 + a_h - p.ph, d0 + a_d - p.pd, n0);
          if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
      }
    } else if (warp == 1) {
      int stage = 0;
      uint32_t phase = 0;
      // MN-major, 128B swizzle: atom = 64 channels x 8 positions (1024 B); SBO = next 8 positions,
      // LBO = next 64-channel atom (one TMA box further).  Warp-uniform operands, elected-lane issue.
      const uint32_t d_hi = desc_hi(1024, 2);
      const uint32_t leader = elect_one();
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa16 = smem_u32(smem + (size_t)stage * p.stage_bytes) >> 4;
        const uint32_t sb16 = sa16 + ((2 * kBoxBytes) >> 4);
#pragma unroll
        for (int k = 0; k < kWgradPos / 16; ++k) {
          // 16 positions further = 16 rows of 128 B = 2048 B -> +128 in the (addr>>4) field
          if (leader)
            umma_bf16_ss2(tmem_base, desc_lo(sa16 + 128u * k, kBoxBytes), d_hi, desc_lo(sb16 + 128u * k, kBoxBytes),
                          d_hi, p.idesc, (kb | k) != 0 ? 1u : 0u);
        }
        if (leader) {
          umma_commit(&empty_bar[stage]);
          if (kb == nkb - 1) umma_commit(accum_bar);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
    } else {
      const int q = warp & 3;
      const int co = co0 + q * 32 + lane;
      mbar_wait(accum_bar, 0);
      tc_fence_after();
      for (int c = 0; c < p.BN; c += 16) {
        uint32_t v[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, v);
        tmem_ld_wait();
        const int ci = ci0 + c;
        if (co < p.Cout && ci < p.Cin) {
          float* dst = p.dw + ((size_t)co * p.taps_total + tap) * p.Cin + ci;
          if (p.atomic_out) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              red_add_v4(dst + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                         __uint_as_float(v[j + 3]));
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              reinterpret_cast<float4*>(dst)[j] =
                  make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                              __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------ host side
// Optional per-launch timing (bench.py roofline): CUDA events on the launching stream around every
// engine launch; t2v_profile_read() sums elapsed time and useful (live-tap) FLOPs per kernel kind.
bool g_prof_on = false;
static std::vector<ProfRec> g_prof;
static double g_prof_next_scale = 1.0;
void prof_enable(int on) { g_prof_on = on != 0; }
// fraction of the NEXT profiled launch's channels that are real (not zero padding): RGB 3 -> 16, attention
// theta / phi 4 -> 16, render 3 -> 16; the roofline numerator counts real channels only
void prof_next_scale(double s) { g_prof_next_scale = s; }
void prof_begin(cudaStream_t s, ProfRec* r, int kind, double flops, const t2v_conv_geom* g, int ctas) {
  r->kind = kind; r->flops = flops * g_prof_next_scale; r->g = *g; r->ctas = ctas;
  g_prof_next_scale = 1.0;
  cudaEventCreate(&r->a); cudaEventCreate(&r->b);
  cudaEventRecord(r->a, s);
}
void prof_end(cudaStream_t s, ProfRec* r) { cudaEventRecord(r->b, s); g_prof.push_back(*r); }
// out[kind*3 + {0,1,2}] = {milliseconds, flops, launches}; kind 0 = generic fprop/dgrad, 1 = generic wgrad,
// 2 = halo-resident fprop/dgrad, 3 = halo-resident wgrad.  nkinds = 2 folds the halo kernels into 0 / 1.
void prof_read(double* out, int nkinds) {
  for (int i = 0; i < 3 * nkinds; ++i) out[i] = 0.0;
  const char* dump = getenv("T2V_PROFILE_DUMP");
  FILE* f = dump ? fopen(dump, "a") : nullptr;
  for (auto& r : g_prof) {
    cudaEventSynchronize(r.b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.a, r.b);
    if (f)
      fprintf(f, "%d,%d,%d,%d,%d,%d,%d,%d,%d,%d,%d,%.6f,%.0f\n", r.kind >= 4 ? r.kind - 4 : r.kind % 2, r.g.N, r.g.D, r.g.H, r.g.W, r.g.Cin, r.g.Cout,
              r.g.kd, r.g.kh, r.g.kw, r.ctas, ms, r.flops);
    const int kk = nkinds >= 6 ? r.kind : (r.kind >= 4 ? (r.kind - 4) % nkinds : r.kind % nkinds);
    out[kk * 3 + 0] += ms; out[kk * 3 + 1] += r.flops; out[kk * 3 + 2] += 1.0;
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  if (f) fclose(f);
  g_prof.clear();
}

// fprop: shared memory of a CTA on small-stage (<= 12 KB) problems of more than four waves, one tile / persistent
static constexpr uint32_t kFpropSmallSmemKB = 32, kFpropSmallSmemKBPersist = 48;
// fprop: the persistent kernel runs when a tile's K (main + fused skip) reaches this many channels
static constexpr int kFpropPersistMinK = 512;
// wgrad: go beyond two waves of 148 only while each CTA still sums this many position boxes
static constexpr int kWgradMinBoxes = 32;

static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
static int pow2_floor(int v) {
  int r = 1;
  while (r * 2 <= v) r *= 2;
  return r;
}
static int pow2_ceil(int v) {
  int r = 1;
  while (r < v) r *= 2;
  return r;
}

// Choose a position box (bn,bd,bh,bw) with product == rows (a power of two).
static void choose_box(int rows, int N, int D, int H, int W, int* bn, int* bd, int* bh, int* bw) {
  int rem = rows;
  *bw = pow2_ceil(W) < rem ? pow2_ceil(W) : rem; rem /= *bw;
  *bh = pow2_ceil(H) < rem ? pow2_ceil(H) : rem; rem /= *bh;
  *bd = pow2_ceil(D) < rem ? pow2_ceil(D) : rem; rem /= *bd;
  *bn = rem;
  (void)N;
}

static void live_taps(int k, int extent, int* lo, int* hi) {
  // a +-1 tap along an axis of extent 1 only ever reads padding
  if (k == 3 && extent == 1) { *lo = 1; *hi = 2; }
  else { *lo = 0; *hi = k; }
}

bool igemm_fprop_supported(const t2v_conv_geom* g) {
  if (g->Cin % 16 || g->Cout % 16) return false;
  if (g->Cin <= 0 || g->Cout <= 0 || g->N <= 0) return false;
  auto okk = [](int k) { return k == 1 || k == 3; };
  return okk(g->kd) && okk(g->kh) && okk(g->kw);
}

bool igemm_wgrad_supported(const t2v_conv_geom* g) {
  // channel counts below 64 ride on TMA out-of-bounds zero fill of the 64-channel boxes
  return igemm_fprop_supported(g);
}

static int fill_common(IgemmParams& p, const t2v_conv_geom* g, const ConvWindow* win = nullptr) {
  p.N = g->N; p.D = g->D; p.H = g->H; p.W = g->W; p.Cin = g->Cin; p.Cout = g->Cout;
  p.kd = g->kd; p.kh = g->kh; p.kw = g->kw;
  p.pd = g->kd / 2; p.ph = g->kh / 2; p.pw = g->kw / 2;
  live_taps(g->kd, g->D, &p.lo_d, &p.hi_d);
  live_taps(g->kh, g->H, &p.lo_h, &p.hi_h);
  live_taps(g->kw, g->W, &p.lo_w, &p.hi_w);
  if (win) {
    p.lo_d = win->lo_d; p.hi_d = win->hi_d; p.lo_h = win->lo_h; p.hi_h = win->hi_h; p.lo_w = win->lo_w; p.hi_w = win->hi_w;
  }
  p.taps_total = g->kd * g->kh * g->kw;
  return (p.hi_d - p.lo_d) * (p.hi_h - p.lo_h) * (p.hi_w - p.lo_w);
}

int igemm_fprop_launch_aux(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                           const void* residual, void* y, uint32_t flags, cudaStream_t stream, const void* x2,
                           const void* w2, int Cin2, const LstmEpi* lstm = nullptr, const ConvWindow* win = nullptr);

int igemm_fprop_launch(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                       const void* residual, void* y, uint32_t flags, cudaStream_t stream) {
  return igemm_fprop_launch_aux(g, x, w, bias, residual, y, flags, stream, nullptr, nullptr, 0);
}

// x2 / w2 / Cin2: optional fused 1x1x1 convolution of a second tensor over the same positions (w2 bf16 [Cout][Cin2])
int igemm_fprop_launch_aux(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                           const void* residual, void* y, uint32_t flags, cudaStream_t stream, const void* x2,
                           const void* w2, int Cin2, const LstmEpi* lstm, const ConvWindow* win) {
  if (!igemm_fprop_supported(g)) return T2V_ERR_ARG;
  if (win && (x2 || lstm || win->lo_d < 0 || win->hi_d > g->kd || win->lo_h < 0 || win->hi_h > g->kh || win->lo_w < 0 ||
              win->hi_w > g->kw || win->lo_d >= win->hi_d || win->lo_h >= win->hi_h || win->lo_w >= win->hi_w))
    return T2V_ERR_ARG;
  if (lstm && (g->Cout % 128 || !bias || !lstm->c_out || !lstm->gates || !lstm->h_out || !lstm->h_merged ||
               lstm->steps <= 0 || lstm->t < 0 || lstm->t >= lstm->steps))
    return T2V_ERR_ARG;
  IgemmParams p{};
  const int ntaps = fill_common(p, g, win);
  const int BLOCK_K = (g->Cin % 64 == 0) ? 64 : (g->Cin % 32 == 0 ? 32 : 16);
  choose_box(128, g->N, g->D, g->H, g->W, &p.bn, &p.bd, &p.bh, &p.bw);
  p.tn = (g->N + p.bn - 1) / p.bn; p.td = (g->D + p.bd - 1) / p.bd;
  p.th = (g->H + p.bh - 1) / p.bh; p.tw = (g->W + p.bw - 1) / p.bw;
  p.BN = g->Cout >= 128 ? 128 : g->Cout;
  const int mtiles_total = p.tn * p.td * p.th * p.tw;
  // small problems: narrower N tiles -> more CTAs (the kernel is load-latency bound there, not tensor bound)
  if (!lstm)
    while (p.BN > 64 && p.BN % 32 == 0 && mtiles_total * ((g->Cout + p.BN - 1) / p.BN) < 120) p.BN /= 2;
  p.cblocks = g->Cin / BLOCK_K;
  p.num_k_blocks = ntaps * p.cblocks;
  if (x2 != nullptr) {
    if (!w2 || Cin2 <= 0 || Cin2 % BLOCK_K) return T2V_ERR_ARG;
    p.aux_k_blocks = Cin2 / BLOCK_K;
  }
  p.a_bytes = 128u * BLOCK_K * 2u;
  p.b_bytes = (uint32_t)p.BN * BLOCK_K * 2u;
  p.stage_bytes = (p.a_bytes + p.b_bytes + 1023u) & ~1023u;
  // many CTAs: cap shared memory at half an SM so that two CTAs are co-resident and one CTA's prologue /
  // epilogue overlaps the other's main loop (TMEM: 2 x BN <= 512 columns)
  const int total_ctas = mtiles_total * ((g->Cout + p.BN - 1) / p.BN);
  uint32_t budget = total_ctas > 222 ? 106496u : 196608u;
  // short K loops over small tiles are latency bound per CTA: trade pipeline depth for residency (measured:
  // 32->32 channels at 64x64, 9 k-blocks of 10 KB: 0.166 -> 0.082 ms with 3 stages and 6 CTAs per SM)
  // persistent + double-buffered accumulator: more than one wave of tiles and K >= kFpropPersistMinK per tile
  // (measured in situ at b = 2048: 64..1024-channel 3x3(x3) layers +15..30 %, 1x1 / 16-32-channel layers -10 %)
  const bool persist = lstm != nullptr ||        // (the fused LSTM epilogue lives in the persistent kernel)
      (total_ctas > 296 && (p.num_k_blocks + p.aux_k_blocks) * BLOCK_K >= kFpropPersistMinK);
  if (p.stage_bytes <= 12288u && total_ctas > 4 * 148)
    budget = (persist ? kFpropSmallSmemKBPersist : kFpropSmallSmemKB) * 1024u;
  int stages = (int)(budget / p.stage_bytes);
  if (stages < 2) stages = 2;
  if (stages > 8) stages = 8;
  // one tile per CTA: no point in more stages than k-blocks; persistent: the ring runs ahead into the next tiles
  if (!persist && stages > p.num_k_blocks + p.aux_k_blocks)
    stages = p.num_k_blocks + p.aux_k_blocks < 2 ? 2 : p.num_k_blocks + p.aux_k_blocks;
  p.stages = stages;
  p.idesc = make_idesc_bf16(128, (uint32_t)p.BN, 0, 0);
  // persistent: two accumulator buffers (double-buffered epilogue), each a power-of-two column count >= BN
  p.tmem_cols = persist ? 2u * (uint32_t)(pow2_ceil(p.BN) < 16 ? 16 : pow2_ceil(p.BN))
                        : (uint32_t)(pow2_ceil(p.BN) < 32 ? 32 : pow2_ceil(p.BN));
  p.bias = bias;
  p.residual = reinterpret_cast<const __nv_bfloat16*>(residual);
  p.out = y;
  p.out_f32 = (flags & T2V_EPI_OUT_F32) ? 1 : 0;
  p.relu = (flags & T2V_EPI_RELU) ? 1 : 0;
  p.relu_mask = (flags & T2V_EPI_RELU_MASK) ? 1 : 0;
  p.tiles_total = total_ctas;
  if (lstm) {
    p.lstm = 1; p.lstm_t = lstm->t; p.lstm_steps = lstm->steps; p.lstm_plane = g->D * g->H * g->W;
    p.c_prev = lstm->c_prev; p.c_out = lstm->c_out; p.gates_out = lstm->gates;
    p.h_out = reinterpret_cast<__nv_bfloat16*>(lstm->h_out);
    p.h_merged = reinterpret_cast<__nv_bfloat16*>(lstm->h_merged);
  }

  CUtensorMap tmA, tmB;
  int rc = make_act_map(&tmA, x, g->N, win ? win->iD : g->D, win ? win->iH : g->H, win ? win->iW : g->W, g->Cin, BLOCK_K,
                        p.bw, p.bh, p.bd, p.bn);
  if (rc) return rc;
  rc = make_w_map(&tmB, w, g->Cout, p.taps_total * g->Cin, BLOCK_K, p.BN);
  if (rc) return rc;
  CUtensorMap tmA2 = tmA, tmB2 = tmB;
  if (p.aux_k_blocks > 0) {
    rc = make_act_map(&tmA2, x2, g->N, g->D, g->H, g->W, Cin2, BLOCK_K, p.bw, p.bh, p.bd, p.bn);
    if (rc) return rc;
    rc = make_w_map(&tmB2, w2, g->Cout, Cin2, BLOCK_K, p.BN);
    if (rc) return rc;
  }

  const size_t smem = (size_t)p.stages * p.stage_bytes + 1024 + (2 * p.stages + 4) * 8 + 16;
  if (!persist) {                               // one tile per CTA (grid = m tiles x column tiles)
    dim3 grid2((unsigned)total_ctas, 1, 1);
    auto launch2 = [&](auto kern) {
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      kern<<<grid2, kThreads, smem, stream>>>(tmA, tmB, tmA2, tmB2, p);
    };
    ProfRec rec2;
    if (g_prof_on)
      prof_begin(stream, &rec2, 0,
                 2.0 * g->N * g->D * g->H * g->W * ((double)g->Cin * ntaps + (double)(x2 ? Cin2 : 0)) * g->Cout, g,
                 total_ctas);
    if (BLOCK_K == 64) launch2(igemm_fprop_simple_kernel<64>);
    else if (BLOCK_K == 32) launch2(igemm_fprop_simple_kernel<32>);
    else launch2(igemm_fprop_simple_kernel<16>);
    if (g_prof_on) prof_end(stream, &rec2);
    count_launch();
    return check_last("igemm_fprop");
  }
  // persistent grid: as many CTAs as stay resident (shared memory, TMEM columns, threads), each walking
  // tiles blockIdx.x, + gridDim.x, ...
  int grid_x = total_ctas;
  auto launch = [&](auto kern) {
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    static int regs_cached[3] = {0, 0, 0};
    int& rc_ = regs_cached[BLOCK_K == 64 ? 0 : (BLOCK_K == 32 ? 1 : 2)];
    if (rc_ == 0) {
      cudaFuncAttributes fa{};
      cudaFuncGetAttributes(&fa, kern);
      rc_ = fa.numRegs > 0 ? fa.numRegs : 96;
    }
    const int regs = (rc_ + 7) & ~7;                                                    // allocation granularity
    int per_sm = 65536 / (regs * kThreads);                                             // registers ...
    if (per_sm > (int)((228u * 1024u) / (smem + 1024u))) per_sm = (int)((228u * 1024u) / (smem + 1024u));
    if (per_sm > 2048 / kThreads) per_sm = 2048 / kThreads;                             // ... shared memory, threads
    if (per_sm > (int)(512u / p.tmem_cols)) per_sm = (int)(512u / p.tmem_cols);        // ... and TMEM columns
    if (per_sm < 1) per_sm = 1;
    if (grid_x > 148 * per_sm) grid_x = 148 * per_sm;
    static const int dbg = env_int("T2V_DEBUG_LAUNCH", 0);
    if (dbg)
      fprintf(stderr, "igemm_fprop N%d D%d H%d W%d Cin%d Cout%d k%d%d%d: tiles %d grid %d stages %d stage_bytes %u smem %zu "
              "tmem_cols %u BN %d BLOCK_K %d\n", g->N, g->D, g->H, g->W, g->Cin, g->Cout, g->kd, g->kh, g->kw, total_ctas,
              grid_x, p.stages, p.stage_bytes, smem, p.tmem_cols, p.BN, BLOCK_K);
    kern<<<dim3((unsigned)grid_x, 1, 1), kThreads, smem, stream>>>(tmA, tmB, tmA2, tmB2, p);
  };
  ProfRec rec;
  if (g_prof_on)
    prof_begin(stream, &rec, 0,
               2.0 * g->N * g->D * g->H * g->W * ((double)g->Cin * ntaps + (double)(x2 ? Cin2 : 0)) * g->Cout, g,
               total_ctas);
  if (BLOCK_K == 64) launch(igemm_fprop_kernel<64>);
  else if (BLOCK_K == 32) launch(igemm_fprop_kernel<32>);
  else launch(igemm_fprop_kernel<16>);
  if (g_prof_on) prof_end(stream, &rec);
  count_launch();
  return check_last("igemm_fprop");
}

int igemm_wgrad_launch(const t2v_conv_geom* g, const void* dy, const void* x, float* dw, int accumulate,
                       cudaStream_t stream, const ConvWindow* win) {
  if (!igemm_wgrad_supported(g)) return T2V_ERR_ARG;
  if (win && (win->lo_d < 0 || win->hi_d > g->kd || win->lo_h < 0 || win->hi_h > g->kh || win->lo_w < 0 ||
              win->hi_w > g->kw || win->lo_d >= win->hi_d || win->lo_h >= win->hi_h || win->lo_w >= win->hi_w))
    return T2V_ERR_ARG;
  IgemmParams p{};
  const int ntaps = fill_common(p, g, win);
  choose_box(kWgradPos, g->N, g->D, g->H, g->W, &p.bn, &p.bd, &p.bh, &p.bw);
  p.tn = (g->N + p.bn - 1) / p.bn; p.td = (g->D + p.bd - 1) / p.bd;
  p.th = (g->H + p.bh - 1) / p.bh; p.tw = (g->W + p.bw - 1) / p.bw;
  p.tiles_total = p.tn * p.td * p.th * p.tw;
  p.BN = g->Cin >= 128 ? 128 : 64;
  const int mtiles = (g->Cout + 127) / 128, ntiles = (g->Cin + p.BN - 1) / p.BN;
  const int base_ctas = mtiles * ntiles * ntaps;
  // two CTAs per SM (shared memory capped at half an SM: one CTA's prologue / atomics epilogue overlaps the
  // other's main loop): fill at most two FULL waves of 2 x 148 so that no nearly empty extra wave runs
  int splits = (2 * 2 * 148) / base_ctas;
  // every split adds a full Cout x taps x Cin round of fp32 atomics: only go beyond two waves of 148 when each
  // CTA still sums >= kWgradMinBoxes position boxes (position-heavy layers), else the atomics of weight-heavy layers
  // dominate
  if (splits < 1 || p.tiles_total / splits < kWgradMinBoxes) splits = (2 * 148) / base_ctas;
  const int max_splits = (p.tiles_total + 3) / 4;  // keep >= 4 k-blocks per CTA
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  p.splits = splits;
  p.a_bytes = 2u * kWgradPos * 128u;
  p.b_bytes = (uint32_t)(p.BN / 64) * kWgradPos * 128u;
  p.stage_bytes = p.a_bytes + p.b_bytes;
  int stages = (int)(106496u / p.stage_bytes);
  if (stages > 8) stages = 8;
  p.stages = stages;
  p.idesc = make_idesc_bf16(128, (uint32_t)p.BN, 1, 1);
  p.tmem_cols = (uint32_t)(p.BN < 32 ? 32 : p.BN);
  p.dw = dw;
  p.atomic_out = (splits > 1 || accumulate) ? 1 : 0;

  const size_t dw_elems = (size_t)g->Cout * p.taps_total * g->Cin;
  if (!accumulate && (p.atomic_out || ntaps < p.taps_total))
    cudaMemsetAsync(dw, 0, dw_elems * sizeof(float), stream);

  CUtensorMap tmDy, tmX;
  int rc = make_act_map(&tmDy, dy, g->N, g->D, g->H, g->W, g->Cout, 64, p.bw, p.bh, p.bd, p.bn);
  if (rc) return rc;
  rc = make_act_map(&tmX, x, g->N, win ? win->iD : g->D, win ? win->iH : g->H, win ? win->iW : g->W, g->Cin, 64, p.bw,
                    p.bh, p.bd, p.bn);
  if (rc) return rc;
  const size_t smem = (size_t)p.stages * p.stage_bytes + 1024 + (2 * p.stages + 1) * 8 + 16;
  dim3 grid(mtiles, ntiles, ntaps * splits);
  cudaFuncSetAttribute(igemm_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  ProfRec rec;
  if (g_prof_on)
    prof_begin(stream, &rec, 1, 2.0 * g->N * g->D * g->H * g->W * (double)g->Cin * g->Cout * ntaps, g,
               (int)(grid.x * grid.y * grid.z));
  igemm_wgrad_kernel<<<grid, kThreads, smem, stream>>>(tmDy, tmX, p);
  if (g_prof_on) prof_end(stream, &rec);
  count_launch();
  return check_last("igemm_wgrad");
}

}  // namespace t2v
