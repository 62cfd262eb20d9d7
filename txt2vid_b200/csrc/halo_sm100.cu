// Halo-resident convolution kernels for the 64-channel 3x3(x3) layers (sm_100a).
//
// Why: for Cin = 64 the generic implicit GEMM (igemm_sm100.cu) re-reads a 16 KB activation box from
// L2 for every filter tap; with N = 64 output channels that is 24 KB of L2->SMEM traffic per 128
// tensor-core cycles and the kernel runs at the L2 bandwidth, not at the tensor-core rate (the
// discriminator stem of txt2vid/models/resnet3d.py:12-14 -- 48 % of a D pass -- sat at 113-295 TFLOP/s).
// Here ONE shared-memory tile with a one-voxel halo, [bd+2][bh+2][bw+2] rows of 64 channels (128 B,
// TMA SWIZZLE_128B, out-of-bounds zero fill = the conv padding), feeds all 27 taps: a tap is a ROW
// OFFSET into that tile.  tcgen05 shared-memory descriptors take any 16-byte-aligned start address and
// the 128B swizzle is a function of the absolute address, so row-shifted views of a TMA-written tile
// are valid operands (pinned by scripts/umma_probe.cu on a B200).
//
//   wgrad: dW[co][tap][ci] = sum_pos dy[pos,co] * x[pos+tap,ci]
//          positions are the GEMM K dimension, so each MMA instruction (K = 16 rows = two 8-voxel lines)
//          gets its own start address: no padding rows are ever multiplied.
//          A = x view, MN-major, M = 128 = [tap_a ci | tap_b ci] (two taps stacked: the second 64-channel
//          group sits LBO = (row(tap_b) - row(tap_a)) * 128 B further), B = dy tile, MN-major, N = Cout.
//          TMEM holds 512/Cout tap pairs; the taps are split over `classes` CTAs per position range.
//   fprop / dgrad (Cout = 64): D[128 voxels x 64 cout] += A[voxel + tap, ci] * W_tap[cout, ci], K-major.
//          An M tile is 16 LINES of 8 voxels (the 8-row groups of the canonical layout) a constant stride
//          (the descriptor's SBO) apart: lines along h inside one plane, or along d, so no halo row is ever
//          multiplied.  Persistent CTAs (one per SM): double-buffered halo tile, double-buffered TMEM
//          accumulators (the epilogue of tile i overlaps the MMAs of tile i+1), and a ring of 8 KB weight taps.
#include <cstdio>
#include <cstdlib>

#include "t2v_common.cuh"
#include "tmap.cuh"

namespace t2v {

static constexpr int kHaloThreads = 192;
static constexpr int kXW = 10;   // x-tile rows per h line: 8 voxels + 2 halo

struct HaloWgParams {
  int N, D, H, W, Cout;
  int kd3;                 // 1: 3x3x3 taps, 0: 1x3x3
  int bd, bh;              // interior tile (bw = 8)
  int td, th, tw, tiles_total;
  int ntaps, taps_per_cta, splits;
  int stages;
  uint32_t stage_bytes, dy_bytes, dy_box_bytes, x_bytes;
  uint32_t tmem_cols, idesc;
  int xpitch_d;            // x-tile rows per d plane = (bh+2)*kXW
  int xd_mul;              // x plane of dy plane d = xd_mul * d (2: convolution with stride 2 along d)
  float* dw;
};

__device__ __forceinline__ int halo_tap_row(int t, int kd3, int xpitch_d) {
  const int a_w = t % 3;
  const int a_h = (t / 3) % 3;
  const int a_d = kd3 ? t / 9 : 0;
  return a_d * xpitch_d + a_h * kXW + a_w;
}

__global__ void __launch_bounds__(kHaloThreads, 1)
halo_wgrad_kernel(const __grid_constant__ CUtensorMap tmDy, const __grid_constant__ CUtensorMap tmX,
                  const HaloWgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* accum_bar = empty_bar + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int t0 = blockIdx.y * p.taps_per_cta;
  const int t1 = min(p.ntaps, t0 + p.taps_per_cta);
  const int npairs = (t1 - t0 + 1) >> 1;
  const int per = (p.tiles_total + p.splits - 1) / p.splits;
  const int tile_begin = blockIdx.x * per;
  const int tile_end = min(p.tiles_total, tile_begin + per);
  const int ntiles = max(0, tile_end - tile_begin);

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

  if (ntiles > 0) {
    if (warp == 0) {
      if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        const int nboxes = p.Cout > 64 ? p.Cout >> 6 : 1;     // Cout < 64: one 64-channel box, upper channels zero filled
        for (int it = 0; it < ntiles; ++it) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          int mt = tile_begin + it;
          const int tw_i = mt % p.tw; mt /= p.tw;
          const int th_i = mt % p.th; mt /= p.th;
          const int td_i = mt % p.td; mt /= p.td;
          const int n = mt, d0 = td_i * p.bd, h0 = th_i * p.bh, w0 = tw_i * 8;
          uint8_t* sdy = smem + (size_t)stage * p.stage_bytes;
          uint8_t* sx = sdy + p.dy_bytes;
          mbar_expect_tx(&full_bar[stage], p.dy_bytes + p.x_bytes);
          for (int j = 0; j < nboxes; ++j)
            tma_load_5d(sdy + (size_t)j * p.dy_box_bytes, &tmDy, &full_bar[stage], 64 * j, w0, h0, d0, n);
          tma_load_5d(sx, &tmX, &full_bar[stage], 0, w0 - 1, h0 - 1, p.xd_mul * d0 - (p.kd3 ? 1 : 0), n);
          if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
      }
    } else if (warp == 1) {
      int stage = 0;
      uint32_t phase = 0;
      const int ksteps = (p.bd * p.bh) >> 1;     // two 8-voxel lines per MMA (K = 16 positions)
      // Everything below is computed by all 32 lanes (warp-uniform) and only the tcgen05 instructions are
      // predicated on one elected lane, so the descriptors live in uniform registers.
      // per tap pair: row offset of tap_a (>> 4) and LBO = distance to tap_b
      uint32_t off_a[8], lbo_a[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int ta = min(t0 + 2 * q, t1 - 1), tb = min(ta + 1, t1 - 1);
        const int ra = halo_tap_row(ta, p.kd3, p.xpitch_d), rb = halo_tap_row(tb, p.kd3, p.xpitch_d);
        off_a[q] = (uint32_t)ra * 8u;                                    // rows * 128 B >> 4
        lbo_a[q] = (uint32_t)(rb - ra) * 128u;
      }
      const uint32_t a_hi = desc_hi((uint32_t)kXW * 128u, 2), b_hi = desc_hi(1024, 2);
      const uint32_t leader = elect_one();
      for (int it = 0; it < ntiles; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sdy = smem_u32(smem + (size_t)stage * p.stage_bytes);
        const uint32_t sx16 = (sdy + p.dy_bytes) >> 4;
        int d = 0, h = 0;
        for (int j = 0; j < ksteps; ++j) {
          const uint32_t line16 = sx16 + (uint32_t)(d * p.xd_mul * p.xpitch_d + h * kXW) * 8u;
          const uint32_t b_lo = desc_lo((sdy >> 4) + 128u * (uint32_t)j, p.dy_box_bytes);
          const uint32_t acc = (it | j) != 0 ? 1u : 0u;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            if (q < npairs) {
              const uint32_t a_lo = desc_lo(line16 + off_a[q], lbo_a[q]);
              if (leader) umma_bf16_ss2(tmem_base + (uint32_t)(q * p.Cout), a_lo, a_hi, b_lo, b_hi, p.idesc, acc);
            }
          }
          h += 2;
          if (h >= p.bh) { h = 0; ++d; }
        }
        if (leader) {
          umma_commit(&empty_bar[stage]);
          if (it == ntiles - 1) umma_commit(accum_bar);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
    } else {
      // epilogue: TMEM lane = (tap half, ci), column = pair * Cout + co  ->  red.add into dw[co][tap][ci]
      const int q4 = warp & 3;
      const int row = q4 * 32 + lane;
      const int half = row >> 6, ci = row & 63;
      mbar_wait(accum_bar, 0);
      tc_fence_after();
      for (int q = 0; q < npairs; ++q) {
        const int tap = t0 + 2 * q + half;
        for (int c = 0; c < p.Cout; c += 16) {
          uint32_t v[16];
          tmem_ld16(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(q * p.Cout + c), v);
          tmem_ld_wait();
          if (tap < t1) {
            float* dst = p.dw + ((size_t)c * p.ntaps + tap) * 64 + ci;
#pragma unroll
            for (int j = 0; j < 16; ++j) atomicAdd(dst + (size_t)j * p.ntaps * 64, __uint_as_float(v[j]));
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
static constexpr uint32_t kSmemBudget = 227u * 1024u - 2048u;

// g describes the dy grid (for sd2: D = the number of OUTPUT planes, x has 2*D planes)
static bool halo_wgrad_plan(const t2v_conv_geom* g, HaloWgParams* p, int sd2 = 0) {
  // Cout 16 / 32 / 48: the MMA's N is the real channel count, read from the first part of the 64-channel dy box
  if (g->Cin != 64 || (g->Cout != 64 && g->Cout != 128 && !(g->Cout >= 16 && g->Cout < 64 && g->Cout % 16 == 0)))
    return false;
  if (g->kh != 3 || g->kw != 3 || (g->kd != 1 && g->kd != 3)) return false;
  if (g->W < 8 || g->H < 4) return false;
  if (g->kd == 3 && g->D < 2 && !sd2) return false;     // dead taps: the generic kernel skips them
  if (g->kd == 1 && g->D != 1) return false;
  if (sd2 && g->kd != 3) return false;
  p->N = g->N; p->D = g->D; p->H = g->H; p->W = g->W; p->Cout = g->Cout;
  p->kd3 = g->kd == 3;
  p->ntaps = g->kd * 9;
  p->xd_mul = sd2 ? 2 : 1;
  // candidate interior tiles, largest first (more reuse of the halo); need >= 2 pipeline stages
  const int cand3[][2] = {{4, 8}, {2, 8}, {2, 4}, {1, 16}, {1, 8}};
  const int cand1[][2] = {{1, 32}, {1, 16}, {1, 8}, {1, 4}, {1, 4}};
  bool ok = false;
  for (int i = 0; i < 5 && !ok; ++i) {
    const int bd = p->kd3 ? cand3[i][0] : cand1[i][0], bh = p->kd3 ? cand3[i][1] : cand1[i][1];
    if (bd > 2 && bd > g->D) continue;
    if (bd == 2 && g->D < 2) continue;
    if (bd == 1 && p->kd3 && g->D >= 2) continue;
    if (bh > 4 && bh > g->H) continue;
    const uint32_t dy_box = (uint32_t)bd * bh * 1024u;
    const uint32_t dyb = dy_box * (uint32_t)(g->Cout > 64 ? g->Cout / 64 : 1);
    const uint32_t xb = (uint32_t)((p->kd3 ? p->xd_mul * (bd - 1) + 3 : bd) * (bh + 2) * kXW) * 128u;
    const uint32_t stage = (dyb + xb + 1023u) & ~1023u;
    const int stages = (int)(kSmemBudget / stage);
    if (stages < 2) continue;
    p->bd = bd; p->bh = bh;
    p->dy_box_bytes = dy_box; p->dy_bytes = dyb; p->x_bytes = xb; p->stage_bytes = stage;
    p->stages = stages > 4 ? 4 : stages;
    ok = true;
  }
  if (!ok) return false;
  p->xpitch_d = (p->bh + 2) * kXW;
  p->td = (g->D + p->bd - 1) / p->bd; p->th = (g->H + p->bh - 1) / p->bh; p->tw = (g->W + 7) / 8;
  p->tiles_total = g->N * p->td * p->th * p->tw;
  const int max_pairs = 512 / g->Cout < 8 ? 512 / g->Cout : 8;     // the MMA warp keeps 8 tap-pair descriptors
  const int classes = (p->ntaps + 2 * max_pairs - 1) / (2 * max_pairs);
  int per = (p->ntaps + classes - 1) / classes;
  per = (per + 1) & ~1;
  p->taps_per_cta = per;
  const int npairs = per / 2;
  uint32_t cols = (uint32_t)(npairs * g->Cout);
  uint32_t tc = 32;
  while (tc < cols) tc *= 2;
  p->tmem_cols = tc;
  int splits = 148 / classes;
  if (splits > p->tiles_total) splits = p->tiles_total;
  if (splits < 1) splits = 1;
  p->splits = splits;
  p->idesc = make_idesc_bf16(128, (uint32_t)g->Cout, 1, 1);
  return true;
}

bool halo_wgrad_supported(const t2v_conv_geom* g) {
  HaloWgParams p{};
  return halo_wgrad_plan(g, &p);
}

bool halo_sd2_supported(const t2v_conv_geom* g);

// sd2 = 1: the convolution has stride 2 along d: g is the geometry of x (D planes), dy has D/2 planes
int halo_wgrad_launch(const t2v_conv_geom* g_in, const void* dy, const void* x, float* dw, int accumulate,
                      cudaStream_t stream, int sd2) {
  HaloWgParams p{};
  t2v_conv_geom gg = *g_in;
  if (sd2) {
    if (!halo_sd2_supported(g_in)) return T2V_ERR_ARG;
    gg.D = g_in->D / 2;
  }
  const t2v_conv_geom* g = &gg;
  if (!halo_wgrad_plan(g, &p, sd2)) return T2V_ERR_ARG;
  p.dw = dw;
  if (!accumulate) cudaMemsetAsync(dw, 0, (size_t)g->Cout * p.ntaps * 64 * sizeof(float), stream);
  CUtensorMap tmDy, tmX;
  int rc = make_act_map(&tmDy, dy, g->N, g->D, g->H, g->W, g->Cout, 64, 8, p.bh, p.bd, 1);
  if (rc) return rc;
  rc = make_act_map(&tmX, x, g->N, g_in->D, g->H, g->W, 64, 64, kXW, p.bh + 2,
                    p.kd3 ? p.xd_mul * (p.bd - 1) + 3 : p.bd, 1);
  if (rc) return rc;
  const size_t smem = (size_t)p.stages * p.stage_bytes + 1024 + (2 * p.stages + 1) * 8 + 16;
  const int classes = (p.ntaps + p.taps_per_cta - 1) / p.taps_per_cta;
  dim3 grid(p.splits, classes, 1);
  cudaFuncSetAttribute(halo_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  ProfRec rec;
  if (g_prof_on)
    prof_begin(stream, &rec, 3, 2.0 * g->N * g->D * g->H * g->W * 64.0 * g->Cout * p.ntaps, g,
               (int)(grid.x * grid.y));
  halo_wgrad_kernel<<<grid, kHaloThreads, smem, stream>>>(tmDy, tmX, p);
  if (g_prof_on) prof_end(stream, &rec);
  count_launch();
  return check_last("halo_wgrad");
}

// ==================================================================================== fprop / dgrad
static constexpr int kFpThreads = 224;     // warp 0: A tiles, 1: MMA, 2-5: epilogue, 6: weight ring
static constexpr int kWStagesMax = 8;
static constexpr uint32_t kWTapBytes = 64u * 128u;

// One kernel, four uses (mode):
//   0  stride-1 "same" convolution (fprop, or dgrad with the flipped pack)
//   1  fprop with stride 2 along d: output plane j reads input planes 2j-1, 2j, 2j+1
//   2  dgrad of (1), ODD  dx planes: dx[2j+1] = Wflip[0] * dy[j] + Wflip[2] * dy[j+1]
//   3  dgrad of (1), EVEN dx planes: dx[2j]   = Wflip[1] * dy[j]   (a 2-D convolution over merged (n, j))
// expressed through: the d taps of the tile (nd consecutive smem planes, weight d index wd[t]), the first input
// plane of a tile (in_dmul * d0 + in_dadd) and the output plane number q = n * oq_n + d * oq_d + oq_0.
struct HaloFpParams {
  int N, D, H, W;          // OUTPUT iteration extents (samples, planes) and the plane size
  int kd3, np, ntaps;
  int nd, wd[3];           // d taps per tile and their weight d index
  int in_dmul, in_dadd;    // TMA d coordinate of a tile = in_dmul * d0 + in_dadd
  int oq_n, oq_d, oq_0;    // output plane number of (n, d)
  int wstages;
  int t_w, t_h, t_d, tiles_total, iters;
  int th_step, td_step, tn_step;   // tile origin steps along h, d, n
  int mn, md, mh, ld, lh;          // voxel of (M tile m, line l): n0 + m*mn, d0 + m*md + l*ld, h0 + m*mh + l*lh
  int Pd, MS, LS;                  // rows per d plane, rows between M tiles, rows between lines
  int box_d, box_n, box_h;         // TMA box extents of the halo tile
  uint32_t a_bytes, a_tx, tmem_cols, idesc;
  const float* bias;
  const __nv_bfloat16* residual;
  void* out;
  int out_f32, relu, relu_mask;
};

struct FpTile { int n0, d0, h0, w0; };

__device__ __forceinline__ FpTile fp_tile(const HaloFpParams& p, int t) {
  FpTile r;
  if (t >= p.tiles_total) { r.n0 = p.N; r.d0 = 0; r.h0 = 0; r.w0 = 0; return r; }   // dummy: all zero fill
  const int tw_i = t % p.t_w; t /= p.t_w;
  const int th_i = t % p.t_h; t /= p.t_h;
  const int td_i = t % p.t_d; t /= p.t_d;
  r.w0 = tw_i * 8; r.h0 = th_i * p.th_step; r.d0 = td_i * p.td_step; r.n0 = t * p.tn_step;
  return r;
}

__global__ void __launch_bounds__(kFpThreads, 1)
halo_fprop_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                  const HaloFpParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  const int kWStages = p.wstages;
  uint8_t* sA = smem;
  uint8_t* sW = smem + 2 * (size_t)p.a_bytes;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(sW + kWStages * kWTapBytes);
  uint64_t* a_empty = a_full + 2;
  uint64_t* w_full = a_empty + 2;
  uint64_t* w_empty = w_full + kWStagesMax;
  uint64_t* acc_full = w_empty + kWStagesMax;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4);
    }
    for (int i = 0; i < kWStages; ++i) {
      mbar_init(&w_full[i], 1);
      mbar_init(&w_empty[i], 1);
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
  const int acc_cols = p.np * 64;

  if (warp == 0) {
    // ---------------- halo tiles (this CTA's own)
    if (lane == 0) {
      for (int it = 0; it < p.iters; ++it) {
        const int buf = it & 1;
        mbar_wait(&a_empty[buf], ((uint32_t)(it >> 1) & 1u) ^ 1u);
        const FpTile t = fp_tile(p, it * (int)gridDim.x + (int)blockIdx.x);
        mbar_expect_tx(&a_full[buf], p.a_tx);
        tma_load_5d(sA + (size_t)buf * p.a_bytes, &tmA, &a_full[buf], 0, t.w0 - 1, t.h0 - 1,
                    p.in_dmul * t.d0 + p.in_dadd, t.n0);
      }
    }
  } else if (warp == 6) {
    // ---------------- weight ring: one whole 64-row tap per stage
    if (lane == 0) {
      int st = 0;
      uint32_t ph = 0;
      for (int it = 0; it < p.iters; ++it) {
        int t9 = 0, a_d = 0;
        for (int tap = 0; tap < p.ntaps; ++tap) {
          mbar_wait(&w_empty[st], ph ^ 1u);
          mbar_expect_tx(&w_full[st], kWTapBytes);
          tma_load_2d(sW + (size_t)st * kWTapBytes, &tmW, &w_full[st], (p.wd[a_d] * 9 + t9) * 64, 0);
          if (++st == kWStages) { st = 0; ph ^= 1u; }
          if (++t9 == 9) { t9 = 0; ++a_d; }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issue
    int st = 0;
    uint32_t ph = 0;
    // warp-uniform operand computation; only the tcgen05 instructions are predicated on the elected lane
    const uint32_t a_hi = desc_hi((uint32_t)p.LS * 128u, 2), b_hi = desc_hi(1024, 2);
    const uint32_t ms16 = (uint32_t)p.MS * 8u;
    const uint32_t leader = elect_one();
    for (int it = 0; it < p.iters; ++it) {
      const int buf = it & 1;
      const uint32_t par = (uint32_t)(it >> 1) & 1u;
      mbar_wait(&a_full[buf], par);
      mbar_wait(&acc_empty[buf], par ^ 1u);
      tc_fence_after();
      const uint32_t a16 = smem_u32(sA + (size_t)buf * p.a_bytes) >> 4;
      const uint32_t tacc = tmem_base + (uint32_t)(buf * acc_cols);
      int a_w = 0, a_h = 0, a_d = 0;
      for (int tap = 0; tap < p.ntaps; ++tap) {
        mbar_wait(&w_full[st], ph);
        tc_fence_after();
        const uint32_t row16 = a16 + (uint32_t)(a_d * p.Pd + a_h * kXW + a_w) * 8u;
        const uint32_t b16 = smem_u32(sW + (size_t)st * kWTapBytes) >> 4;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          if (m < p.np) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t a_lo = desc_lo(row16 + (uint32_t)m * ms16 + 2u * k, 0);
              const uint32_t b_lo = desc_lo(b16 + 2u * k, 0);
              if (leader)
                umma_bf16_ss2(tacc + (uint32_t)(m * 64), a_lo, a_hi, b_lo, b_hi, p.idesc, (tap | k) != 0 ? 1u : 0u);
            }
          }
        }
        if (leader) umma_commit(&w_empty[st]);
        __syncwarp();
        if (++st == kWStages) { st = 0; ph ^= 1u; }
        if (++a_w == 3) { a_w = 0; if (++a_h == 3) { a_h = 0; ++a_d; } }
      }
      if (leader) {
        umma_commit(&a_empty[buf]);
        umma_commit(&acc_full[buf]);
      }
      __syncwarp();
    }
  } else {
    // ---------------- epilogue (warps 2-5): TMEM lane = line*8 + w
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int l = row >> 3, wv = row & 7;
    for (int it = 0; it < p.iters; ++it) {
      const int buf = it & 1;
      const FpTile t = fp_tile(p, it * (int)gridDim.x + (int)blockIdx.x);
      mbar_wait(&acc_full[buf], (uint32_t)(it >> 1) & 1u);
      tc_fence_after();
      for (int m = 0; m < p.np; ++m) {
        const int n = t.n0 + m * p.mn, d = t.d0 + m * p.md + l * p.ld, h = t.h0 + m * p.mh + l * p.lh;
        const int w = t.w0 + wv;
        const bool row_ok = (n < p.N) && (d < p.D) && (h < p.H) && (w < p.W);
        const size_t pos = (((size_t)n * p.oq_n + (size_t)(d * p.oq_d + p.oq_0)) * p.H + h) * p.W + w;
#pragma unroll
        for (int c = 0; c < 64; c += 16) {
          uint32_t v[16];
          tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * acc_cols + m * 64 + c), v);
          tmem_ld_wait();
          if (row_ok) {
            float f[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j]);
            if (p.bias != nullptr) {
#pragma unroll
              for (int j = 0; j < 16; j += 4) {
                const float4 b = *reinterpret_cast<const float4*>(p.bias + c + j);
                f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
              }
            }
            if (p.residual != nullptr) {
              const uint4* rp = reinterpret_cast<const uint4*>(p.residual + pos * 64 + c);
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
              float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + pos * 64 + c);
#pragma unroll
              for (int j = 0; j < 4; ++j) op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
            } else {
              st_global_v8(reinterpret_cast<__nv_bfloat16*>(p.out) + pos * 64 + c,
                           make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7])),
                           make_uint4(pack_bf16x2(f[8], f[9]), pack_bf16x2(f[10], f[11]), pack_bf16x2(f[12], f[13]), pack_bf16x2(f[14], f[15])));
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// g: geometry of the tensor the kernel READS (x for modes 0/1, dy for modes 2/3); see HaloFpParams for the modes
static bool halo_fprop_plan(const t2v_conv_geom* g, HaloFpParams* p, int mode = 0) {
  if (g->Cin != 64 || g->Cout != 64) return false;
  if (g->kh != 3 || g->kw != 3 || (g->kd != 1 && g->kd != 3)) return false;
  if (g->W < 8) return false;
  if (mode != 0 && (g->kd != 3 || g->H < 16)) return false;
  p->N = g->N; p->D = g->D; p->H = g->H; p->W = g->W;
  p->kd3 = g->kd == 3;
  p->mn = p->md = p->mh = p->ld = p->lh = 0;
  p->t_w = (g->W + 7) / 8;
  p->nd = p->kd3 ? 3 : 1;
  p->wd[0] = 0; p->wd[1] = 1; p->wd[2] = 2;
  p->in_dmul = 1; p->in_dadd = p->kd3 ? -1 : 0;
  p->oq_n = g->D; p->oq_d = 1; p->oq_0 = 0;
  int planes_d = 1, planes_n = 1;          // TMA box extents along d and n
  bool merged2d = !p->kd3;                 // 16 lines along h, np consecutive SAMPLES per tile
  if (mode == 1) {                         // g = x geometry (D planes, even): output has D/2 planes
    if (g->D < 2 || (g->D & 1)) return false;
    p->D = g->D / 2;
    p->oq_n = p->D;
    if (p->D == 1) {                       // only output plane 0: reads planes 0, 1 (plane -1 is padding): 18 taps,
      p->nd = 2; p->wd[0] = 1; p->wd[1] = 2;   // M tiles = np samples (box: 2 planes x np samples)
      p->in_dmul = 0; p->in_dadd = 0;
      p->np = 2; p->mn = 1; p->lh = 1;
      p->Pd = 18 * kXW; p->MS = 2 * p->Pd; p->LS = kXW;
      p->th_step = 16; p->td_step = 1; p->tn_step = p->np;
      planes_d = 2; planes_n = p->np;
      p->t_h = (g->H + 15) / 16; p->t_d = 1;
      p->tiles_total = ((g->N + p->np - 1) / p->np) * p->t_h * p->t_w;
      merged2d = false;
      goto done;
    }
    p->in_dmul = 2; p->in_dadd = -1;
  } else if (mode == 2) {                  // g = dy geometry (D = output planes of the forward conv)
    if (g->D < 2) return false;            // D == 1: only tap 0 is live -> the caller uses mode 3 with wd = 0
    p->nd = 2; p->wd[0] = 0; p->wd[1] = 2;
    p->in_dmul = 1; p->in_dadd = 0;
    p->oq_n = 2 * g->D; p->oq_d = 2; p->oq_0 = 1;
  } else if (mode == 3 || mode == 4) {     // 2-D over merged (n, j); mode 4: the odd plane of a one-plane dy
    p->N = g->N * g->D; p->D = 1;
    p->kd3 = 0; p->nd = 1; p->wd[0] = mode == 3 ? 1 : 0;
    p->in_dmul = 0; p->in_dadd = 0;
    p->oq_n = 2; p->oq_d = 0; p->oq_0 = mode == 3 ? 0 : 1;
    merged2d = true;
  }
  if (!merged2d) {
    if (g->D < 2 && mode == 0) return false;
    if (g->H >= 16) {                 // 16 lines along h inside one d plane; a tile = np planes
      p->np = mode == 1 ? 1 : 2;
      p->Pd = 18 * kXW; p->MS = (p->in_dmul ? p->in_dmul : 1) * p->Pd; p->LS = kXW;
      p->th_step = 16; p->td_step = p->np; p->tn_step = 1;
      p->md = 1; p->lh = 1;
      planes_d = (p->in_dmul ? p->in_dmul : 1) * (p->np - 1) + p->nd;
    } else if (mode == 0 && g->D >= 16 && g->H >= 2) {   // 16 lines along d; a tile = np h rows
      p->np = 2;
      p->Pd = (p->np + 2) * kXW; p->MS = kXW; p->LS = p->Pd;
      p->th_step = p->np; p->td_step = 16; p->tn_step = 1;
      p->mh = 1; p->ld = 1;
      planes_d = 18;
    } else {
      return false;
    }
    p->t_h = (p->H + p->th_step - 1) / p->th_step;
    p->t_d = (p->D + p->td_step - 1) / p->td_step;
    p->tiles_total = p->N * p->t_d * p->t_h * p->t_w;
  } else {
    if ((mode == 0 && g->D != 1) || g->H < 16) return false;   // 2-D maps: a tile = 16 lines of np consecutive samples
    p->np = 4;
    p->Pd = 18 * kXW; p->MS = p->Pd; p->LS = kXW;
    p->th_step = 16; p->td_step = 1; p->tn_step = p->np;
    p->mn = 1; p->lh = 1;
    planes_d = 1; planes_n = p->np;
    p->t_h = (g->H + 15) / 16;
    p->t_d = 1;
    p->tiles_total = ((p->N + p->np - 1) / p->np) * p->t_h * p->t_w;
  }
done:
  p->box_d = planes_d; p->box_n = planes_n;
  p->box_h = (p->lh ? 18 : p->np + 2);
  p->ntaps = p->nd * 9;
  {
    const int rows = planes_d * planes_n * (p->lh ? 18 * kXW : p->Pd);
    p->a_tx = (uint32_t)rows * 128u;
  }
  p->a_bytes = (p->a_tx + 1023u) & ~1023u;
  p->tmem_cols = (uint32_t)(2 * p->np * 64);
  if (p->tmem_cols < 32) p->tmem_cols = 32;
  { uint32_t tc = 32; while (tc < p->tmem_cols) tc *= 2; p->tmem_cols = tc; }
  p->idesc = make_idesc_bf16(128, 64, 0, 0);
  {
    int ws = (int)((kSmemBudget - 2u * p->a_bytes - 1024u) / kWTapBytes);
    if (ws > kWStagesMax) ws = kWStagesMax;
    if (ws < 2) return false;
    p->wstages = ws;
  }
  return true;
}

bool halo_fprop_supported(const t2v_conv_geom* g) {
  HaloFpParams p{};
  return halo_fprop_plan(g, &p);
}

static int halo_fprop_launch_mode(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                                  const void* residual, void* y, uint32_t flags, cudaStream_t stream, int mode) {
  HaloFpParams p{};
  if (!halo_fprop_plan(g, &p, mode)) return T2V_ERR_ARG;
  if (mode != 0 && residual != nullptr && !(flags & T2V_EPI_RELU_MASK)) return T2V_ERR_ARG;
  p.bias = bias;
  p.residual = reinterpret_cast<const __nv_bfloat16*>(residual);
  p.out = y;
  p.out_f32 = (flags & T2V_EPI_OUT_F32) ? 1 : 0;
  p.relu = (flags & T2V_EPI_RELU) ? 1 : 0;
  p.relu_mask = (flags & T2V_EPI_RELU_MASK) ? 1 : 0;
  const size_t smem = 2 * (size_t)p.a_bytes + p.wstages * kWTapBytes + 1024 + (8 + 2 * kWStagesMax) * 8 + 16;
  cudaFuncSetAttribute(halo_fprop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  // persistent: one CTA per SM (the weight ring is not multicast over a cluster: measured on B200, clusters of 2 tie
  // with single CTAs because the kernel is not weight-traffic bound, and clusters of 4 lose SMs)
  const int grid = p.tiles_total < 148 ? p.tiles_total : 148;
  p.iters = (p.tiles_total + grid - 1) / grid;

  CUtensorMap tmA, tmW;
  int rc;
  if (mode == 3 || mode == 4)      // merged (n, j) samples of single planes
    rc = make_act_map(&tmA, x, g->N * g->D, 1, g->H, g->W, 64, 64, kXW, p.box_h, p.box_d, p.box_n);
  else
    rc = make_act_map(&tmA, x, g->N, g->D, g->H, g->W, 64, 64, kXW, p.box_h, p.box_d, p.box_n);
  if (rc) return rc;
  rc = make_w_map(&tmW, w, 64, g->kd * 9 * 64, 64, 64);
  if (rc) return rc;

  ProfRec rec;
  if (g_prof_on)     // useful MACs: output voxels x live taps
    prof_begin(stream, &rec, 2, 2.0 * p.N * p.D * g->H * g->W * 64.0 * 64.0 * p.ntaps, g, grid);
  halo_fprop_kernel<<<grid, kFpThreads, smem, stream>>>(tmA, tmW, p);
  if (g_prof_on) prof_end(stream, &rec);
  count_launch();
  return check_last("halo_fprop");
}

int halo_fprop_launch(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                      const void* residual, void* y, uint32_t flags, cudaStream_t stream) {
  return halo_fprop_launch_mode(g, x, w, bias, residual, y, flags, stream, 0);
}

// ---- convolution with stride (2,1,1): Conv3d(64 -> 64, 3, padding 1) of which only the even output planes are
// used (the discriminator stem: txt2vid/models/resnet3d.py:15-16, AvgPool3d((1,2,2), 2) has stride 2 along d
// with kernel 1, so the odd planes of the second conv are never read).  g = geometry of x (D even).
bool halo_sd2_supported(const t2v_conv_geom* g) {
  HaloFpParams p{};
  if (g->Cin != 64 || g->Cout != 64 || g->kd != 3 || g->kh != 3 || g->kw != 3) return false;
  return halo_fprop_plan(g, &p, 1);
}

int halo_fprop_sd2_launch(const t2v_conv_geom* g, const void* x, const void* w, const float* bias, void* y,
                          uint32_t flags, cudaStream_t stream) {
  if (!halo_sd2_supported(g)) return T2V_ERR_ARG;
  return halo_fprop_launch_mode(g, x, w, bias, nullptr, y, flags, stream, 1);
}

// dx (N, D, H, W, 64) = conv_transpose(dy (N, D/2, H, W, 64), w) with the flipped pack: even and odd planes of dx are
// two different sub-convolutions of dy (27 taps per TWO dx planes).  g = geometry of x / dx.
int halo_dgrad_sd2_launch(const t2v_conv_geom* g, const void* dy, const void* wT, const void* relu_ref, void* dx,
                          uint32_t flags, cudaStream_t stream) {
  if (!halo_sd2_supported(g)) return T2V_ERR_ARG;
  t2v_conv_geom gd = *g;
  gd.D = g->D / 2;
  flags = relu_ref ? (flags | T2V_EPI_RELU_MASK) : (flags & ~T2V_EPI_RELU_MASK);
  int rc = halo_fprop_launch_mode(&gd, dy, wT, nullptr, relu_ref, dx, flags, stream, 3);
  if (rc) return rc;
  return halo_fprop_launch_mode(&gd, dy, wT, nullptr, relu_ref, dx, flags, stream, gd.D >= 2 ? 2 : 4);
}

}  // namespace t2v
