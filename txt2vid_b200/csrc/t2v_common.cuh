// Shared device helpers for the txt2vid B200 kernels (sm_100a only).
// Raw PTX wrappers for mbarrier / TMA / tcgen05 / TMEM; no CUTLASS dependency.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/t2v.h"

#define T2V_DEVINL __device__ __forceinline__

namespace t2v {

// ---------------------------------------------------------------- launch-count bookkeeping
// Every C-ABI entry point bumps this once per kernel it launches; bench.py reads it
// through t2v_launch_count() to report "gpu_launches".
extern unsigned long long g_launch_count;
inline void count_launch(int n = 1) { g_launch_count += (unsigned long long)n; }

inline int check_last(const char* /*what*/) {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? T2V_OK : T2V_ERR_LAUNCH;
}

// ---------------------------------------------------------------- small math
T2V_DEVINL float bf2f(__nv_bfloat16 v) { return __bfloat162float(v); }
T2V_DEVINL __nv_bfloat16 f2bf(float v) { return __float2bfloat16_rn(v); }
T2V_DEVINL float bf2f(float v) { return v; }   // fp32-storage instantiations of the typed kernels

T2V_DEVINL uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
T2V_DEVINL float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

T2V_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------- shared-memory address
T2V_DEVINL uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
T2V_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
T2V_DEVINL void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
T2V_DEVINL void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
T2V_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
T2V_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
T2V_DEVINL uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// Bounded spin: a pipeline bug traps (-> CUDA error at the next sync) instead of hanging the GPU.
#ifndef T2V_HANG_GUARD_SPINS
#define T2V_HANG_GUARD_SPINS (1u << 26)
#endif
T2V_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > T2V_HANG_GUARD_SPINS) __trap();
  }
}

// ---------------------------------------------------------------- TMA (cp.async.bulk.tensor)
T2V_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
T2V_DEVINL void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
T2V_DEVINL void tma_load_5d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
      "r"(c4)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
T2V_DEVINL void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
T2V_DEVINL void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
T2V_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
T2V_DEVINL void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
T2V_DEVINL void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate, issued by ONE thread.
T2V_DEVINL void umma_bf16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread retire.
T2V_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread (thread i = lane i of the
// warp's TMEM quadrant).
T2V_DEVINL void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
T2V_DEVINL void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr)
      : "memory");
}
T2V_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ConvLSTM step fused into the gate GEMM's epilogue (igemm_sm100.cu): the extra operands of t2v_conv_lstm_step
struct LstmEpi {
  const float* c_prev;   // fp32 [P][Hd] or null (first step)
  float* c_out;          // fp32 [P][Hd]
  float* gates;          // fp32 [P][4 Hd], [i | f | g | o], pre-activation incl. bias (saved for the backward pass)
  void* h_out;           // bf16 [P][Hd]: the next step's GEMM operand
  void* h_merged;        // bf16 [(n * steps + t) * plane + pos_in_plane][Hd]: the merged (b, t) frame map
  int t, steps;
};

// Window of a convolution whose input extents differ from its output extents (t2v_conv_fprop_win / _wgrad_win): the
// kernels only see the input through its tensor map (coordinates + out-of-bounds zero fill), so the tile grid walks
// the OUTPUT positions of the geometry while the input map takes these extents, and the live tap range per axis is
// given explicitly (tap t reads input coordinate o + t - k/2).
struct ConvWindow {
  int iD, iH, iW;
  int lo_d, hi_d, lo_h, hi_h, lo_w, hi_w;
};

// UMMA shared-memory matrix descriptor (sm_100 format, version 1).
//   start address >>4 in [0,14), LBO>>4 in [16,30), SBO>>4 in [32,46), version=1 in [46,48),
//   layout type in [61,64): 0 none, 2 = 128B swizzle, 4 = 64B, 6 = 32B.
T2V_DEVINL uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                   uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(layout_type & 7u) << 61;
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B and fp32 accumulate.
//   c_format F32 (1) at [4,6); a/b_format BF16 (1) at [7,10)/[10,13); a_major [15], b_major [16]
//   (0 = K-major, 1 = MN-major); N>>3 at [17,23); M>>4 at [24,29).
// 16-byte vector reduction: four fp32 adds in ONE memory operation (the scalar form costs ~1.3 cycles per lane per
// element at the L2: the split-K epilogues of the weight-gradient kernels were bound by it)
T2V_DEVINL void red_add_v4(float* dst, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// One 32-byte store (SASS STG.E.256): a conv epilogue thread owns 16 bf16 output channels of its row; two 16-byte
// stores half-fill each 32-byte sector twice (ncu: 2x the store sectors of the output tensor)
T2V_DEVINL void st_global_v8(void* dst, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(a.x), "r"(a.y), "r"(a.z),
               "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}

__host__ __device__ inline uint32_t make_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn_major,
                                                    uint32_t b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;
  d |= 1u << 7;
  d |= 1u << 10;
  d |= (a_mn_major & 1u) << 15;
  d |= (b_mn_major & 1u) << 16;
  d |= ((N >> 3) & 0x3Fu) << 17;
  d |= ((M >> 4) & 0x1Fu) << 24;
  return d;
}

// One elected lane of a fully active warp (same lane every time for the same mask).  Code that feeds
// tcgen05 instructions should compute its operands in WARP-UNIFORM control flow and only predicate the
// instruction itself on this: ptxas then keeps descriptors in uniform registers instead of running an
// ELECT / R2UR.BROADCAST waterfall loop (~18 instructions) in front of every UTCHMMA.
T2V_DEVINL uint32_t elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(pred));
  return pred;
}
// descriptor halves: lo = start>>4 | (LBO>>4) << 16, hi = SBO>>4 | version 1 << 14 | layout << 29
T2V_DEVINL uint32_t desc_lo(uint32_t saddr16, uint32_t lbo_bytes) {
  return (saddr16 & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
T2V_DEVINL uint32_t desc_hi(uint32_t sbo_bytes, uint32_t layout_type) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((layout_type & 7u) << 29);
}
T2V_DEVINL void umma_bf16_ss2(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

}  // namespace t2v
