// Common device helpers for the sm_100a kernels of monoflex_b200: mbarrier / cp.async / TMA / tcgen05 PTX.
// Everything here is hand-written inline PTX (no CUTLASS); compile with -gencode arch=compute_100a,code=sm_100a.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda.h>
#include <stdint.h>

#define MF_DEVINL __device__ __forceinline__

namespace mf {

// ------------------------------------------------------------------------------------------------ error state
void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

// <<<>>> replacement through cudaLaunchKernelEx
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = nullptr;
  cfg.numAttrs = 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

MF_DEVINL uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ------------------------------------------------------------------------------------------------ mbarrier
MF_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
MF_DEVINL void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
MF_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
MF_DEVINL void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
MF_DEVINL uint32_t mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(addr), "r"(parity)
      : "memory");
  return ok;
}
MF_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  while (!mbar_try_wait(addr, parity)) {
  }
}

// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA reads)
MF_DEVINL void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ explicit shared-space ld/st
// (pointers carved out of the dynamic smem block through integer alignment lose their address space: the compiler then
// emits generic LD.E / ST.E with 64-bit address arithmetic; these keep the hot loops on LDS / STS with 32-bit addresses)
MF_DEVINL uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
MF_DEVINL float4 lds128f(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
MF_DEVINL void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
MF_DEVINL void sts128f(uint32_t addr, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
MF_DEVINL void sts32f(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }

// ------------------------------------------------------------------------------------------------ packed fp32 math (sm_100: FFMA2 / FMUL2)
MF_DEVINL unsigned long long f2_pack(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
MF_DEVINL float2 f2_unpack(unsigned long long v) {
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
  return r;
}
MF_DEVINL unsigned long long f2_mul(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
MF_DEVINL unsigned long long f2_fma(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// ------------------------------------------------------------------------------------------------ cp.async
// 16-byte global->shared copy; src_bytes == 0 zero-fills the destination (used for conv padding / K tail).
MF_DEVINL void cp_async16(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
// same, allocating in L1 (.ca): the gather of small-Cin layers re-reads every input pixel kh*kw times from the same CTA
MF_DEVINL void cp_async16_ca(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
MF_DEVINL void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
MF_DEVINL void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------------ TMA
MF_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
MF_DEVINL void tma_load_2d(uint32_t dst_smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          dst_smem),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// One lane of a fully converged warp. The MMA / TMA issuing warps walk their loops with ALL lanes (warp-uniform control flow
// keeps descriptors and addresses in uniform registers) and issue under `if (elect_one())`: under `if (lane == 0)` ptxas
// wraps every UTCHMMA / UTMALDG in an ELECT + R2UR + BRA.U.ANY "waterfall" loop (~8 dependent instructions per MMA, which
// made the issuing thread the bottleneck of every tile narrower than ~256 columns).
MF_DEVINL bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "elect.sync _|P1, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P1;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------------------------------------ named barriers, TMA store, im2col-mode TMA load
MF_DEVINL void tma_load_im2col_4d(uint32_t dst_smem, const CUtensorMap* m, uint64_t* bar, int c, int w, int h, int n,
                                  uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2], {%7, %8};" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}

MF_DEVINL void bar_sync_named(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// tiled 4D load (coordinates may lie outside the tensor: those elements are zero-filled and still counted in the tx bytes)
MF_DEVINL void tma_load_4d(uint32_t dst_smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          dst_smem),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
MF_DEVINL void tma_store_2d(const CUtensorMap* m, uint32_t src_smem, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}
MF_DEVINL void tma_store_4d(const CUtensorMap* m, uint32_t src_smem, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src_smem), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
MF_DEVINL void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
MF_DEVINL void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
MF_DEVINL void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }


// ------------------------------------------------------------------------------------------------ tcgen05
MF_DEVINL void tmem_alloc(uint32_t* dst_in_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_in_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
MF_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
MF_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
MF_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], kind::f16 (fp16/bf16 operands, fp32 accumulate), one CTA.
MF_DEVINL void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
MF_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i <-> TMEM lane base+i)
MF_DEVINL void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
MF_DEVINL void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
MF_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile in shared memory, 128-byte swizzle, rows of 64 fp16 (=128 B), 8-row atoms of 1024 B.
// Descriptor fields (sm_100 "SmemDescriptor"): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48)
// | layout_type=2 (SWIZZLE_128B) [61,64). LBO is ignored for swizzled K-major; SBO = 1024 B between 8-row atoms.
MF_DEVINL uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// generic K-major descriptor: layout_type 0 = no swizzle (LBO = byte distance between the two 16-byte K chunks of an MMA,
// SBO = distance between 8-row groups), 6 / 4 / 2 = 32B / 64B / 128B swizzle (LBO ignored, SBO = 8 * row bytes)
MF_DEVINL uint64_t umma_desc_kmajor(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  return static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu) | (static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         (static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) |
         (static_cast<uint64_t>(layout_type) << 61);
}
// kind::f16 instruction descriptor: D=f32 (bit 4), A=B=f16 (0), both K-major, N>>3 at [17,23), M>>4 at [24,29).
MF_DEVINL constexpr uint32_t umma_idesc_f16(int m, int n) {
  return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// byte offset of 16-byte chunk `c` (0..7) of row `r` inside a [rows x 64 fp16] SWIZZLE_128B tile
MF_DEVINL uint32_t sw128_off(int r, int c) { return (r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4); }

}  // namespace mf
