// Launch helpers for the bind family, shared by the api_vsa_bind_*.cu translation units (the 10 sizes x 5 modes
// are split over two units to keep the build parallel).
#pragma once
#include "launch.cuh"
#include "vsa_kernels.cuh"

namespace cvb {

template <int LOG2N, int MODE>
int launch_bind_fast(const BindParams& p_in, cudaStream_t st) {
  BindParams p = p_in;
  using Pl = WideFftPlan<LOG2N>;
  const cplx* tw = device_twiddles();
  if (!tw) return kCudaError;
  const long long work = (p.rows + Pl::GROUPS - 1) / Pl::GROUPS;
  // staging measured on B200 (tools/bench_ops.py, DESIGN.md section 4): a and b through TMA from d = 8192 up (a only was
  // measured too: no gain); shorter rows use plain loads, and the staged variant is not instantiated for them
  if constexpr (LOG2N >= 12) {
    if (aligned(p.a, 16) && aligned(p.b, 16))
      return launch_persistent_pdl(bind_v3_kernel<LOG2N, MODE, 2>, "bind_v3_kernel<staged ab>", Pl::THREADS,
                                   bind_v3_smem_bytes<LOG2N, 2>(), work, &p.sched, st, p, tw);
  }
  return launch_persistent_pdl(bind_v3_kernel<LOG2N, MODE, 0>, "bind_v3_kernel<direct>", Pl::THREADS,
                               bind_v3_smem_bytes<LOG2N, 0>(), work, &p.sched, st, p, tw);
}

template <int MODE>
int dispatch_bind(const BindParams& p, int d, cudaStream_t st) {
  const bool fast = is_pow2(d) && d >= 32 && d <= 16384 && aligned(p.a, 8) && aligned(p.b, 8) && aligned(p.out, 8);
  if (fast) return with_int<4, 13>(ilog2(d) - 1, [&](auto L) { return launch_bind_fast<decltype(L)::value, MODE>(p, st); });
  // any other length: the bilinear modes fold a zero-padded power-of-two convolution (bind_pad_kernel) once the
  // O(d^2) direct DFT would cost more (d > 48); the quotient modes need the true length-d spectrum (direct DFT)
  constexpr bool kBilinear = (MODE == kBindMul || MODE == kBindMulConj || MODE == kBindNegMulConj);
  if (d <= kBindSmallMaxD && (!kBilinear || d <= 48)) {
    // short vectors: a tile of pairs per CTA (rows per tile sized so that small batches stay spread over the SMs)
    int rt = 32;
    while (rt > 4 && ((p.rows + rt - 1) / rt < 2LL * sm_count() || bind_small_smem(d, rt) > 48 * 1024)) rt >>= 1;
    return launch_persistent(bind_small_kernel<MODE>, "bind_small_kernel", kBindSmallThreads, bind_small_smem(d, rt),
                             (p.rows + rt - 1) / rt, st, p, d, rt);
  }
  if constexpr (kBilinear) {
    if (d > 48 && d <= 8192) {
      int log2m = 1;
      while ((1 << log2m) < 2 * d) ++log2m;
      return with_int<6, 13>(log2m - 1, [&](auto L) -> int {
        using Pl = WideFftPlan<decltype(L)::value>;
        const cplx* tw = device_twiddles();
        if (!tw) return kCudaError;
        return launch_persistent(bind_pad_kernel<decltype(L)::value, MODE>, "bind_pad_kernel", Pl::THREADS,
                                 bind_pad_smem_bytes<decltype(L)::value>(), (p.rows + Pl::GROUPS - 1) / Pl::GROUPS, st, p, d, tw);
      });
    }
  }
  const size_t smem = sizeof(cplx) * d + sizeof(float) * (2 * d + 2) + sizeof(cplx) * (d / 2 + 1);
  CVB_REQUIRE(smem <= kGenericSmemLimit, kUnsupported, "vsa bind: d=%d too large for the direct-DFT path", d);
  return launch_persistent(bind_generic_kernel<MODE>, "bind_generic_kernel", 256, smem, p.rows, st, p, d);
}

}  // namespace cvb
