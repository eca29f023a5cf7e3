// C ABI entry points for the Clifford-torus kernels (include/clifford_b200.h).
#include "launch.cuh"
#include <cstdlib>
#include "clifford_kernels.cuh"
#include "clifford_small.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

namespace {

constexpr size_t kGenericSmemLimit = 200 * 1024;

template <int LOG2N, bool ROWK, bool FWD_ONLY = false, bool VM = false>
int launch_lp_fast(const CliffordLogProbParams& p, cudaStream_t st) {
  if constexpr (ROWK && !FWD_ONLY && !VM) {
    if (!p.dlp_dF && !p.dlp_dloc && !p.dlp_dkappa) return launch_lp_fast<LOG2N, ROWK, true>(p, st);   // evaluation
  }
  using Pl = FftPlan<LOG2N>;
  const cplx* tw = device_twiddles();
  if (!tw) return kCudaError;
  const size_t smem = sizeof(cplx) * Pl::XCH * Pl::GROUPS + sizeof(float) * 32 * Pl::GROUPS + sizeof(float2) * kLpConstCache * Pl::GROUPS +
                      sizeof(float) * Pl::N * Pl::GROUPS;
  auto kern = clifford_log_prob_kernel<LOG2N, ROWK, FWD_ONLY, VM>;
  int grid = 0;
  const long long work = (p.rows + Pl::GROUPS - 1) / Pl::GROUPS;
  if (int rc = persistent_grid(kern, Pl::THREADS, smem, work, &grid)) return rc;
  launch_pdl(kern, grid, Pl::THREADS, smem, st, p, tw);
  return check_launch("clifford_log_prob_kernel");
}

template <bool ROWK, bool VM = false>
int dispatch_lp(const CliffordLogProbParams& p, cudaStream_t st) {
  const bool fast = is_pow2(p.d) && p.d >= 16 && p.d <= 8192 && aligned(p.value, 8);
  if (fast) {
    switch (ilog2(p.d)) {
#define CVB_CASE(L) case L: return launch_lp_fast<L, ROWK, false, VM>(p, st);
      CVB_CASE(4) CVB_CASE(5) CVB_CASE(6) CVB_CASE(7) CVB_CASE(8) CVB_CASE(9) CVB_CASE(10) CVB_CASE(11) CVB_CASE(12)
      CVB_CASE(13)
#undef CVB_CASE
    }
  }
  static const bool no_small = getenv("CVB_NO_SMALL_ROWS") != nullptr;
  if (2 * p.d <= kSmallMaxN && !no_small) {
    const int rt = small_rows_per_tile(p.rows, sm_count(), [&](int r) { return clifford_lp_small_smem(p.d, r); });
    const size_t smem_s = clifford_lp_small_smem(p.d, rt);
    auto kern_s = clifford_lp_small_kernel<ROWK, VM>;
    int grid_s = 0;
    if (int rc = persistent_grid(kern_s, kSmallThreads, smem_s, (p.rows + rt - 1) / rt, &grid_s)) return rc;
    kern_s<<<grid_s, kSmallThreads, smem_s, st>>>(p, rt);
    return check_launch("clifford_log_prob_small_kernel");
  }
  const int n = 2 * p.d;
  const size_t smem = sizeof(cplx) * n + sizeof(float) * (n + 32);
  CVB_REQUIRE(smem <= kGenericSmemLimit, kUnsupported, "clifford log_prob: d=%d too large for the direct-DFT path", p.d);
  auto kern = clifford_log_prob_generic_kernel<ROWK, VM>;
  int grid = 0;
  if (int rc = persistent_grid(kern, kGenericThreads, smem, p.rows, &grid)) return rc;
  kern<<<grid, kGenericThreads, smem, st>>>(p);
  return check_launch("clifford_log_prob_generic_kernel");
}

}  // namespace

extern "C" {

int cvb_clifford_ps_log_prob(const float* value, const float* loc, const float* kappa, long long kappa_row_stride,
                             int kappa_el_stride, long long loc_rows, float* log_prob, float* dlp_dloc,
                             float* dlp_dkappa, float* dlp_dF, long long rows, int d, void* stream) {
  CVB_REQUIRE(value && loc && kappa && log_prob, kBadArgument, "cvb_clifford_ps_log_prob: null pointer");
  CVB_REQUIRE(rows > 0 && d >= 1 && loc_rows > 0, kBadArgument, "cvb_clifford_ps_log_prob: bad sizes");
  CVB_REQUIRE((dlp_dloc == nullptr) == (dlp_dkappa == nullptr), kBadArgument, "cvb_clifford_ps_log_prob: give both derivative outputs or neither");
  CliffordLogProbParams p{};
  p.value = value; p.loc = loc; p.kappa = kappa; p.kappa_row_stride = kappa_row_stride;
  p.kappa_el_stride = kappa_el_stride; p.loc_rows = (int)loc_rows; p.log_prob = log_prob; p.dlp_dloc = dlp_dloc;
  p.dlp_dkappa = dlp_dkappa; p.dlp_dF = dlp_dF; p.rows = rows; p.d = d;
  cudaStream_t st = (cudaStream_t)stream;
  return kappa_el_stride == 0 ? dispatch_lp<true>(p, st) : dispatch_lp<false>(p, st);
}

// CliffordTorusDistribution.log_prob: sum over circles k >= 1 of kappa cos(angle(F_k) - loc_k) - ln(2 pi I0(kappa))
int cvb_clifford_vm_log_prob(const float* value, const float* loc, const float* kappa, long long kappa_row_stride,
                             int kappa_el_stride, long long loc_rows, float* log_prob, float* dlp_dloc,
                             float* dlp_dkappa, float* dlp_dF, long long rows, int d, void* stream) {
  CVB_REQUIRE(value && loc && kappa && log_prob, kBadArgument, "cvb_clifford_vm_log_prob: null pointer");
  CVB_REQUIRE(rows > 0 && d >= 1 && loc_rows > 0, kBadArgument, "cvb_clifford_vm_log_prob: bad sizes");
  CVB_REQUIRE((dlp_dloc == nullptr) == (dlp_dkappa == nullptr), kBadArgument, "cvb_clifford_vm_log_prob: give both derivative outputs or neither");
  CliffordLogProbParams p{};
  p.value = value; p.loc = loc; p.kappa = kappa; p.kappa_row_stride = kappa_row_stride;
  p.kappa_el_stride = kappa_el_stride; p.loc_rows = (int)loc_rows; p.log_prob = log_prob; p.dlp_dloc = dlp_dloc;
  p.dlp_dkappa = dlp_dkappa; p.dlp_dF = dlp_dF; p.rows = rows; p.d = d;
  cudaStream_t st = (cudaStream_t)stream;
  return kappa_el_stride == 0 ? dispatch_lp<true, true>(p, st) : dispatch_lp<false, true>(p, st);
}

}  // extern "C"
