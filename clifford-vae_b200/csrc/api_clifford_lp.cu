// C ABI entry points for the Clifford-torus kernels (include/clifford_b200.h).
#include "clifford_launch.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

namespace {

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
  return launch_persistent_pdl(clifford_log_prob_kernel<LOG2N, ROWK, FWD_ONLY, VM>, "clifford_log_prob_kernel", Pl::THREADS,
                               smem, (p.rows + Pl::GROUPS - 1) / Pl::GROUPS, nullptr, st, p, tw);
}

template <bool ROWK, bool VM = false>
int dispatch_lp(const CliffordLogProbParams& p, cudaStream_t st) {
  const int n = 2 * p.d;
  return dispatch_clifford(
      "clifford log_prob", p, n, p.value, [&](auto L) { return launch_lp_fast<decltype(L)::value, ROWK, false, VM>(p, st); },
      clifford_lp_small_kernel<ROWK, VM>, [&](int r) { return clifford_lp_small_smem(p.d, r); },
      clifford_log_prob_generic_kernel<ROWK, VM>, sizeof(cplx) * n + sizeof(float) * (n + 32), st);
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
