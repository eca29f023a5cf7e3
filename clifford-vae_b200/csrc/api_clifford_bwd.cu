// C ABI entry points for the Clifford-torus kernels (include/clifford_b200.h).
#include <cstdlib>
#include "launch.cuh"
#include "clifford_kernels.cuh"
#include "clifford_small.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

namespace {

constexpr size_t kGenericSmemLimit = 200 * 1024;

template <int LOG2N, bool ROWK, bool FAST = false, bool VM = false>
int launch_bwd_fast(const CliffordBwdParams& p, cudaStream_t st) {
  if constexpr (ROWK && !FAST && !VM) {
    if (p.tp_signed && p.staged) return launch_bwd_fast<LOG2N, ROWK, true>(p, st);   // the training path
  }
  using Pl = FftPlan<LOG2N>;
  const cplx* tw = device_twiddles();
  const float2* icdf = device_icdf_table();
  if (!tw || !icdf) return kCudaError;
  const size_t smem = clifford_bwd_smem_bytes<LOG2N, ROWK, FAST, VM>();
  auto kern = clifford_bwd_kernel<LOG2N, ROWK, FAST, VM>;
  int grid = 0;
  const long long work = (p.rows + Pl::GROUPS - 1) / Pl::GROUPS;
  if (int rc = persistent_grid(kern, Pl::THREADS, smem, work, &grid)) return rc;
  CliffordBwdParams q = p;
  static const bool static_sched = getenv("CVB_STATIC_SCHEDULE") != nullptr;
  q.sched = (Pl::GROUPS == 1 && !static_sched && work > grid) ? next_sched_slot() : nullptr;   // dynamic rows when CTAs loop
  launch_pdl(kern, grid, Pl::THREADS, smem, st, q, tw, icdf);
  return check_launch("clifford_bwd_kernel");
}

template <bool ROWK, bool VM = false>
int dispatch_bwd(const CliffordBwdParams& p_in, cudaStream_t st) {
  CliffordBwdParams p = p_in;
  p.staged = aligned(p.loc, 16) && (!p.tp_signed || aligned(p.tp_signed, 16)) && (!p.tprime || aligned(p.tprime, 16)) &&
             (!p.gnoise || aligned(p.gnoise, 16)) && getenv("CVB_NO_TMA") == nullptr;
  const bool fast = is_pow2(p.d) && p.d >= 16 && p.d <= 8192 && aligned(p.grad_z, 8);
  if (fast) {
    switch (ilog2(p.d)) {
#define CVB_CASE(L) case L: return launch_bwd_fast<L, ROWK, false, VM>(p, st);
      CVB_CASE(4) CVB_CASE(5) CVB_CASE(6) CVB_CASE(7) CVB_CASE(8) CVB_CASE(9) CVB_CASE(10) CVB_CASE(11) CVB_CASE(12)
      CVB_CASE(13)
#undef CVB_CASE
    }
  }
  static const bool no_small = getenv("CVB_NO_SMALL_ROWS") != nullptr;
  if (2 * p.d <= kSmallMaxN && !no_small) {
    const int rt = small_rows_per_tile(p.rows, sm_count(), [&](int r) { return clifford_bwd_small_smem(p.d, r); });
    const size_t smem_s = clifford_bwd_small_smem(p.d, rt);
    auto kern_s = clifford_bwd_small_kernel<ROWK, VM>;
    int grid_s = 0;
    if (int rc = persistent_grid(kern_s, kSmallThreads, smem_s, (p.rows + rt - 1) / rt, &grid_s)) return rc;
    kern_s<<<grid_s, kSmallThreads, smem_s, st>>>(p, rt);
    return check_launch("clifford_bwd_small_kernel");
  }
  const int n = 2 * p.d;
  const size_t smem = sizeof(cplx) * n + sizeof(float) * (n + 32);
  CVB_REQUIRE(smem <= kGenericSmemLimit, kUnsupported, "clifford backward: d=%d too large for the direct-DFT path", p.d);
  auto kern = clifford_bwd_generic_kernel<ROWK, VM>;
  int grid = 0;
  if (int rc = persistent_grid(kern, kGenericThreads, smem, p.rows, &grid)) return rc;
  kern<<<grid, kGenericThreads, smem, st>>>(p);
  return check_launch("clifford_bwd_generic_kernel");
}

}  // namespace

extern "C" {

static int clifford_ps_rsample_backward_impl(const float* grad_z, const float* loc, const float* kappa,
                                             long long kappa_row_stride, int kappa_el_stride, long long loc_rows,
                                             const float* tprime, const float* gnoise, const float* tp_signed, float* dloc,
                                             float* dkappa, long long rows, int d, KappaHead head, void* stream) {
  CVB_REQUIRE(grad_z && loc && kappa && dloc && dkappa, kBadArgument, "cvb_clifford_ps_rsample_backward: null pointer");
  CVB_REQUIRE(rows > 0 && d >= 1 && loc_rows > 0, kBadArgument, "cvb_clifford_ps_rsample_backward: bad sizes");
  CVB_REQUIRE(tp_signed || (tprime && gnoise), kBadArgument, "cvb_clifford_ps_rsample_backward: need tp_signed or (tprime, gnoise)");
  CliffordBwdParams p{};
  p.grad_z = grad_z; p.loc = loc; p.kappa = kappa; p.kappa_row_stride = kappa_row_stride;
  p.kappa_el_stride = kappa_el_stride; p.loc_rows = (int)loc_rows; p.tprime = tprime; p.gnoise = gnoise;
  p.tp_signed = tp_signed; p.dloc = dloc; p.dkappa = dkappa; p.rows = rows; p.d = d; p.head = head;
  cudaStream_t st = (cudaStream_t)stream;
  return kappa_el_stride == 0 ? dispatch_bwd<true>(p, st) : dispatch_bwd<false>(p, st);
}

int cvb_clifford_ps_rsample_backward(const float* grad_z, const float* loc, const float* kappa,
                                     long long kappa_row_stride, int kappa_el_stride, long long loc_rows,
                                     const float* tprime, const float* gnoise, const float* tp_signed, float* dloc,
                                     float* dkappa, long long rows, int d, void* stream) {
  return clifford_ps_rsample_backward_impl(grad_z, loc, kappa, kappa_row_stride, kappa_el_stride, loc_rows, tprime, gnoise,
                                           tp_signed, dloc, dkappa, rows, d, KappaHead{0, 0.f, 0.f}, stream);
}

// backward of cvb_clifford_ps_rsample_head: draw_scale (rows) = d L / d raw_scale (softplus and clamp chain applied)
int cvb_clifford_ps_rsample_backward_head(const float* grad_z, const float* loc, const float* raw_scale, long long loc_rows,
                                          float floor, float kmax, const float* tprime, const float* gnoise,
                                          const float* tp_signed, float* dloc, float* draw_scale, long long rows, int d,
                                          void* stream) {
  return clifford_ps_rsample_backward_impl(grad_z, loc, raw_scale, 1, 0, loc_rows, tprime, gnoise, tp_signed, dloc,
                                           draw_scale, rows, d, KappaHead{1, floor, kmax}, stream);
}

int cvb_ps_entropy_kl(const float* kappa, long long kappa_row_stride, int kappa_el_stride, long long rows, int d,
                      double half_dm1, int torus, double prior_entropy, float* entropy, float* kl, float* dentropy,
                      void* stream) {
  CVB_REQUIRE(kappa && rows > 0 && d >= 1, kBadArgument, "cvb_ps_entropy_kl: bad arguments");
  EntropyParams p{};
  p.kappa = kappa; p.kappa_row_stride = kappa_row_stride; p.kappa_el_stride = kappa_el_stride; p.entropy = entropy;
  p.kl = kl; p.dentropy = dentropy; p.rows = rows; p.d = d; p.half_dm1 = half_dm1; p.skip_first = torus ? 1 : 0;
  p.prior_entropy = prior_entropy;
  long long warps = rows;
  int blocks = (int)((warps * 32 + 255) / 256);
  const int cap = sm_count() * 8;
  if (blocks > cap) blocks = cap;
  ps_entropy_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(p);
  return check_launch("ps_entropy_kernel");
}

// Backward of cvb_clifford_vm_rsample_kl: phi (rows, d) = the offsets that launch saved
int cvb_clifford_vm_rsample_backward(const float* grad_z, const float* loc, const float* kappa, long long kappa_row_stride,
                                     int kappa_el_stride, long long loc_rows, const float* phi, float* dloc, float* dkappa,
                                     long long rows, int d, void* stream) {
  CVB_REQUIRE(grad_z && loc && kappa && phi && dloc && dkappa, kBadArgument, "cvb_clifford_vm_rsample_backward: null pointer");
  CVB_REQUIRE(rows > 0 && d >= 1 && loc_rows > 0, kBadArgument, "cvb_clifford_vm_rsample_backward: bad sizes");
  CliffordBwdParams p{};
  p.grad_z = grad_z; p.loc = loc; p.kappa = kappa; p.kappa_row_stride = kappa_row_stride;
  p.kappa_el_stride = kappa_el_stride; p.loc_rows = (int)loc_rows; p.tp_signed = phi; p.dloc = dloc; p.dkappa = dkappa;
  p.rows = rows; p.d = d;
  cudaStream_t st = (cudaStream_t)stream;
  return kappa_el_stride == 0 ? dispatch_bwd<true, true>(p, st) : dispatch_bwd<false, true>(p, st);
}

// CliffordTorusDistribution.entropy (dists/clifford.py:21-31, :277-278): sum over circles k >= 1 of the von Mises entropy
int cvb_clifford_vm_entropy(const float* kappa, long long kappa_row_stride, int kappa_el_stride, long long rows, int d,
                            float* entropy, float* dentropy, void* stream) {
  CVB_REQUIRE(kappa && rows > 0 && d >= 1 && (entropy || dentropy), kBadArgument, "cvb_clifford_vm_entropy: bad arguments");
  EntropyParams p{};
  p.kappa = kappa; p.kappa_row_stride = kappa_row_stride; p.kappa_el_stride = kappa_el_stride; p.entropy = entropy;
  p.dentropy = dentropy; p.rows = rows; p.d = d;
  int blocks = (int)((rows * 32 + 255) / 256);
  const int cap = sm_count() * 8;
  if (blocks > cap) blocks = cap;
  vm_entropy_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(p);
  return check_launch("vm_entropy_kernel");
}

}  // extern "C"
