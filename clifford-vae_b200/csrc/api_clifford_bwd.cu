// C ABI entry points for the Clifford-torus kernels (include/clifford_b200.h).
#include "clifford_launch.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

namespace {

template <int LOG2N, bool ROWK, bool FAST = false, bool VM = false>
int launch_bwd_fast(const CliffordBwdParams& p, cudaStream_t st) {
  if constexpr (ROWK && !FAST && !VM) {
    if (p.tp_signed && p.staged) return launch_bwd_fast<LOG2N, ROWK, true>(p, st);   // the training path
  }
  using Pl = FftPlan<LOG2N>;
  const cplx* tw = device_twiddles();
  const float2* icdf = device_icdf_table();
  if (!tw || !icdf) return kCudaError;
  CliffordBwdParams q = p;
  // dynamic rows only with one row per CTA
  return launch_persistent_pdl(clifford_bwd_kernel<LOG2N, ROWK, FAST, VM>, "clifford_bwd_kernel", Pl::THREADS,
                               clifford_bwd_smem_bytes<LOG2N, ROWK, FAST, VM>(), (p.rows + Pl::GROUPS - 1) / Pl::GROUPS,
                               Pl::GROUPS == 1 ? &q.sched : nullptr, st, q, tw, icdf);
}

template <bool ROWK, bool VM = false>
int dispatch_bwd(const CliffordBwdParams& p_in, cudaStream_t st) {
  CliffordBwdParams p = p_in;
  p.staged = aligned(p.loc, 16) && (!p.tp_signed || aligned(p.tp_signed, 16)) && (!p.tprime || aligned(p.tprime, 16)) &&
             (!p.gnoise || aligned(p.gnoise, 16));
  const int n = 2 * p.d;
  return dispatch_clifford(
      "clifford backward", p, n, p.grad_z, [&](auto L) { return launch_bwd_fast<decltype(L)::value, ROWK, false, VM>(p, st); },
      clifford_bwd_small_kernel<ROWK, VM>, [&](int r) { return clifford_bwd_small_smem(p.d, r); },
      clifford_bwd_generic_kernel<ROWK, VM>, sizeof(cplx) * n + sizeof(float) * (n + 32), st);
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
  // every tier reads tp_signed whenever it is given, injected draws or not
  CVB_REQUIRE(!tp_signed || !ps_saved_draws_need_fft(d, kappa_el_stride == 0) || aligned(grad_z, 8), kUnsupported,
              "cvb_clifford_ps_rsample_backward: grad_z must be 8-byte aligned with tp_signed at d=%d and one concentration "
              "per row (the forward saved those draws in the FFT engine's format)", d);
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
