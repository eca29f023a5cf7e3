// C ABI entry points for the Clifford-torus kernels (include/clifford_b200.h).
#include "clifford_launch.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

namespace {

template <int LOG2N, int MODE, bool ROWK, bool LEAN = false>
int launch_fwd_fast(const CliffordFwdParams& p, cudaStream_t st) {
  if constexpr (MODE == kPsRng && ROWK && !LEAN) {
    // plain forward sampling: the specialised variant (no optional outputs, staged inputs)
    if (!p.tp_signed && !p.log_prob && p.staged && !p.head.on) return launch_fwd_fast<LOG2N, MODE, ROWK, true>(p, st);
  }
  using Pl = FftPlan<LOG2N>;
  const cplx* tw = device_twiddles();
  const float2* icdf = device_icdf_table();
  if (!tw || !icdf) return kCudaError;
  CliffordFwdParams q = p;
  return launch_persistent_pdl(clifford_fwd_kernel<LOG2N, MODE, ROWK, false, LEAN>, "clifford_fwd_kernel", Pl::THREADS,
                               clifford_fwd_smem_bytes<LOG2N, MODE>(), (p.rows + Pl::GROUPS - 1) / Pl::GROUPS, &q.sched,
                               st, q, tw, icdf);
}

template <int LOG2N, int MODE>
int launch_fwd_bind(const CliffordFwdParams& p, cudaStream_t st) {
  using Pl = FftPlan<LOG2N>;
  static_assert(clifford_fwd_smem_bytes<LOG2N, MODE, true>() <= 227 * 1024, "bind kernel exceeds a CTA's shared memory");
  const cplx* tw = device_twiddles();
  const float2* icdf = device_icdf_table();
  if (!tw || !icdf) return kCudaError;
  CliffordFwdParams q = p;
  return launch_persistent_pdl(clifford_fwd_kernel<LOG2N, MODE, true, true>, "clifford_fwd_kernel<bind>", Pl::THREADS,
                               clifford_fwd_smem_bytes<LOG2N, MODE, true>(), (p.rows + Pl::GROUPS - 1) / Pl::GROUPS,
                               &q.sched, st, q, tw, icdf);
}

template <int MODE>
int dispatch_fwd_bind(const CliffordFwdParams& p_in, cudaStream_t st) {
  CliffordFwdParams p = p_in;
  p.staged = aligned(p.loc, 16) && (!p.tprime || aligned(p.tprime, 16)) && (!p.gnoise || aligned(p.gnoise, 16));
  return with_int<4, 13>(ilog2(p.d), [&](auto L) { return launch_fwd_bind<decltype(L)::value, MODE>(p, st); });
}

template <int MODE, bool ROWK>
int dispatch_fwd(const CliffordFwdParams& p_in, cudaStream_t st) {
  CliffordFwdParams p = p_in;
  p.staged = (!p.loc || aligned(p.loc, 16)) && (!p.tprime || aligned(p.tprime, 16)) && (!p.gnoise || aligned(p.gnoise, 16)) &&
             (!p.phases || aligned(p.phases, 16));
  const int nph = (p.n - 1) / 2;
  return dispatch_clifford(
      "clifford rsample", p, p.n, p.z, [&](auto L) { return launch_fwd_fast<decltype(L)::value, MODE, ROWK>(p, st); },
      clifford_fwd_small_kernel<MODE, ROWK>, [&](int r) { return clifford_fwd_small_smem(p.n, r); },
      clifford_fwd_generic_kernel<MODE, ROWK>, sizeof(cplx) * ((size_t)p.n + nph + 1), st);
}

}  // namespace

extern "C" {

static int clifford_ps_rsample_impl(const float* loc, const float* kappa, long long kappa_row_stride, int kappa_el_stride,
                                    long long loc_rows, const float* tprime, const float* gnoise, unsigned long long seed,
                                    unsigned long long offset, float* z, float* tp_signed, float* entropy, float* kl,
                                    float* dentropy, long long rows, int d, KappaHead head, void* stream) {
  CVB_REQUIRE(loc && kappa && z, kBadArgument, "cvb_clifford_ps_rsample: null pointer");
  CVB_REQUIRE(rows > 0 && d >= 1 && loc_rows > 0, kBadArgument, "cvb_clifford_ps_rsample: rows=%lld d=%d loc_rows=%lld", rows, d, loc_rows);
  CVB_REQUIRE((tprime == nullptr) == (gnoise == nullptr), kBadArgument, "cvb_clifford_ps_rsample: give both tprime and gnoise or neither");
  CVB_REQUIRE(kappa_el_stride == 0 || (!entropy && !kl && !dentropy), kBadArgument,
              "cvb_clifford_ps_rsample: fused entropy/kl needs one concentration per row; use cvb_ps_entropy_kl");
  CVB_REQUIRE(tprime || !tp_signed || !ps_saved_draws_need_fft(d, kappa_el_stride == 0) || aligned(z, 8), kUnsupported,
              "cvb_clifford_ps_rsample: z must be 8-byte aligned to save tp_signed in RNG mode at d=%d with one "
              "concentration per row (the backward reads those draws in the FFT engine's format)", d);
  CliffordFwdParams p{};
  p.loc = loc; p.kappa = kappa; p.kappa_row_stride = kappa_row_stride; p.kappa_el_stride = kappa_el_stride;
  p.loc_rows = (int)loc_rows; p.tprime = tprime; p.gnoise = gnoise; p.z = z; p.tp_signed = tp_signed;
  p.entropy = entropy; p.kl = kl; p.dentropy = dentropy; p.rows = rows; p.d = d; p.n = 2 * d;
  p.key = make_key(seed, offset, 0);
  p.head = head;
  cudaStream_t st = (cudaStream_t)stream;
  const bool rowk = kappa_el_stride == 0;
  if (tprime) return rowk ? dispatch_fwd<kPsInjected, true>(p, st) : dispatch_fwd<kPsInjected, false>(p, st);
  return rowk ? dispatch_fwd<kPsRng, true>(p, st) : dispatch_fwd<kPsRng, false>(p, st);
}

int cvb_clifford_ps_rsample(const float* loc, const float* kappa, long long kappa_row_stride, int kappa_el_stride,
                            long long loc_rows, const float* tprime, const float* gnoise, unsigned long long seed,
                            unsigned long long offset, float* z, float* tp_signed, float* entropy, float* kl,
                            float* dentropy, long long rows, int d, void* stream) {
  return clifford_ps_rsample_impl(loc, kappa, kappa_row_stride, kappa_el_stride, loc_rows, tprime, gnoise, seed, offset, z,
                                  tp_signed, entropy, kl, dentropy, rows, d, KappaHead{0, 0.f, 0.f}, stream);
}

// the same launch with the concentration head folded in: kappa = min(softplus(raw_scale) + floor, kmax) per row
// (mnist/mlp_vae.py:69-71, cnn/models.py:96,99); dentropy_draw = d entropy / d raw_scale
int cvb_clifford_ps_rsample_head(const float* loc, const float* raw_scale, long long loc_rows, float floor, float kmax,
                                 const float* tprime, const float* gnoise, unsigned long long seed,
                                 unsigned long long offset, float* z, float* tp_signed, float* entropy, float* kl,
                                 float* dentropy_draw, long long rows, int d, void* stream) {
  CVB_REQUIRE(kmax > floor && floor >= 0.f, kBadArgument, "cvb_clifford_ps_rsample_head: need 0 <= floor < kmax (floor=%g kmax=%g)", (double)floor, (double)kmax);
  return clifford_ps_rsample_impl(loc, raw_scale, 1, 0, loc_rows, tprime, gnoise, seed, offset, z, tp_signed, entropy, kl,
                                  dentropy_draw, rows, d, KappaHead{1, floor, kmax}, stream);
}

// rsample + log q(z) of the drawn sample in one pass (IWAE / evaluation path, mnist/mlp_vae.py:146-190)
int cvb_clifford_ps_rsample_log_prob(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                     const float* gnoise, unsigned long long seed, unsigned long long offset, float* z,
                                     float* log_prob, float* entropy, float* kl, long long rows, int d, void* stream) {
  CVB_REQUIRE(loc && kappa && z && log_prob, kBadArgument, "cvb_clifford_ps_rsample_log_prob: null pointer");
  CVB_REQUIRE(rows > 0 && loc_rows > 0, kBadArgument, "cvb_clifford_ps_rsample_log_prob: rows=%lld loc_rows=%lld", rows, loc_rows);
  CVB_REQUIRE((tprime == nullptr) == (gnoise == nullptr), kBadArgument, "cvb_clifford_ps_rsample_log_prob: give both tprime and gnoise or neither");
  CVB_REQUIRE(is_pow2(d) && d >= 16 && d <= 8192 && aligned(z, 8), kUnsupported,
              "cvb_clifford_ps_rsample_log_prob: d=%d must be a power of two in [16, 8192] (use rsample + log_prob otherwise)", d);
  cudaStream_t st = (cudaStream_t)stream;
  CVB_CUDA(cudaMemsetAsync(log_prob, 0, sizeof(float) * (size_t)rows, st));     // the kernel accumulates two addends per row
  CliffordFwdParams p{};
  p.loc = loc; p.kappa = kappa; p.kappa_row_stride = 1; p.kappa_el_stride = 0; p.loc_rows = (int)loc_rows;
  p.tprime = tprime; p.gnoise = gnoise; p.z = z; p.entropy = entropy; p.kl = kl; p.log_prob = log_prob; p.rows = rows;
  p.d = d; p.n = 2 * d; p.key = make_key(seed, offset, 0);
  return tprime ? dispatch_fwd<kPsInjected, true>(p, st) : dispatch_fwd<kPsRng, true>(p, st);
}

int cvb_clifford_phases_to_vector(const float* phases, float phase_scale, unsigned long long seed,
                                  unsigned long long offset, float* z, long long rows, int d, void* stream) {
  CVB_REQUIRE(z && rows > 0 && d >= 1, kBadArgument, "cvb_clifford_phases_to_vector: bad arguments");
  CliffordFwdParams p{};
  p.loc_rows = 1; p.phases = phases; p.phase_scale = phase_scale; p.z = z; p.rows = rows; p.d = d; p.n = 2 * d;
  p.key = make_key(seed, offset, 1);
  cudaStream_t st = (cudaStream_t)stream;
  return phases ? dispatch_fwd<kPhases, true>(p, st) : dispatch_fwd<kUniformRng, true>(p, st);
}

// CliffordTorusDistribution.rsample (dists/clifford.py:261-275): von Mises phases -> Hermitian phasors -> C2R iFFT
int cvb_clifford_vm_rsample(const float* loc, const float* kappa, long long kappa_row_stride, int kappa_el_stride,
                            long long loc_rows, unsigned long long seed, unsigned long long offset, float* z,
                            long long rows, int d, void* stream) {
  CVB_REQUIRE(loc && kappa && z, kBadArgument, "cvb_clifford_vm_rsample: null pointer");
  CVB_REQUIRE(rows > 0 && d >= 1 && loc_rows > 0, kBadArgument, "cvb_clifford_vm_rsample: rows=%lld d=%d loc_rows=%lld", rows, d, loc_rows);
  CliffordFwdParams p{};
  p.loc = loc; p.kappa = kappa; p.kappa_row_stride = kappa_row_stride; p.kappa_el_stride = kappa_el_stride;
  p.loc_rows = (int)loc_rows; p.z = z; p.rows = rows; p.d = d; p.n = 2 * d;
  p.key = make_key(seed, offset, 3);
  return dispatch_fwd<kVonMisesRng, false>(p, (cudaStream_t)stream);
}

// the same draws (same key, same kernels) with the offsets phi saved for cvb_clifford_vm_rsample_backward and, for one
// concentration per row, the row entropy / KL to the uniform prior / dH/dkappa of vm_entropy_kernel in the same launch
int cvb_clifford_vm_rsample_kl(const float* loc, const float* kappa, long long kappa_row_stride, int kappa_el_stride,
                               long long loc_rows, unsigned long long seed, unsigned long long offset, float* z, float* phi,
                               float* entropy, float* kl, float* dentropy, long long rows, int d, void* stream) {
  CVB_REQUIRE(loc && kappa && z, kBadArgument, "cvb_clifford_vm_rsample_kl: null pointer");
  CVB_REQUIRE(rows > 0 && d >= 1 && loc_rows > 0, kBadArgument, "cvb_clifford_vm_rsample_kl: rows=%lld d=%d loc_rows=%lld", rows, d, loc_rows);
  CVB_REQUIRE(kappa_el_stride == 0 || (!entropy && !kl && !dentropy), kBadArgument,
              "cvb_clifford_vm_rsample_kl: fused entropy/kl needs one concentration per row; use cvb_clifford_vm_entropy");
  CliffordFwdParams p{};
  p.loc = loc; p.kappa = kappa; p.kappa_row_stride = kappa_row_stride; p.kappa_el_stride = kappa_el_stride;
  p.loc_rows = (int)loc_rows; p.z = z; p.tp_signed = phi; p.entropy = entropy; p.kl = kl; p.dentropy = dentropy;
  p.rows = rows; p.d = d; p.n = 2 * d;
  p.key = make_key(seed, offset, 3);
  return dispatch_fwd<kVonMisesRng, false>(p, (cudaStream_t)stream);
}

// fused sample + entropy/KL + bind with a second vector (one concentration per row; power-of-two d in [16, 8192])
int cvb_clifford_ps_rsample_bind(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                 const float* gnoise, unsigned long long seed, unsigned long long offset, const float* b,
                                 long long b_rows, float* z, float* bound, float* entropy, float* kl, float* dentropy,
                                 long long rows, int d, void* stream) {
  CVB_REQUIRE(loc && kappa && b && bound, kBadArgument, "cvb_clifford_ps_rsample_bind: null pointer");
  CVB_REQUIRE(rows > 0 && loc_rows > 0 && b_rows > 0, kBadArgument, "cvb_clifford_ps_rsample_bind: bad sizes");
  CVB_REQUIRE((tprime == nullptr) == (gnoise == nullptr), kBadArgument, "cvb_clifford_ps_rsample_bind: give both tprime and gnoise or neither");
  CVB_REQUIRE(is_pow2(d) && d >= 16 && d <= 8192 && aligned(b, 8) && aligned(bound, 8) && (!z || aligned(z, 8)), kUnsupported,
              "cvb_clifford_ps_rsample_bind: d=%d must be a power of two in [16, 8192] (use rsample + vsa_bind otherwise)", d);
  CliffordFwdParams p{};
  p.loc = loc; p.kappa = kappa; p.kappa_row_stride = 1; p.kappa_el_stride = 0; p.loc_rows = (int)loc_rows;
  p.tprime = tprime; p.gnoise = gnoise; p.z = z; p.entropy = entropy; p.kl = kl; p.dentropy = dentropy; p.rows = rows;
  p.d = d; p.n = 2 * d; p.key = make_key(seed, offset, 0); p.bind_b = b; p.bind_b_rows = b_rows; p.bind_out = bound;
  cudaStream_t st = (cudaStream_t)stream;
  return tprime ? dispatch_fwd_bind<kPsInjected>(p, st) : dispatch_fwd_bind<kPsRng>(p, st);
}

// adjoint of "first d bins of the real FFT of a length-2d row": grad_value (rows, 2d) from H (rows, d) complex
int cvb_clifford_spectrum_adjoint(const float* h_complex, float* grad_value, long long rows, int d, void* stream) {
  CVB_REQUIRE(h_complex && grad_value && rows > 0 && d >= 1, kBadArgument, "cvb_clifford_spectrum_adjoint: bad arguments");
  CliffordFwdParams p{};
  // X_k = (n/2) H_k so that irfft's 1/n leaves H_k / 2 (and Re H_0 after the DC doubling)
  p.loc_rows = 1; p.phases = h_complex; p.phase_scale = (float)d; p.z = grad_value; p.rows = rows; p.d = d; p.n = 2 * d;
  p.spectrum_input = 1;
  return dispatch_fwd<kSpectrum, true>(p, (cudaStream_t)stream);
}

// used by api_vsa.cu
int cvb_internal_unitary(float* out, long long n, int d, float eps, unsigned long long seed, unsigned long long offset,
                         void* stream) {
  CliffordFwdParams p{};
  // n = d output samples, (d-1)/2 free phases at bins 1..; p.d is only the per-row pitch of the RNG index
  p.loc_rows = 1; p.phase_scale = eps; p.z = out; p.rows = n; p.n = d; p.d = (d & 1) ? (d + 1) / 2 : d / 2;
  p.key = make_key(seed, offset, 2);
  return dispatch_fwd<kUnitaryRng, true>(p, (cudaStream_t)stream);
}

}  // extern "C"
