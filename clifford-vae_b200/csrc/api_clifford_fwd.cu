// C ABI entry points for the Clifford-torus kernels (include/clifford_b200.h).
#include <cstdlib>
#include "launch.cuh"
#include "clifford_kernels.cuh"
#include "clifford_small.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

namespace {

constexpr size_t kGenericSmemLimit = 200 * 1024;

template <int LOG2N, int MODE, bool ROWK, bool LEAN = false>
int launch_fwd_fast(const CliffordFwdParams& p, cudaStream_t st) {
  using Pl = FftPlan<LOG2N>;
  const cplx* tw = device_twiddles();
  const float2* icdf = device_icdf_table();
  if (!tw || !icdf) return kCudaError;
  const size_t smem = clifford_fwd_smem_bytes<LOG2N, MODE>();
  auto kern = clifford_fwd_kernel<LOG2N, MODE, ROWK, false, LEAN>;
  int grid = 0;
  const long long work = (p.rows + Pl::GROUPS - 1) / Pl::GROUPS;
  if (int rc = persistent_grid(kern, Pl::THREADS, smem, work, &grid)) return rc;
  if constexpr (LEAN) {
    // (only reachable when the kernel is built for 7 resident CTAs / SM, -DCVB_FWD_LEAN_MINB=7: they won 2-3 % once a CTA
    // looped over >= 8 rows, but the longer row latency cost 1-2 % when a CTA only gets 3-5 rows (B = 4096 at d = 2048);
    // the default build is capped for 6, see clifford_kernels.cuh)
    const int sms = sm_count();
    if (grid == sms * 7) {
      const double rows_per_cta = (double)work / (double)grid;
      if (rows_per_cta > 2.0 && rows_per_cta < 6.0) grid = sms * 6;
    }
  }
  static const bool static_sched = getenv("CVB_STATIC_SCHEDULE") != nullptr;
  const bool dynamic = !static_sched && work > grid;                         // dynamic rows only when CTAs loop
  if constexpr (MODE == kPsRng && ROWK && !LEAN) {
    // plain forward sampling: the specialised variant (no optional outputs, staged inputs)
    if (!p.tp_signed && !p.log_prob && p.staged && !p.head.on) return launch_fwd_fast<LOG2N, MODE, ROWK, true>(p, st);
  }
  CliffordFwdParams q = p;
  q.sched = dynamic ? next_sched_slot() : nullptr;
  launch_pdl(kern, grid, Pl::THREADS, smem, st, q, tw, icdf);
  return check_launch("clifford_fwd_kernel");
}

template <int LOG2N, int MODE>
int launch_fwd_bind(const CliffordFwdParams& p, cudaStream_t st) {
  using Pl = FftPlan<LOG2N>;
  const cplx* tw = device_twiddles();
  const float2* icdf = device_icdf_table();
  if (!tw || !icdf) return kCudaError;
  const size_t smem = clifford_fwd_smem_bytes<LOG2N, MODE, true>();
  auto kern = clifford_fwd_kernel<LOG2N, MODE, true, true>;
  int grid = 0;
  const long long work = (p.rows + Pl::GROUPS - 1) / Pl::GROUPS;
  if (int rc = persistent_grid(kern, Pl::THREADS, smem, work, &grid)) return rc;
  CliffordFwdParams q = p;
  static const bool static_sched = getenv("CVB_STATIC_SCHEDULE") != nullptr;
  q.sched = (!static_sched && work > grid) ? next_sched_slot() : nullptr;
  launch_pdl(kern, grid, Pl::THREADS, smem, st, q, tw, icdf);
  return check_launch("clifford_fwd_kernel<bind>");
}

template <int MODE>
int dispatch_fwd_bind(const CliffordFwdParams& p_in, cudaStream_t st) {
  CliffordFwdParams p = p_in;
  p.staged = aligned(p.loc, 16) && (!p.tprime || aligned(p.tprime, 16)) && (!p.gnoise || aligned(p.gnoise, 16)) &&
             getenv("CVB_NO_TMA") == nullptr;
  switch (ilog2(p.d)) {
#define CVB_CASE(L) case L: return launch_fwd_bind<L, MODE>(p, st);
    CVB_CASE(4) CVB_CASE(5) CVB_CASE(6) CVB_CASE(7) CVB_CASE(8) CVB_CASE(9) CVB_CASE(10) CVB_CASE(11) CVB_CASE(12)
    CVB_CASE(13)
#undef CVB_CASE
  }
  return kUnsupported;
}

template <int MODE, bool ROWK>
int dispatch_fwd(const CliffordFwdParams& p_in, cudaStream_t st) {
  CliffordFwdParams p = p_in;
  p.staged = (!p.loc || aligned(p.loc, 16)) && (!p.tprime || aligned(p.tprime, 16)) && (!p.gnoise || aligned(p.gnoise, 16)) &&
             (!p.phases || aligned(p.phases, 16)) && getenv("CVB_NO_TMA") == nullptr;
  const bool fast = is_pow2(p.d) && p.d >= 16 && p.d <= 8192 && p.n == 2 * p.d && aligned(p.z, 8);
  if (fast) {
    switch (ilog2(p.d)) {
#define CVB_CASE(L) case L: return launch_fwd_fast<L, MODE, ROWK>(p, st);
      CVB_CASE(4) CVB_CASE(5) CVB_CASE(6) CVB_CASE(7) CVB_CASE(8) CVB_CASE(9) CVB_CASE(10) CVB_CASE(11) CVB_CASE(12)
      CVB_CASE(13)
#undef CVB_CASE
    }
  }
  static const bool no_small = getenv("CVB_NO_SMALL_ROWS") != nullptr;    // A/B switch: the one-CTA-per-row direct DFT
  if (p.n <= kSmallMaxN && !no_small) {
    // short rows (the reference's default MNIST latents, per-token latents): a tile of rows per CTA
    const int rt = small_rows_per_tile(p.rows, sm_count(), [&](int r) { return clifford_fwd_small_smem(p.n, r); });
    const size_t smem_s = clifford_fwd_small_smem(p.n, rt);
    auto kern_s = clifford_fwd_small_kernel<MODE, ROWK>;
    int grid_s = 0;
    if (int rc = persistent_grid(kern_s, kSmallThreads, smem_s, (p.rows + rt - 1) / rt, &grid_s)) return rc;
    kern_s<<<grid_s, kSmallThreads, smem_s, st>>>(p, rt);
    return check_launch("clifford_fwd_small_kernel");
  }
  const int nph = (p.n - 1) / 2;
  const size_t smem = sizeof(cplx) * ((size_t)p.n + nph + 1);
  CVB_REQUIRE(smem <= kGenericSmemLimit, kUnsupported, "clifford rsample: length n=%d too large for the direct-DFT path", p.n);
  auto kern = clifford_fwd_generic_kernel<MODE, ROWK>;
  int grid = 0;
  if (int rc = persistent_grid(kern, kGenericThreads, smem, p.rows, &grid)) return rc;
  kern<<<grid, kGenericThreads, smem, st>>>(p);
  return check_launch("clifford_fwd_generic_kernel");
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
