// Fused Clifford-torus kernels: sample -> Hermitian phasors -> C2R iFFT -> z, with the row
// entropy / KL in the same pass; backward (R2C FFT of grad_z -> dloc, dkappa); log_prob (R2C FFT
// -> angle -> power-spherical log density).  Power-of-two d uses the register/shared-memory FFT
// engine (fft_core.cuh); any other d uses the direct-DFT kernels at the bottom (same element
// math, O(d^2) per row) so every length the reference accepts runs on the device.
//
// Reference semantics: dists/clifford.py:281-327 (CliffordPowerSphericalDistribution),
// :215-242 (CliffordTorusUniform), utils/vsa.py:15-36 (unitary_init); closed forms in
// SURVEY.md section 8(a).
#pragma once
#include "fft_core.cuh"
#include "tma.cuh"
#include "rng.cuh"
#include "icdf_table.cuh"
#include "special.cuh"
// Minimum resident CTAs per SM requested for the forward kernel's 128-thread configurations (register cap 102 at 5).
// Measured on B200 (device RNG, >= 1 GiB per launch): 5 beats 4 by 2-4 % at d = 512 / 2048 and loses 2 % at d = 1024.
#ifndef CVB_FWD_MINB
#define CVB_FWD_MINB 5
#endif
// backward: 5 resident CTAs help at d = 2048 (+7 %) and d = 512 (+6 %), hurt at d = 1024 (-2 %); log_prob: 4 is best at every size
template <int LOG2N>
constexpr int clifford_bwd_min_blocks() { return LOG2N == 10 ? 4 : 5; }
#ifndef CVB_FWD_BIND_MINB
#define CVB_FWD_BIND_MINB 4
#endif
// the fused-bind variant carries a second set of transforms; since its pair stage forms each (k, N-k) pair once it fits 124
// registers without spilling: 4 resident CTAs / SM measured 0.1166 -> 0.1069 ms at the headline shape (3 before; 5 does not
// fit the shared memory)
#ifndef CVB_FWD_KEEP_OWN
#define CVB_FWD_KEEP_OWN 1
#endif
#ifndef CVB_ICDF_LOOP_UNROLL
#define CVB_ICDF_LOOP_UNROLL 4
#endif
// The lean forward sampler at d = 2048: its shared memory (33.9 KB per CTA) admits 6 resident CTAs, so the register cap
// is set for 6 (85 registers) -- room to keep a table row's own phasors in registers between the sampling loop and the
// C2R pre-tangle (CVB_FWD_KEEP_OWN: -16 shared-memory reads per thread and row, +3 %; at the 72-register cap of 7 CTAs
// that spills 116 bytes and loses 10 %).
#ifndef CVB_FWD_LEAN_MINB
#define CVB_FWD_LEAN_MINB 6
#endif
template <int LOG2N, bool BIND = false, bool LEAN = false>
constexpr int clifford_fwd_min_blocks() {
  return BIND ? CVB_FWD_BIND_MINB : ((LEAN && LOG2N == 11) ? CVB_FWD_LEAN_MINB : (LOG2N == 10 ? 4 : CVB_FWD_MINB));
}

namespace cvb {

enum CliffordMode : int {
  kPsInjected = 0,   // t' and g supplied (parity mode)
  kPsRng = 1,        // Philox on device
  kPhases = 2,       // theta = phase_scale * phases[row, k]   (uniform prior with injected u; unitary init)
  kUniformRng = 3,   // theta = 2 pi U
  kUnitaryRng = 4,   // theta = sign * pi * (eps + a (1 - 2 eps))   (utils/vsa.py:15-36)
  kSpectrum = 5,     // X_k = phase_scale * H[row, k] given as complex (rows, d): adjoint of the truncated real FFT
  kVonMisesRng = 6,  // theta = loc + VonMises(0, kappa) draw  (CliffordTorusDistribution, dists/clifford.py:261-275)
};

struct CliffordFwdParams {
  const float* loc;        // (loc_rows, d)
  const float* kappa;      // element (r, k) at kappa[r * kappa_row_stride + k * kappa_el_stride]
  long long kappa_row_stride;
  int kappa_el_stride;     // 0: one concentration per row
  int loc_rows;            // rows are (sample, batch) flattened: row r uses loc/kappa row r % loc_rows
  const float* tprime;     // (rows, d) injected Beta draws           [kPsInjected]
  const float* gnoise;     // (rows, d) injected N(0,1) sign draws    [kPsInjected]
  const float* phases;     // (rows, d)                               [kPhases]
  float phase_scale;       //                                         [kPhases]; eps for kUnitaryRng
  float* z;                // (rows, n) out
  float* tp_signed;        // (rows, d) out, optional: copysign(t', s) saved for backward [kPsRng]; the von Mises offset
                           // phi [kVonMisesRng]
  float* entropy;          // (rows) out, optional (row-scalar kappa only)
  float* kl;               // (rows) out, optional (row-scalar kappa only)
  float* dentropy;         // (rows) out, optional: d entropy / d kappa (row-scalar kappa only)
  float* log_prob;         // (rows) in/out, optional, ZERO on entry: log q(z) of the drawn sample itself (row-scalar kappa,
                           // FFT path only) -- the phases are known, so no FFT -> angle round trip (clifford.py:310-316)
  long long rows;
  int d;                   // phases per row (row pitch of loc / draws / phases)
  int n;                   // output length: 2d for the torus (fast path); any n >= 2 on the direct-DFT path
  int staged;              // 1: input rows are 16-byte aligned -> stage them with cp.async.bulk
  int spectrum_input;      // kSpectrum: `phases` holds (rows, d) complex values
  int* sched;              // [0] next-row counter, [1] finished-group counter (both zero between launches); null = static
  const float* bind_b;     // fused bind tail: rows of length 2d to bind each sample with (row r uses r % bind_b_rows), or null
  long long bind_b_rows;
  float* bind_out;         // (rows, 2d): irfft(S * rfft(bind_b)) = bind(z, b) without re-transforming z (its spectrum S is known)
  KappaHead head;          // on: `kappa` holds the raw head output (row scalar only); dentropy is then d entropy / d raw
  PhiloxKey key;
};
// the row's concentration (row-scalar layouts): through the folded head when one is given
// (NOHEAD: the launcher guarantees head.on == 0 -- the register-capped LEAN variant compiles the head out)
template <bool NOHEAD = false>
__device__ __forceinline__ float fwd_row_kappa(const CliffordFwdParams& p, long long prow) {
  const float raw = __ldg(p.kappa + prow * p.kappa_row_stride);
  return NOHEAD ? raw : head_kappa(p.head, raw);
}

constexpr float kEps = 1e-7f;
// the forward sampler's table carries the padding cell of icdf_build_row<.., PAD> (index = floor(x) unclamped)
constexpr int kFwdIcdfCells = kIcdfCells + 1;
constexpr int kIcdfLoopUnroll = CVB_ICDF_LOOP_UNROLL;   // Philox calls (4 circles each) of the table sampling loop unrolled together
// the reference's atan2(s sqrt(max(1 - t^2, eps)), t) (clifford.py:44-48) never returns a phase below sqrt(eps) or above
// pi - sqrt(eps): the table sampler clamps |phi| to that range
constexpr float kIcdfPhiMin = 3.16227766e-4f, kIcdfPhiMax = 3.14127642f;
#ifndef CVB_TABLE_COORD_MIN_LOG2N
#define CVB_TABLE_COORD_MIN_LOG2N 9
#endif
// which row lengths save the table coordinate instead of t' on table-sampled rows (see clifford_bwd_smem_bytes)
template <int LOG2N>
constexpr bool clifford_saves_table_coord() { return LOG2N >= CVB_TABLE_COORD_MIN_LOG2N; }

__device__ __forceinline__ float sign_from_normal(float g) { return g / (fabsf(g) + kEps); }

// Pieces of phi = atan2(s sqrt(max(1 - t^2, eps)), t), t = 2 t' - 1   (clifford.py:44-48,:300)
struct CirclePhase {
  float c, s;        // cos phi, sin phi
  float dphi_dt;     // d phi / d t
};
__device__ __forceinline__ CirclePhase circle_phase(float tp, float sgn) {
  const float t = 2.0f * tp - 1.0f;
  const float om = fmaf(-t, t, 1.0f);
  const float sq = fast_sqrt(fmaxf(om, kEps));
  const float y1 = sgn * sq;
  const float r2 = fmaf(t, t, y1 * y1);
  const float rinv = rsqrtf(r2);
  CirclePhase o;
  o.c = t * rinv;
  o.s = y1 * rinv;
  const float dy1 = (om > kEps) ? (-sgn * t / sq) : 0.0f;
  o.dphi_dt = (t * dy1 - y1) / r2;
  return o;
}

// sin/cos of an arbitrary-range angle.  FAST: two-constant Cody-Waite reduction to [-pi, pi] + the
// MUFU approximations (abs error ~4e-7; used with device RNG where the draw itself is random);
// otherwise the accurate library routine (parity mode).
template <bool FAST>
__device__ __forceinline__ void sincos_any(float x, float& s, float& c) {
  if (FAST) {
    // n = rint(x / 2 pi) by the 1.5 * 2^23 trick (|x| < 2^22 * 2 pi): two FP-pipe instructions, no FRND on the MUFU unit
    const float n = fmaf(x, 0.15915494309189535f, 12582912.0f) - 12582912.0f;
    float r = fmaf(-n, 6.28318548202514648f, x);        // 2 pi rounded to fp32 ...
    r = fmaf(-n, -1.74845553146951715e-7f, r);          // ... and its remainder
    __sincosf(r, &s, &c);
  } else {
    sincosf(x, &s, &c);
  }
}

// e^{i (loc + phi)} from a Beta draw t' and a sign
template <bool FAST>
__device__ __forceinline__ cplx ps_phasor(float tp, float sgn, float loc) {
  float pc, psn;
  if (FAST) {
    // (t, s sqrt(max(1 - t^2, eps))) already has norm 1 to within 1e-7 (also when the clamp is active), so the
    // atan2 -> exp round trip of the reference is the identity here: skip the renormalisation
    pc = fmaf(2.0f, tp, -1.0f);
    psn = sgn * fast_sqrt(fmaxf(fmaf(-pc, pc, 1.0f), kEps));
  } else {
    const CirclePhase ph = circle_phase(tp, sgn);
    pc = ph.c; psn = ph.s;
  }
  float sl, cl;
  sincos_any<FAST>(loc, sl, cl);
  return make_float2(fmaf(cl, pc, -sl * psn), fmaf(sl, pc, cl * psn));
}

// One von Mises(0, kappa) draw by Best & Fisher's wrapped-Cauchy rejection, in double like the sampler the reference
// calls (torch/distributions/von_mises.py:93-190 `_rejection_sample` + `_proposal_r` with its small-kappa Taylor
// branch); acceptance >= 0.66.  Its pathwise gradient is the implicit one of vm_dphi_dkappa below (the draw itself is
// not a differentiable function of kappa).
__device__ __forceinline__ float von_mises_draw(float kappa_f, const PhiloxKey& key, uint64_t elem) {
  const double kap = (double)kappa_f;
  const double tau = 1.0 + sqrt(1.0 + 4.0 * kap * kap);
  const double rho = (tau - sqrt(2.0 * tau)) / (2.0 * kap);
  const double r = (kap < 1e-5) ? (1.0 / kap + kap) : (1.0 + rho * rho) / (2.0 * rho);
  double x = 0.0;
  for (uint32_t attempt = 0; attempt < 1024; ++attempt) {
    const uint4 w = philox_draw(key, elem, attempt);
    const double u1 = (double)u01_open1(w.x), u2 = (double)u01_open0(w.y);
    const double z = cospi(u1);
    const double f = (1.0 + r * z) / (r + z);
    const double c = kap * (r - f);
    if ((c * (2.0 - c) - u2 > 0.0) || (log(c / u2) + 1.0 - c >= 0.0)) {
      x = ((w.z & 0x80000000u) ? -1.0 : 1.0) * acos(fmin(fmax(f, -1.0), 1.0));
      break;
    }
  }
  return (float)x;
}

// Row constants of the von Mises circle law, fp64 -> fp32: b = 1 - A(kappa), A = I1/I0 (kept as 1 - A: it is 1/(2 kappa)
// for large kappa and every use subtracts from 1), and lnk = ln(2 pi I0(kappa)) - kappa = ln 2 pi + log_ive(0, kappa)
// (the log-normaliser without its kappa, which the log density cancels against kappa cos: see vm_lp_element).
// kappa <= 0 (or NaN) is the uniform circle.
struct VmRowConsts { float b, lnk; };
__device__ __forceinline__ VmRowConsts vm_row_consts(float kappa_f) {
  const double k = (double)kappa_f;
  VmRowConsts c;
  if (k > 0.0) {
    const double l0 = log_ive(0.0, k), l1 = log_ive(1.0, k);
    c.b = (float)(-expm1(l1 - l0));
    c.lnk = (float)(1.83787706640934548356 + l0);
  } else {
    c.b = 1.0f;
    c.lnk = 1.83787706640934548356f;
  }
  return c;
}

// Implicit reparameterisation gradient of a von Mises(0, kappa) draw phi (Figurnov et al. 2018): phi stays at its CDF
// level, d phi / d kappa = -d_kappa F / f, which the even symmetry and int_{-pi}^{pi} (cos t - A) e^{kappa cos t} dt = 0
// reduce to
//   J(phi) = -int_0^phi (cos t - A) e^{kappa (cos t - cos phi)} dt = +int_phi^pi (cos t - A) e^{kappa (cos t - cos phi)} dt
// (odd in phi; -sin phi as kappa -> 0).  fp32, 12-point Gauss-Legendre per panel, b = 1 - A from vm_row_consts.  With
// S = sin(phi/2), C = cos(phi/2), x = kappa (1 - cos phi) = 2 kappa S^2:
//   x <= 3 (the bulk of every law): the first form on [0, |phi|] in t; the exponent lies in [0, x], the integrand is
//     smooth, and kappa (cos t - cos phi) = 2 kappa sin((phi+t)/2) sin((phi-t)/2), cos t - A = b - 2 sin^2(t/2) keep
//     their relative accuracy when kappa is large;
//   x > 3 (tail draws): the second form, whose integrand has one sign and exponent <= 0 (the first form cancels e^x-sized
//     halves there).  With s = sin(t/2), s^2 = S^2 + C^2 sin^2 psi it is
//       int_0^{pi/2} ((cos phi - A) - 2 C^2 sin^2 psi) e^{-2 kappa C^2 sin^2 psi} 2 C sin psi / sqrt(S^2 + C^2 sin^2 psi) dpsi,
//     integrated on [pi/4, pi/2] in psi (skipped once e^{-kappa C^2} is below fp32 resolution) and on [0, pi/4] in
//     eta, C sin psi = S sinh eta, which removes the branch point near psi = 0: the integrand becomes
//     ((cos phi - A) - 2 S^2 sinh^2 eta) e^{-x sinh^2 eta} 2 tan psi, cut where x sinh^2 eta = 40.
// Against fp64 adaptive quadrature over kappa in [1e-6, 1e4] and phi up to pi: <= 6.2e-7 max(1, |J|) (12 nodes; 8 give
// 1.5e-5).  Finite for every finite (phi, kappa >= 0): every exponent is <= 3.
__device__ __forceinline__ float vm_dphi_dkappa(float phi, float kap, float b) {
  constexpr float kNode[12] = {9.219682877e-03f, 4.794137181e-02f, 1.150486629e-01f, 2.063410229e-01f, 3.160842505e-01f,
                               4.373832957e-01f, 5.626167043e-01f, 6.839157495e-01f, 7.936589771e-01f, 8.849513371e-01f,
                               9.520586282e-01f, 9.907803171e-01f};
  constexpr float kWeight[12] = {2.358766819e-02f, 5.346966300e-02f, 8.003916427e-02f, 1.015837134e-01f, 1.167462683e-01f,
                                 1.245735229e-01f, 1.245735229e-01f, 1.167462683e-01f, 1.015837134e-01f, 8.003916427e-02f,
                                 5.346966300e-02f, 2.358766819e-02f};     // Gauss-Legendre on [0, 1]
  const float a = fabsf(phi);
  float S, C;
  sincosf(0.5f * a, &S, &C);
  const float x = 2.0f * kap * S * S;
  float J;
  if (!(x > 3.0f)) {
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const float t = a * kNode[i];
      const float st = sinf(0.5f * t);
      const float e = 2.0f * kap * sinf(0.5f * (a + t)) * sinf(0.5f * (a - t));
      acc = fmaf(kWeight[i], fmaf(-2.0f * st, st, b) * expf(e), acc);
    }
    J = -a * acc;
  } else {
    const float cma = fmaf(-2.0f * S, S, b);                  // cos phi - A  (< 0 here)
    const float r = S / C;
    const float e1 = asinhf(fminf(0.70710678f / r, sqrtf(40.0f / x)));
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const float sh = sinhf(e1 * kNode[i]);
      const float sp = r * sh;                                // sin psi <= 1/sqrt 2
      const float tanp = sp * rsqrtf(fmaf(-sp, sp, 1.0f));
      acc = fmaf(kWeight[i], fmaf(-2.0f * S * S, sh * sh, cma) * expf(-x * sh * sh) * 2.0f * tanp, acc);
    }
    J = e1 * acc;
    if (kap * C * C < 40.0f) {
      float acc2 = 0.0f;
#pragma unroll
      for (int i = 0; i < 12; ++i) {
        const float sp = sinf(0.78539816f * (1.0f + kNode[i]));
        const float c2s2 = C * C * sp * sp;
        acc2 = fmaf(kWeight[i], fmaf(-2.0f, c2s2, cma) * expf(-2.0f * kap * c2s2) * 2.0f * C * sp * rsqrtf(fmaf(S, S, c2s2)), acc2);
      }
      J = fmaf(0.78539816f, acc2, J);
    }
  }
  return phi < 0.0f ? -J : J;                        // odd in phi
}

// von Mises torus entropy (reference dists/clifford.py:21-31 `_von_mises_entropy`, :277-278): per circle
//   h(kappa) = ln 2 pi + ln a + kappa - kappa b / a,   a = i0e(kappa) + 1e-7,  b = i1e(kappa) + 1e-7
// summed over circles k >= 1.  i0e / i1e from the fp64 log I_v e^{-x} of special.cuh (the reference's are torch's fp32
// Chebyshev fits: agreement ~1e-7 relative); the eps regularisation and the final arithmetic follow the reference.
// dh/dkappa (optional) is the exact derivative of that regularised expression:
//   a' = i1e - i0e,  b' = i0e - i1e (1 + 1/kappa):   h' = a'/a + 1 - b/a - kappa (b' a - b a') / a^2
struct VmEntropy { float h, dh; };
__device__ __forceinline__ VmEntropy vm_circle_entropy(float kappa_f) {
  const double k = (double)kappa_f;
  double i0e = 1.0, i1e = 0.0;
  if (k > 0.0) { i0e = exp(log_ive(0.0, k)); i1e = exp(log_ive(1.0, k)); }
  const double eps = (double)1e-7f;
  const double a = (double)(float)(i0e) + eps, b = (double)(float)(i1e) + eps;   // the reference adds eps to fp32 values
  VmEntropy o;
  o.h = (float)(1.83787706640934548356 + log(a) + k - k * (b / a));
  const double da = i1e - i0e, db = (k > 0.0) ? i0e - i1e * (1.0 + 1.0 / k) : 0.5;
  o.dh = (float)(da / a + 1.0 - b / a - k * (db * a - b * da) / (a * a));
  return o;
}

// Per-row input pointers, indexed by the bin k: either the global rows or their staged copies in
// shared memory (generic loads serve both).
struct RowSrc {
  const float* loc;
  const float* tprime;
  const float* gnoise;
  const float* phases;
};
__device__ __forceinline__ RowSrc global_row_src(const CliffordFwdParams& p, long long row, long long prow) {
  RowSrc s;
  s.loc = p.loc ? p.loc + prow * p.d : nullptr;
  s.tprime = p.tprime ? p.tprime + row * p.d : nullptr;
  s.gnoise = p.gnoise ? p.gnoise + row * p.d : nullptr;
  s.phases = p.phases ? p.phases + row * p.d * (p.spectrum_input ? 2 : 1) : nullptr;
  return s;
}

// e^{i theta_k} for bin k (1 <= k <= d-1) of `row`.  For kPsRng a rejected first half-angle envelope
// proposal returns false (the caller queues k and finishes it with clifford_phasor_retry).
template <int MODE, bool ROWK>
__device__ __forceinline__ bool clifford_phasor(const CliffordFwdParams& p, const RowSrc& src, long long row,
                                                long long prow, int k, HalfAngle& gm, cplx& out) {
  const long long idx = row * p.d + k;
  if (MODE == kPsInjected) {
    const float tp = src.tprime[k];
    const float s = sign_from_normal(src.gnoise[k]);
    out = ps_phasor<false>(tp, s, src.loc[k]);
    return true;
  }
  if (MODE == kPsRng) {
    if (!ROWK) gm = HalfAngle(__ldg(p.kappa + prow * p.kappa_row_stride + (long long)k * p.kappa_el_stride) + kEps);
    float tp, s;
    if (!circle_beta_first(gm, p.key, (uint64_t)idx, tp, s)) return false;
    if (p.tp_signed) stg_stream1(p.tp_signed + idx, copysignf(tp, s));
    out = ps_phasor<true>(tp, s, src.loc[k]);
    return true;
  }
  float th;
  if (MODE == kVonMisesRng) {
    const float kap = __ldg(p.kappa + prow * p.kappa_row_stride + (long long)k * p.kappa_el_stride);
    PhiloxKey vkey = p.key;
    vkey.stream = 11;
    const float phi = von_mises_draw(kap, vkey, (uint64_t)idx);
    if (p.tp_signed) stg_stream1(p.tp_signed + idx, phi);     // the drawn offset, saved for the backward
    th = src.loc[k] + phi;
    sincosf(th, &out.y, &out.x);
    return true;
  }
  if (MODE == kSpectrum) {
    const float2 hv = reinterpret_cast<const float2*>(src.phases)[k];
    out = make_float2(p.phase_scale * hv.x, p.phase_scale * hv.y);
    return true;
  }
  if (MODE == kPhases) {
    th = p.phase_scale * src.phases[k];
    sincosf(th, &out.y, &out.x);
    return true;
  }
  const uint4 r = philox_draw(p.key, (uint64_t)idx, 0);
  if (MODE == kUniformRng) {
    th = 6.283185307179586f * u01_open1(r.x) - 3.14159265358979f;      // same law as 2 pi U, kept in [-pi, pi)
  } else {
    const float a = u01_open1(r.x);
    const float sg = (r.y & 0x80000000u) ? -1.0f : 1.0f;
    th = sg * 3.14159265358979f * (p.phase_scale + a * (1.0f - 2.0f * p.phase_scale));
  }
  __sincosf(th, &out.y, &out.x);
  return true;
}

template <bool ROWK, bool LEAN = false>
__device__ __forceinline__ cplx clifford_phasor_retry(const CliffordFwdParams& p, const RowSrc& src, long long row,
                                                      long long prow, int k, HalfAngle& gm, float& tp_out) {
  const long long idx = row * p.d + k;
  if (!ROWK) gm = HalfAngle(__ldg(p.kappa + prow * p.kappa_row_stride + (long long)k * p.kappa_el_stride) + kEps);
  float s;
  const float tp = circle_beta_retry(gm, p.key, (uint64_t)idx, s);
  if (!LEAN && p.tp_signed) stg_stream1(p.tp_signed + idx, copysignf(tp, s));
  tp_out = tp;
  return ps_phasor<true>(tp, s, src.loc[k]);
}

// log1p(clamp(t, -1 + eps, 1 - eps)) - ln 2 for t = 2 t' - 1, i.e. ln of t' clamped to the fp32 images of the
// reference's bounds (clifford.py:200-201: float32(-1 + 1e-7) = -1 + 2^-23, float32(1 - 1e-7) = 1 - 2^-23)
template <bool FAST>
__device__ __forceinline__ float circle_log_half_1pt(float tp) {
  const float c = fminf(fmaxf(tp, 5.9604645e-8f), 0.99999994f);
  return FAST ? __logf(c) : logf(c);
}

template <bool NOHEAD = false>
__device__ __forceinline__ void clifford_row_entropy(const CliffordFwdParams& p, long long row, float kap_row, const PsConsts& c);
template <bool NOHEAD = false>
__device__ __forceinline__ void clifford_row_entropy(const CliffordFwdParams& p, long long row, float kap_row) {
  clifford_row_entropy<NOHEAD>(p, row, kap_row, ps_consts((double)kap_row, 0.5));
}
template <bool NOHEAD>
__device__ __forceinline__ void clifford_row_entropy(const CliffordFwdParams& p, long long row, float kap_row, const PsConsts& c) {
  const double ent = (double)(p.d - 1) * c.entropy;
  if (p.entropy) p.entropy[row] = (float)ent;
  if (p.kl) p.kl[row] = (float)((double)(p.d - 1) * 1.83787706640934548356 - ent);
  if (p.dentropy) {
    const float chain = (!NOHEAD && p.head.on) ? head_dkappa(p.head, __ldg(p.kappa + (row % p.loc_rows) * p.kappa_row_stride)) : 1.0f;
    p.dentropy[row] = (float)((double)(p.d - 1) * c.dentropy) * chain;
  }
  if (p.log_prob) {
    // the sample-independent part of log q(z): d log C + kappa ((d-1) ln 2 + log1p(clamp(cos loc_0)))  (bin 0 has angle 0);
    // the row loop adds kappa * sum_k ln t'_k.  Two commutative adds onto zero: order-independent.
    const float c0 = cosf(__ldg(p.loc + (row % p.loc_rows) * p.d));
    const double l0 = log1p((double)fminf(fmaxf(c0, -1.0f + kEps), 1.0f - kEps));
    atomicAdd(p.log_prob + row, (float)((double)p.d * c.log_norm +
                                        (double)kap_row * ((double)(p.d - 1) * 0.69314718055994530942 + l0)));
  }
}

// von Mises torus rows (kVonMisesRng, one concentration per row): the row entropy / KL to the uniform prior / dH/dkappa
// of the sampled rows, the same arithmetic as vm_entropy_kernel, one row per thread of the whole launch (the launcher
// requests them only when kappa_el_stride == 0)
__device__ __forceinline__ void vm_fwd_row_entropies(const CliffordFwdParams& p, long long first, long long step) {
  if (!(p.entropy || p.kl || p.dentropy)) return;
  for (long long row = first; row < p.rows; row += step) {
    const VmEntropy e = vm_circle_entropy(__ldg(p.kappa + (row % p.loc_rows) * p.kappa_row_stride));
    const float h = (float)(p.d - 1) * e.h;
    if (p.entropy) p.entropy[row] = h;
    if (p.kl) p.kl[row] = (float)((double)(p.d - 1) * 1.83787706640934548356 - (double)h);
    if (p.dentropy) p.dentropy[row] = (float)(p.d - 1) * e.dh;
  }
}

// Shared memory per group: exchange buffer (XCH cplx) | retry queue (N ints) | up to 3 staged input
// rows (N floats each) ; then per group one mbarrier and one queue counter.
typedef unsigned short QueueIndex;   // retry-queue entries are bin indices < N <= 8192
constexpr int kLpSlots = 16;   // per-warp partial sums of the fused log_prob (groups of up to 512 threads)
constexpr int clifford_fwd_stages(int mode) { return mode == kPsInjected ? 3 : ((mode == kPsRng || mode == kPhases) ? 1 : 0); }
// Device-RNG rows with one concentration <= kIcdfKappaMax are sampled through the row's inverse-CDF table
// (icdf_table.cuh) when the row is long enough to amortise building it (d >= 512: 256 cells by >= 32 threads).
template <int LOG2N, int MODE>
constexpr bool clifford_fwd_has_icdf() { return MODE == kPsRng && LOG2N >= 9; }
template <int LOG2N, int MODE, bool BIND = false>
constexpr size_t clifford_fwd_smem_bytes() {
  using Pl = FftPlan<LOG2N>;
  return (sizeof(cplx) * Pl::XCH + sizeof(QueueIndex) * Pl::N + sizeof(float) * Pl::N * clifford_fwd_stages(MODE) +
          (BIND ? sizeof(cplx) * Pl::N : 0) + (clifford_fwd_has_icdf<LOG2N, MODE>() ? sizeof(float4) * kFwdIcdfCells : 0)) * Pl::GROUPS +
         (sizeof(uint64_t) + sizeof(int) * 2 + sizeof(float) * kLpSlots) * Pl::GROUPS;
}

// BIND: after the sample is written, the row is also bound with a second vector -- out = irfft(S * rfft(b)) -- reusing
// the sample's known spectrum S (the phasors), i.e. bind(z, b) for two transforms instead of three and without
// reading z back.  p.z may then be null (only the bound vector is wanted): the sample's own inverse FFT is skipped.
// LEAN: the launcher guarantees tp_signed == log_prob == nullptr (plain forward sampling) and staged inputs, so the
// predicated-off instructions of the optional outputs and the global-memory input path are compiled out (+8 %).
// (Also assuming the dynamic schedule / always-valid rows was measured: +2 % at d = 512 / 1024, -2 % at d = 2048.)
template <int LOG2N, int MODE, bool ROWK, bool BIND = false, bool LEAN = false>
__global__ void __launch_bounds__(FftPlan<LOG2N>::THREADS, (FftPlan<LOG2N>::THREADS <= 128 ? clifford_fwd_min_blocks<LOG2N, BIND, LEAN>() : 1))
clifford_fwd_kernel(const CliffordFwdParams p, const cplx* __restrict__ tw, const float2* __restrict__ icdf) {
  pdl_wait_and_release();
  using Pl = FftPlan<LOG2N>;
  constexpr int d = Pl::N, T = Pl::T, E = Pl::E, G = Pl::GROUPS;
  constexpr int NST = clifford_fwd_stages(MODE);
  constexpr bool ICDF = clifford_fwd_has_icdf<LOG2N, MODE>() && ROWK;
  constexpr uint32_t kRowBytes = d * sizeof(float);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int group = threadIdx.x / T, t = threadIdx.x % T;
  // layout: [G x NST x stage rows][G x xch][G x queue][G x mbarrier][G x (qcount, pad)]
  float* stage = reinterpret_cast<float*>(smem_raw) + (size_t)group * NST * d;
  unsigned char* after_stage = smem_raw + sizeof(float) * (size_t)G * NST * d;
  cplx* xch = reinterpret_cast<cplx*>(after_stage) + (size_t)group * Pl::XCH;
  QueueIndex* queue = reinterpret_cast<QueueIndex*>(after_stage + sizeof(cplx) * (size_t)G * Pl::XCH) + (size_t)group * d;
  uint64_t* bar = reinterpret_cast<uint64_t*>(after_stage + (sizeof(cplx) * Pl::XCH + sizeof(QueueIndex) * d) * (size_t)G) + group;
  int* qcount = reinterpret_cast<int*>(after_stage + (sizeof(cplx) * Pl::XCH + sizeof(QueueIndex) * d + sizeof(uint64_t)) * (size_t)G) + 2 * group;
  float* lps = reinterpret_cast<float*>(after_stage + (sizeof(cplx) * Pl::XCH + sizeof(QueueIndex) * d + sizeof(uint64_t) + 2 * sizeof(int)) * (size_t)G) + kLpSlots * group;
  cplx* spec = reinterpret_cast<cplx*>(after_stage + (sizeof(cplx) * Pl::XCH + sizeof(QueueIndex) * d + sizeof(uint64_t) + 2 * sizeof(int) + kLpSlots * sizeof(float)) * (size_t)G) + (size_t)group * d;   // BIND only
  // row inverse-CDF cells (16-byte aligned: every block before it is a multiple of 16 bytes per CTA)
  float4* cells = reinterpret_cast<float4*>(after_stage + (sizeof(cplx) * Pl::XCH + sizeof(QueueIndex) * d + sizeof(uint64_t) + 2 * sizeof(int) + kLpSlots * sizeof(float) + (BIND ? sizeof(cplx) * d : 0)) * (size_t)G) + (size_t)group * kFwdIcdfCells;
  constexpr bool PS = (MODE == kPsInjected || MODE == kPsRng);
  const long long stride = (long long)gridDim.x * G;
  const bool staged = LEAN ? true : (NST > 0 && p.staged);   // LEAN implies TMA-staged inputs (16-byte aligned rows)

  // issue the bulk copies of one row's inputs (thread 0 of the group)
  auto issue = [&](long long row) {
    const long long prow = row % p.loc_rows;
    mbar_expect_tx(bar, NST * kRowBytes);
    if (MODE == kPsInjected) {
      tma_load_1d(stage, p.loc + prow * d, kRowBytes, bar);
      tma_load_1d(stage + d, p.tprime + row * d, kRowBytes, bar);
      tma_load_1d(stage + 2 * d, p.gnoise + row * d, kRowBytes, bar);
    } else if (MODE == kPsRng) {
      tma_load_1d(stage, p.loc + prow * d, kRowBytes, bar);
    } else if (MODE == kPhases) {
      tma_load_1d(stage, p.phases + row * d, kRowBytes, bar);
    }
  };

  if (t == 0) {
    *qcount = 0;
    if (staged) { mbar_init(bar, 1); mbar_init_fence(); }
  }
  __syncthreads();
  const long long first_row = (long long)blockIdx.x * G + group;
  if (staged && t == 0 && first_row < p.rows) issue(first_row);
  // a row is table-sampled when its concentration is inside the table's range; the cells of the first row are built
  // here, those of every later row right after the previous row's sampling phase (their loads overlap its FFT)
  // (kap >= 0: the unclamped cell index floor(256 v^(1/(2 kap + 1))) stays inside the table only for a valid concentration;
  // a negative or NaN one -- invalid input -- takes the exact sampler like before)
  auto icdf_row_ok = [&](float kap) { return kap >= 0.0f && kap + kEps <= kIcdfKappaMax; };
  if (ICDF && first_row < p.rows) {
    const float k0 = fwd_row_kappa<LEAN || BIND>(p, first_row % p.loc_rows);
    if (icdf_row_ok(k0)) icdf_build_row<false, 4, true>(cells, k0 + kEps, icdf, t, T);
  }

  // Prologue: the closed-form row entropy / KL / dH/dkappa (fp64 special functions) of every row this
  // group will process, one row per thread, so the per-row loop carries no serial fp64 chain.
  const bool want_lp = !LEAN && PS && ROWK && p.log_prob != nullptr;
  if (PS && ROWK && (p.entropy || p.kl || p.dentropy || p.log_prob)) {
    if constexpr (T >= 32) {
      // A PAIR of lanes per row: the even lane evaluates lgamma / digamma / trigamma of a = 1/2 + kappa + eps, the odd lane
      // those of a + 1/2 -- one instruction stream, so the two chains run side by side and the serial fp64 chain ahead of
      // the group's first row is halved (a group rarely has more than T/2 rows: 4096 rows over 888 groups = 5 each).
      const int part = t & 1;
      for (long long jb = 0; first_row + jb * stride < p.rows; jb += T / 2) {      // uniform over the group's warps
        const long long row = first_row + (jb + (t >> 1)) * stride;
        const bool mine = row < p.rows;
        const float kap = mine ? fwd_row_kappa<LEAN || BIND>(p, row % p.loc_rows) : 1.0f;
        const double a = 0.5 + ((double)kap + 1e-7);
        double lg, ps, p1;
        gamma_family(part ? a + 0.5 : a, lg, ps, p1);
        const double lgt = __shfl_xor_sync(0xffffffffu, lg, 1), pst = __shfl_xor_sync(0xffffffffu, ps, 1),
                     p1t = __shfl_xor_sync(0xffffffffu, p1, 1);
        if (mine && !part)
          clifford_row_entropy<LEAN || BIND>(p, row, kap, ps_consts_from((double)kap, 0.5, lg, ps, p1, lgt, pst, p1t));
      }
    } else {
      for (long long row = first_row + (long long)t * stride; row < p.rows; row += (long long)T * stride)
        clifford_row_entropy<LEAN || BIND>(p, row, fwd_row_kappa<LEAN || BIND>(p, row % p.loc_rows));
    }
  }
  if constexpr (MODE == kVonMisesRng)
    vm_fwd_row_entropies(p, (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);

  // Row schedule.  Static: group g of CTA b takes rows b*G + g + i*stride.  Dynamic (sched != null, groups of
  // >= 32 threads): after its first row a group fetches the next unprocessed row from a global counter, which
  // removes the tail imbalance when rows / (CTAs * G) is small (4096 rows over 740 CTAs: 5 vs 6 rows each).
  const bool dynamic = (T >= 32) && p.sched != nullptr;
  uint32_t parity = 0;
  long long row = first_row;
  const long long loop_end = dynamic ? p.rows : p.rows + (long long)group;   // static: keep trip counts CTA-uniform
  for (; row < loop_end; parity ^= 1u) {
    const bool valid = row < p.rows;
    const long long prow = valid ? (row % p.loc_rows) : 0;
    float kap_row = 1.0f;
    if (PS && valid) kap_row = fwd_row_kappa<LEAN || BIND>(p, prow);
    HalfAngle gm(kap_row + kEps);
    if (dynamic && t == 0) qcount[1] = atomicAdd(p.sched, 1);              // broadcast through smem after the barrier
    RowSrc src;
    if (staged) {
      src.loc = stage; src.tprime = stage + d; src.gnoise = stage + 2 * d; src.phases = stage;
      if (valid) mbar_wait(bar, parity);
    } else {
      src = global_row_src(p, valid ? row : 0, prow);
    }
    group_sync<LOG2N>();                       // the previous row's exchange-buffer readers are done
    const long long next_row = dynamic ? (long long)qcount[1] + stride : row + stride;
    float lp_acc = 0.0f;                       // fused log_prob: this thread's sum of ln t'_k
    // per-warp partial sums into the group's slots (read by thread 0 after the next group barrier)
    auto lp_reduce = [&]() {
      constexpr int W = T < 32 ? T : 32;
      float sum = lp_acc;
#pragma unroll
      for (int o = W / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if ((t & 31) == 0) lps[t >> 5] = sum;
    };
    auto lp_emit = [&]() {
      if (t == 0 && valid) {
        float sum = 0.0f;
#pragma unroll
        for (int i = 0; i < (T + 31) / 32; ++i) sum += lps[i];
        atomicAdd(p.log_prob + row, kap_row * sum);
      }
    };
    // phase 1: phasors of the half spectrum into the exchange buffer (lightly unrolled: small code, some ILP)
    const bool table_row = ICDF && icdf_row_ok(kap_row);      // uniform over the group
    constexpr bool KEEP_OWN = CVB_FWD_KEEP_OWN && ICDF && !BIND;    // table rows keep their own phasors in registers
    cplx xown[KEEP_OWN ? E : 1];
    if (ICDF && table_row) {
      // device RNG through the row's inverse-CDF cells: one Philox call per FOUR circles, no rejection, no queue
      const uint64_t quad_base = (uint64_t)row * (uint64_t)(d / 4) + (uint64_t)t * (E / 4);
      const uint32_t call_off = philox_call_offset(p.key);      // once per row, not once per Philox call
      const float inv_p = __frcp_rn(fmaf(2.0f, kap_row + kEps, 1.0f));
#pragma unroll kIcdfLoopUnroll
      for (int e = 0; e < E; e += 4) {
        const uint4 r = philox_draw_at(p.key, 10u, call_off, quad_base + (e >> 2));
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = t + (e + j) * T;
          // phi = s max(|phi|, sqrt(eps)): the reference's atan2(s sqrt(max(1 - t^2, eps)), t) (clifford.py:44-48) never
          // returns a phase below sqrt(eps); theta = loc + phi needs ONE sincos instead of sincos(loc), cos/sin(phi)
          // and a complex multiply
          float xs;                                       // table coordinate of this draw (> 0)
          const float aphi = fminf(fmaxf(icdf_sample_phi_t<true>(cells, inv_p, w[j], xs), kIcdfPhiMin), kIcdfPhiMax);   // [sqrt(eps), pi - sqrt(eps)]
          const float phi = __uint_as_float(__float_as_uint(aphi) | (w[j] & 0x80000000u));
          if (!LEAN && valid && k != 0) {
            // saved for the backward: the signed table coordinate (NOT t'): clifford_bwd_kernel re-evaluates the phase and
            // its pathwise kappa-derivative from the row's cells (table rows only; exact-sampler rows save copysign(t', s))
            if (p.tp_signed) {
              const float keep = clifford_saves_table_coord<LOG2N>() ? xs : icdf_tprime(aphi);
              stg_stream1(p.tp_signed + row * d + k, __uint_as_float(__float_as_uint(keep) | (w[j] & 0x80000000u)));
            }
            if (want_lp) lp_acc += circle_log_half_1pt<true>(icdf_tprime(aphi));
          }
          // unconditional (no per-circle branch): bin 0 is overwritten with 1 after the loop, and the phasors of an invalid
          // row (static schedule padding; finite garbage from the staged buffer) are never stored
          cplx x;
          sincos_any<true>(src.loc[k] + phi, x.y, x.x);
          if (KEEP_OWN) {
            if (e + j == 0) x = (t == 0) ? make_float2(1.0f, 0.0f) : x;      // bin 0 (one select in the whole loop)
            xown[KEEP_OWN ? e + j : 0] = x;
          }
          xch[pad16(k)] = x;
        }
      }
      if (!KEEP_OWN && t == 0) xch[pad16(0)] = make_float2(1.0f, 0.0f);      // same thread wrote bin 0 above: program order suffices
    } else if (MODE == kPsRng) {
      // device RNG: one Philox call + one Box-Muller per PAIR of bins (one envelope proposal each);
      // rejected proposals are queued and finished in phase 1b
      const uint64_t pair_base = (uint64_t)row * (uint64_t)(d / 2) + (uint64_t)t * (E / 2);
      PhiloxKey pkey = p.key;
      pkey.stream = 8;
      uint32_t rej_mask = 0;                    // bit e: this thread's element e was rejected
#pragma unroll 2
      for (int e = 0; e < E; e += 2) {
        const int k0 = t + e * T, k1 = k0 + T;
        HalfAngle h0 = gm, h1 = gm;
        if (!ROWK && valid) {
          h0 = HalfAngle(__ldg(p.kappa + prow * p.kappa_row_stride + (long long)k0 * p.kappa_el_stride) + kEps);
          h1 = HalfAngle(__ldg(p.kappa + prow * p.kappa_row_stride + (long long)k1 * p.kappa_el_stride) + kEps);
        }
        float tp[2], sg[2];
        const uint4 r1 = philox_draw(pkey, pair_base + (e >> 1), 0);
        uint4 r2 = r1;
        if (!ROWK && ((h0.sigma > 0.f) != (h1.sigma > 0.f))) r2 = philox_draw(pkey, pair_base + (e >> 1), 0x80u);   // mixed regimes
        const uint32_t acc = half_angle_pair(h0, h1, r1, r2, tp, sg);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int k = j ? k1 : k0;
          cplx x = make_float2(1.0f, 0.0f);
          if (valid && k != 0) {
            if (acc & (1u << j)) {
              if (!LEAN && p.tp_signed) stg_stream1(p.tp_signed + row * d + k, copysignf(tp[j], sg[j]));
              if (want_lp) lp_acc += circle_log_half_1pt<true>(tp[j]);
              x = ps_phasor<true>(tp[j], sg[j], src.loc[k]);
            } else {
              rej_mask |= 1u << (e + j);
            }
          }
          xch[pad16(k)] = x;
        }
      }
      // queue the rejected bins: one shared-memory atomic per warp (exclusive scan of the per-thread counts) instead
      // of one contended atomic per rejected bin
      if (T >= 32) {
        const int lane = threadIdx.x & 31, cnt = __popc(rej_mask);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int up = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += up;
        }
        int base = 0;
        if (lane == 31 && incl > 0) base = atomicAdd(qcount, incl);
        base = __shfl_sync(0xffffffffu, base, 31);
        int pos = base + incl - cnt;
        while (rej_mask) {
          const int e = __ffs(rej_mask) - 1;
          rej_mask &= rej_mask - 1;
          queue[pos++] = (QueueIndex)(t + e * T);
        }
      } else {
        while (rej_mask) {
          const int e = __ffs(rej_mask) - 1;
          rej_mask &= rej_mask - 1;
          queue[atomicAdd(qcount, 1)] = (QueueIndex)(t + e * T);
        }
      }
    } else if (MODE == kUniformRng || MODE == kUnitaryRng) {
      // one uniform phase per circle: one Philox call serves four circles (one 32-bit word each; for the
      // unitary initialiser the top bit is the sign draw and the next 24 bits the magnitude draw)
      const uint32_t call_off = philox_call_offset(p.key);      // once per row, not once per Philox call
      const uint64_t quad_base = (uint64_t)row * (uint64_t)(d / 4) + (uint64_t)t * (E / 4);
#pragma unroll 2
      for (int e = 0; e < E; e += 4) {
        const uint4 r = philox_draw_at(p.key, 9u, call_off, quad_base + (e >> 2));
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = t + (e + j) * T;
          float th;
          if (MODE == kUniformRng) {
            th = 6.283185307179586f * u01_open1(w[j]) - 3.14159265358979f;        // same law as 2 pi U, kept in [-pi, pi)
          } else {
            const float a = (float)((w[j] >> 7) & 0xFFFFFFu) * 0x1p-24f;
            const float sg = (w[j] & 0x80000000u) ? -1.0f : 1.0f;
            th = sg * 3.14159265358979f * (p.phase_scale + a * (1.0f - 2.0f * p.phase_scale));
          }
          cplx x = make_float2(1.0f, 0.0f);
          if (valid && k != 0) __sincosf(th, &x.y, &x.x);
          xch[pad16(k)] = x;
        }
      }
    } else {
#pragma unroll 4
      for (int e = 0; e < E; ++e) {
        const int k = t + e * T;
        cplx x = make_float2(1.0f, 0.0f);
        if (MODE == kSpectrum) {
          // adjoint of F_k = sum_j v_j e^{-2 pi i jk/n}, k < d: grad_v = n irfft(X), X_0 = Re H_0, X_k = H_k / 2, X_d = 0
          x = make_float2(0.f, 0.f);
          if (valid) {
            clifford_phasor<MODE, ROWK>(p, src, row, prow, k, gm, x);
            if (k == 0) x = make_float2(2.0f * x.x, 0.0f);
          }
        } else if (valid && k != 0) {
          clifford_phasor<MODE, ROWK>(p, src, row, prow, k, gm, x);
          if (MODE == kPsInjected && want_lp) lp_acc += circle_log_half_1pt<false>(src.tprime[k]);
        }
        xch[pad16(k)] = x;
      }
    }
    if (t == 0) xch[pad16(d)] = make_float2(MODE == kSpectrum ? 0.0f : 1.0f, 0.0f);
    if (MODE == kPsInjected && want_lp) lp_reduce();
    group_sync<LOG2N>();
    if (MODE == kPsInjected && want_lp) lp_emit();
    if (ICDF && table_row) {
      if (want_lp) { lp_reduce(); group_sync<LOG2N>(); lp_emit(); }
    } else if (MODE == kPsRng) {
      // phase 1b: rejected proposals, spread evenly over the group's threads
      const int nq = *qcount;
#pragma unroll 1
      for (int i = t; i < nq; i += T) {
        const int k = queue[i];
        float tp_r;
        xch[pad16(k)] = clifford_phasor_retry<ROWK, LEAN>(p, src, row, prow, k, gm, tp_r);
        if (want_lp) lp_acc += circle_log_half_1pt<true>(tp_r);
      }
      if (want_lp) lp_reduce();
      group_sync<LOG2N>();
      if (want_lp) lp_emit();
      if (t == 0) *qcount = 0;
    }
    // every thread is done with the staged inputs: fetch the next row's while this one is transformed
    if (staged && t == 0 && next_row < p.rows) issue(next_row);
    if (ICDF && next_row < p.rows) {
      // ... and with this row's cells: build the next row's (the loop-top barrier orders them before its sampling)
      const float kn = fwd_row_kappa<LEAN || BIND>(p, next_row % p.loc_rows);
      if (icdf_row_ok(kn)) icdf_build_row<false, 1, true>(cells, kn + kEps, icdf, t, T);
    }
    // phase 2: Hermitian half spectrum -> packed complex spectrum -> inverse FFT -> real row
    cplx v[E];
    if (BIND) {
      // keep this thread's phasors S[k] for the bind tail (own slots only: no barrier needed)
#pragma unroll
      for (int e = 0; e < E; ++e) spec[t + e * T] = xch[pad16(t + e * T)];
    }
    if (!BIND || p.z) {
      if constexpr (KEEP_OWN) {
        if (table_row) {
#pragma unroll
          for (int e = 0; e < E; ++e) v[e] = xown[KEEP_OWN ? e : 0];
          c2r_pretangle_load<LOG2N, true>(v, xch, t, tw);
        } else {
          c2r_pretangle_load<LOG2N>(v, xch, t, tw);
        }
      } else {
        c2r_pretangle_load<LOG2N>(v, xch, t, tw);
      }
      fft_run<LOG2N, true>(v, xch, t, tw);
      if (valid) {
        float2* zr = reinterpret_cast<float2*>(p.z + row * (2LL * d));
#pragma unroll
        for (int e = 0; e < E; ++e) stg_stream2(zr + t + e * T, v[e]);
      }
    }
    if (BIND) {
      // bind tail: R = rfft(b) (half-length FFT + untangle), P = S * R (S[0] = S[d] = 1), out = irfft(P)
      const float2* br = reinterpret_cast<const float2*>(p.bind_b + (valid ? row % p.bind_b_rows : 0) * (2LL * d));
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = valid ? ldg_stream2(br + t + e * T) : make_float2(0.f, 0.f);
      fft_run<LOG2N, false>(v, xch, t, tw);
      // One partner exchange: bins k and N-k of R = rfft(b) from Z_b[k], Z_b[N-k]; P = S * R with the sample's own
      // phasors S (spec[]; S[0] = S[N] = 1); both re-packed values V[k] = c (s + q), V[N-k] = c conj(s - q) for the inverse
      // half-length transform.  Each pair is formed once, by the owner of k < N/2; the partner value returns through
      // spec[N-k] (the slot this thread just consumed).
      group_sync<LOG2N>();
#pragma unroll
      for (int e = E / 2; e < E; ++e) xch[pad16(t + e * T)] = v[e];      // partners only ever read bins > N/2
      group_sync<LOG2N>();
      auto pair = [&](int k, int kp, cplx zb, cplx& vk, cplx& vkp) {
        constexpr float fold = 0.5f / (2.0f * d);
        const cplx zbp = cconj(kp == k ? zb : xch[pad16(kp)]);
        const cplx w = __ldg(&tw[twiddle_offset(LOG2N) + k]);
        const cplx sb = cadd(zb, zbp), db = cmul_mi(cmul(w, csub(zb, zbp)));
        const cplx Bk = cadd(sb, db), Bkp = cconj(csub(sb, db));             // 2 R[k], 2 R[N-k]
        const cplx Pk = cmul(spec[k], Bk), Pkpc = cconj(cmul(spec[kp], Bkp));
        const cplx s = cadd(Pk, Pkpc), q = cmul_i(cmul(cconj(w), csub(Pk, Pkpc)));
        vk = cadd_scaled(s, q, fold);
        vkp = cconj(cscale(csub(s, q), fold));
      };
#pragma unroll
      for (int e = 0; e < E / 2; ++e) {
        const int k = t + e * T, kp = (d - k) & (d - 1);
        cplx vkp;
        pair(k, kp, v[e], v[e], vkp);
        if (kp != k) spec[kp] = vkp;
      }
      if (t == 0) {
        cplx vk, vkp;
        pair(d / 2, d / 2, v[E / 2], vk, vkp);
        spec[d / 2] = vk;
      }
      group_sync<LOG2N>();
#pragma unroll
      for (int e = E / 2; e < E; ++e) v[e] = spec[t + e * T];
      fft_run<LOG2N, true>(v, xch, t, tw);
      if (valid) {
        float2* orow = reinterpret_cast<float2*>(p.bind_out + row * (2LL * d));
#pragma unroll
        for (int e = 0; e < E; ++e) stg_stream2(orow + t + e * T, v[e]);
      }
    }
    row = next_row;
  }
  if (dynamic && t == 0) {
    // the last group to finish re-arms the counters for the next launch that uses this slot
    if (atomicAdd(p.sched + 1, 1) == (int)stride - 1) { p.sched[0] = 0; p.sched[1] = 0; }
  }
  if (MODE == kPsRng || MODE == kUniformRng || MODE == kUnitaryRng || MODE == kVonMisesRng) rng_launch_done(p.key);
}

// ---- backward of rsample ---------------------------------------------------------------------
struct CliffordBwdParams {
  const float* grad_z;     // (rows, 2d)
  const float* loc;
  const float* kappa;
  long long kappa_row_stride;
  int kappa_el_stride;
  int loc_rows;
  const float* tprime;     // injected draws (rows, d), or null when tp_signed is given
  const float* gnoise;
  const float* tp_signed;  // saved by the RNG forward
  float* dloc;             // (rows, d) out
  float* dkappa;           // ROWK: (rows) row sums; else (rows, d)
  long long rows;
  int d;
  int staged;              // 1: element-input rows are 16-byte aligned -> stage them with cp.async.bulk
  KappaHead head;          // on: `kappa` holds the raw head output (row scalar only) and dkappa receives d L / d raw
  int* sched;              // dynamic row schedule: {next-row counter, finished-CTA counter} (launcher), or null = static
};

// Per-row inputs of the backward, indexed by the bin k (global rows or their TMA-staged copies in smem).
struct BwdRowSrc {
  const float* loc;
  const float* tps;      // saved copysign(t', s)  (RNG forward), or null
  const float* tprime;   // injected draws
  const float* gnoise;
};

// Element k of the backward: returns dL/dtheta_k, accumulates / stores dL/dkappa_k.
// SAVED: the launcher guarantees the RNG forward's saved draws (src.tps != null): the injected-draw path is compiled out.
template <bool ROWK, class RowGrad, bool SAVED = false>
__device__ __forceinline__ float clifford_bwd_element(const CliffordBwdParams& p, const BwdRowSrc& src, long long row,
                                                      long long prow, int k, cplx Gk, RowGrad& bc, float inv_d,
                                                      float& dk) {
  const long long idx = row * p.d + k;
  float tp, s;
  if (SAVED || src.tps) {
    const float ts = src.tps[k];
    tp = fabsf(ts);
    s = (ts < 0.f) ? -1.0f : 1.0f;
  } else {
    tp = src.tprime[k];
    s = sign_from_normal(src.gnoise[k]);
  }
  const CirclePhase ph = circle_phase(tp, s);       // identical arithmetic to the forward
  float sl, cl;
  if (SAVED || src.tps) sincos_any<true>(src.loc[k], sl, cl);
  else sincos_any<false>(src.loc[k], sl, cl);
  const cplx x = make_float2(fmaf(cl, ph.c, -sl * ph.s), fmaf(sl, ph.c, cl * ph.s));
  // dL/dtheta_k = -(2/n) Im(X_k conj(G_k)), 2/n = 1/d
  const float dth = -inv_d * (x.y * Gk.x - x.x * Gk.y);
  float dtp;
  if (ROWK) {
    dtp = bc.grad(tp) * (1.0f - tp);
  } else {
    const BetaGradConsts be(0.5f + (__ldg(p.kappa + prow * p.kappa_row_stride + (long long)k * p.kappa_el_stride) + kEps), 0.5f);
    dtp = dirichlet_grad_one<false>(tp, be) * (1.0f - tp);
  }
  dk = dth * ph.dphi_dt * 2.0f * dtp;
  stg_stream1(p.dloc + idx, dth);
  if (!ROWK) stg_stream1(p.dkappa + idx, dk);
  return dth;
}

// Element k of the von Mises torus backward (src.tps = the offsets phi the forward drew): dL/dloc_k = dL/dtheta_k,
// dL/dkappa_k = dL/dtheta_k * d phi_k / d kappa_k (implicit gradient, vm_dphi_dkappa).  ROWK: kap / b are the row's,
// else the element's are read here.  Returns dL/dkappa_k; stores dL/dloc_k (and dL/dkappa_k unless ROWK).
template <bool ROWK>
__device__ __forceinline__ float vm_bwd_element(const CliffordBwdParams& p, const BwdRowSrc& src, long long row,
                                                long long prow, int k, cplx Gk, float kap, float b, float inv_d) {
  const long long idx = row * p.d + k;
  const float phi = src.tps[k];
  float s, c;
  sincosf(src.loc[k] + phi, &s, &c);                 // theta as the forward formed it
  const float dth = -inv_d * (s * Gk.x - c * Gk.y);   // -(2/n) Im(X_k conj(G_k))
  if (!ROWK) {
    kap = __ldg(p.kappa + prow * p.kappa_row_stride + (long long)k * p.kappa_el_stride);
    b = vm_row_consts(kap).b;
  }
  const float dk = dth * vm_dphi_dkappa(phi, kap, b);
  stg_stream1(p.dloc + idx, dth);
  if (!ROWK) stg_stream1(p.dkappa + idx, dk);
  return dk;
}

// Rows the forward sampled through the inverse-CDF table (device RNG, one concentration <= kIcdfKappaMax per row, d >= 512)
// save the signed TABLE COORDINATE of every draw instead of copysign(t', s), and the backward differentiates
// the table map itself: phase and d phase / d kappa from the row's cells (icdf_phi_and_dkappa) -- the exact pathwise
// derivative of what the sampler evaluated (accurate to 2.5e-5 of the analytic implicit gradient, tests/
// test_icdf_table.py) for ~45 instructions per circle, where ATen's piecewise approximation of the implicit Beta
// gradient (the reference's backward; still used for injected draws and exact-sampler rows) costs ~190 in three
// divergent branches.  (At d = 512 the two 4 KB cell tables per row cost the kernel two of its five resident CTAs and it
// still gains: 25.0 -> 31.9 % of the roofline; d = 2048: 27.6 -> 38.2 %.)
// smem per group: staged rows (loc, tp_signed | tprime, gnoise; FAST: two) | value + derivative cells (table rows) |
// exchange buffer | 32 floats reduction scratch + row constants | mbarrier
template <int LOG2N, bool ROWK = true, bool FAST = false, bool VM = false>
constexpr size_t clifford_bwd_smem_bytes() {
  using Pl = FftPlan<LOG2N>;
  return (sizeof(cplx) * Pl::XCH + sizeof(float) * (32 + 2 * kBetaRowFloats) + sizeof(float) * ((FAST || VM) ? 2 : 3) * Pl::N +
          ((!VM && ROWK && clifford_saves_table_coord<LOG2N>()) ? 2 * sizeof(float4) * kIcdfCells : 0) + sizeof(uint64_t)) * Pl::GROUPS;
}

// FAST: saved draws + TMA-staged element inputs (the training path: backward of a device-RNG rsample with 16-byte
// aligned rows); the injected-draw and unstaged paths are compiled out.
// VM: the von Mises torus family (cvb_clifford_vm_rsample_backward): the staged rows are loc and the saved offsets phi,
// the row constant is 1 - A(kappa) (vm_row_consts) and the element is vm_bwd_element; the R2C transform of grad_z and
// the row schedule are the power-spherical ones.
template <int LOG2N, bool ROWK, bool FAST = false, bool VM = false>
__global__ void __launch_bounds__(FftPlan<LOG2N>::THREADS, (FftPlan<LOG2N>::THREADS <= 128 ? clifford_bwd_min_blocks<LOG2N>() : 1))
clifford_bwd_kernel(const CliffordBwdParams p, const cplx* __restrict__ tw, const float2* __restrict__ icdf) {
  pdl_wait_and_release();
  using Pl = FftPlan<LOG2N>;
  constexpr int d = Pl::N, T = Pl::T, E = Pl::E, G = Pl::GROUPS;
  constexpr uint32_t kRowBytes = d * sizeof(float);
  constexpr bool TABLE = !VM && ROWK && clifford_saves_table_coord<LOG2N>();
  constexpr int NSTAGE = (FAST || VM) ? 2 : 3;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int group = threadIdx.x / T, t = threadIdx.x % T;
  // layout: [G x staged rows][G x (value cells | derivative cells)][G x xch][G x scratch][G x mbarrier]
  float* stage = reinterpret_cast<float*>(smem_raw) + (size_t)group * NSTAGE * d;
  unsigned char* after_rows = smem_raw + sizeof(float) * (size_t)G * NSTAGE * d;
  float4* cells = reinterpret_cast<float4*>(after_rows) + (size_t)group * 2 * kIcdfCells;      // TABLE only
  float4* dcells = cells + kIcdfCells;
  unsigned char* after_stage = after_rows + (TABLE ? sizeof(float4) * 2 * kIcdfCells * (size_t)G : 0);
  cplx* xch = reinterpret_cast<cplx*>(after_stage) + (size_t)group * Pl::XCH;
  constexpr int kScratch = 32 + 2 * kBetaRowFloats;   // reduction scratch | two (double-buffered) row-constant blocks
  float* scratch = reinterpret_cast<float*>(after_stage + sizeof(cplx) * (size_t)G * Pl::XCH) + group * kScratch;
  float* rowconst = scratch + 32;
  uint64_t* bar = reinterpret_cast<uint64_t*>(after_stage + (sizeof(cplx) * Pl::XCH + sizeof(float) * kScratch) * (size_t)G) + group;
  const long long stride = (long long)gridDim.x * G;
  const bool staged = FAST ? true : (p.staged != 0);
  const bool saved = (FAST || VM) ? true : (p.tp_signed != nullptr);

  // bulk copies of one row's element inputs (thread 0 of the group); they land while grad_z is transformed
  auto issue = [&](long long row) {
    const long long prow = row % p.loc_rows;
    mbar_expect_tx(bar, (saved ? 2u : 3u) * kRowBytes);
    tma_load_1d(stage, p.loc + prow * d, kRowBytes, bar);
    if (saved) {
      tma_load_1d(stage + d, p.tp_signed + row * d, kRowBytes, bar);
    } else {
      tma_load_1d(stage + d, p.tprime + row * d, kRowBytes, bar);
      tma_load_1d(stage + 2 * d, p.gnoise + row * d, kRowBytes, bar);
    }
  };
  if (staged) {
    if (t == 0) { mbar_init(bar, 1); mbar_init_fence(); }
    __syncthreads();
    const long long first_row = (long long)blockIdx.x * G + group;
    if (t == 0 && first_row < p.rows) issue(first_row);
  }

  // Row schedule.  Static: CTA b takes rows b*G + g + i*stride.  Dynamic (one row per CTA at a time, sched != null): after
  // its first row a CTA fetches the next unprocessed row from a global counter, which removes the tail imbalance when
  // rows / CTAs is small (4096 rows over 740 CTAs: 5 vs 6 rows each, i.e. 8 % of the launch idle).
  const bool dynamic = (G == 1) && p.sched != nullptr;
  int* next_slot = reinterpret_cast<int*>(scratch) + 31;     // group_sum uses scratch[0 .. T/32)
  uint32_t parity = 0;
  for (long long base = (long long)blockIdx.x * G, next_base = 0; base < p.rows; base = next_base, parity ^= 1u) {
    const long long row = base + group;
    const bool valid = row < p.rows;
    const long long prow = valid ? (row % p.loc_rows) : 0;
    if (dynamic && t == 0) *next_slot = atomicAdd(p.sched, 1);     // published by the barriers of the FFT below
    cplx v[E];
    const float2* gz = reinterpret_cast<const float2*>(p.grad_z + (valid ? row : 0) * (2LL * d));
#pragma unroll
    for (int e = 0; e < E; ++e) v[e] = valid ? ldg_stream2(gz + t + e * T) : make_float2(0.f, 0.f);
    // the row's Beta-gradient constants, built once by the first lanes of the group while grad_z is in flight
    // (published by the barriers of the FFT below; double-buffered against the previous row's readers)
    const float kap_raw = valid ? __ldg(p.kappa + prow * p.kappa_row_stride) : 1.0f;
    const float kap_row = head_kappa(p.head, kap_raw);
    float* rc = rowconst + (parity ? kBetaRowFloats : 0);
    // a row the forward sampled through the table (same predicate as clifford_fwd_kernel; uniform over the group)
    const bool table_row = TABLE && saved && valid && kap_row >= 0.0f && (kap_row + kEps <= kIcdfKappaMax);
    if constexpr (VM) {
      if (ROWK && t == 0) rc[0] = vm_row_consts(kap_row).b;
    } else if (TABLE && table_row) {
      // every thread left the previous row's element loop (its closing barriers) before these are overwritten
      icdf_build_row_both(cells, dcells, kap_row + kEps, icdf, t, T);
    } else if (ROWK) {
      beta_row_build<T>(rc, 0.5f + (kap_row + kEps), 0.5f, t);
    }
    fft_run<LOG2N, false>(v, xch, t, tw);
    r2c_untangle<LOG2N>(v, xch, t, tw);        // v[e] = G[k]
    if constexpr (G == 1) next_base = dynamic ? (long long)*next_slot + stride : base + stride;

    // G[k] goes back to this thread's own exchange slots so that the (large, divergent) element
    // routine runs in a rolled loop: keeps the kernel inside the instruction cache.  (Table-sampled rows consume G[k]
    // straight from the registers instead: their element is ~45 instructions and is unrolled.)
    const bool table_elems = TABLE && table_row;
    if (!table_elems) {
      group_sync<LOG2N>();
#pragma unroll
      for (int e = 0; e < E; ++e) xch[pad16(t + e * T)] = v[e];
    }
    BetaGradRowShared bc(rc);
    BwdRowSrc src;
    if (staged) {
      src.loc = stage;
      src.tps = saved ? stage + d : nullptr;
      src.tprime = stage + d;
      src.gnoise = stage + 2 * d;
      if (valid) mbar_wait(bar, parity);
    } else {
      const long long r0 = valid ? row : 0;
      src.loc = p.loc + prow * d;
      src.tps = saved ? p.tp_signed + r0 * d : nullptr;
      src.tprime = p.tprime ? p.tprime + r0 * d : nullptr;
      src.gnoise = p.gnoise ? p.gnoise + r0 * d : nullptr;
    }
    float dk_sum = 0.f;
    if (TABLE && table_row) {
      // table-sampled row: phase and its pathwise kappa-derivative straight from the row's cells
      const float inv_p = __frcp_rn(fmaf(2.0f, kap_row + kEps, 1.0f));       // as the forward
      constexpr float inv_d = 1.0f / (float)d;
      float* dloc_row = p.dloc + row * d + t;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int k = t + e * T;
        // no branch per circle: bin 0 (only e == 0 of thread 0; the forward never writes its slot) is evaluated like the
        // others on a harmless coordinate and its gradient is zeroed by a select -- two selects in one unrolled iteration
        float sv = src.tps[k];
        if (e == 0) sv = (t == 0) ? 1.0f : sv;
        float dmag;
        const float mag = icdf_phi_and_dkappa(cells, dcells, inv_p, fabsf(sv), dmag);
        const bool clamped = (mag < kIcdfPhiMin) || (mag > kIcdfPhiMax);
        const float aphi = fminf(fmaxf(mag, kIcdfPhiMin), kIcdfPhiMax);
        const float phi = __uint_as_float(__float_as_uint(aphi) | (__float_as_uint(sv) & 0x80000000u));
        cplx x;
        sincos_any<true>(src.loc[k] + phi, x.y, x.x);
        const cplx Gk = v[e];
        float dth = -inv_d * (x.y * Gk.x - x.x * Gk.y);                  // dL/dtheta_k = -(2/n) Im(X_k conj(G_k))
        if (e == 0) dth = (t == 0) ? 0.0f : dth;
        stg_stream1(dloc_row + e * T, dth);
        const float dsigned = __uint_as_float(__float_as_uint(dmag) ^ (__float_as_uint(sv) & 0x80000000u));
        dk_sum = fmaf(dth, clamped ? 0.0f : dsigned, dk_sum);
      }
    } else {
#pragma unroll 2
      for (int e = 0; e < E; ++e) {
        const int k = t + e * T;
        float dk = 0.f;
        if (valid && k != 0) {
          if constexpr (VM) dk = vm_bwd_element<ROWK>(p, src, row, prow, k, xch[pad16(k)], kap_row, rc[0], 1.0f / (float)d);
          else clifford_bwd_element<ROWK, BetaGradRowShared, FAST>(p, src, row, prow, k, xch[pad16(k)], bc, 1.0f / (float)d, dk);
        } else if (valid) {
          stg_stream1(p.dloc + row * d, 0.0f);
          if (!ROWK) stg_stream1(p.dkappa + row * d, 0.0f);
        }
        dk_sum += dk;
      }
    }
    if (staged) {
      group_sync<LOG2N>();                       // every thread is done with the staged rows
      if (t == 0 && (G == 1 ? next_base : base + stride) + group < p.rows) issue((G == 1 ? next_base : base + stride) + group);
    }
    if (ROWK) {
      const float tot = group_sum<LOG2N>(dk_sum, scratch, t);
      if (valid && t == 0) p.dkappa[row] = tot * head_dkappa(p.head, kap_raw);
    } else if (dynamic) {
      group_sync<LOG2N>();                       // next_slot is rewritten at the top of the next row
    }
    if constexpr (G != 1) next_base = base + stride;      // static only: nothing extra kept live across the element loop
  }
  if (dynamic && t == 0) {
    // the last CTA to finish re-arms the counters for the next launch that uses this slot
    if (atomicAdd(p.sched + 1, 1) == (int)stride - 1) { p.sched[0] = 0; p.sched[1] = 0; }
  }
}

// ---- log_prob ----------------------------------------------------------------------------------
struct CliffordLogProbParams {
  const float* value;      // (rows, 2d)
  const float* loc;
  const float* kappa;
  long long kappa_row_stride;
  int kappa_el_stride;
  int loc_rows;
  float* log_prob;         // (rows) out
  float* dlp_dloc;         // optional (rows, d): d log_prob / d loc_k
  float* dlp_dkappa;       // optional; ROWK: (rows), else (rows, d)
  float* dlp_dF;           // optional (rows, d) complex: d log_prob / d (Re F_k, Im F_k), for the gradient w.r.t. value
  long long rows;
  int d;
};

// FWD_ONLY: the launcher guarantees no gradient outputs were requested (evaluation): their code is compiled out.
template <bool ROWK, bool FWD_ONLY = false>
__device__ __forceinline__ void clifford_lp_element(const CliffordLogProbParams& p, long long row, long long prow, int k,
                                                    cplx Fk, float loc_k, float kap, float logc, float dlogc, float& acc,
                                                    float& dk_acc) {
  if (!ROWK) {
    kap = __ldg(p.kappa + prow * p.kappa_row_stride + (long long)k * p.kappa_el_stride);
    const PsConsts c = ps_consts((double)kap, 0.5);
    logc = (float)c.log_norm;
    dlogc = (float)c.dlog_norm;
  }
  // unit vector of the bin's angle; angle(0) = 0 like torch.angle
  const float mag2 = fmaf(Fk.x, Fk.x, Fk.y * Fk.y);
  float ca = 1.0f, sa = 0.0f;
  if (mag2 > 0.f) {
    const float ri = rsqrtf(mag2);
    ca = Fk.x * ri;
    sa = Fk.y * ri;
  }
  float sl, cl;
  // evaluation (no gradient outputs): Cody-Waite reduction + MUFU (abs error 4e-7 on the dot product, against the
  // 1.2e-7 rounding the clamp bounds already carry); the gradient variants keep the accurate routine
  if (FWD_ONLY) sincos_any<true>(loc_k, sl, cl);
  else sincosf(loc_k, &sl, &cl);
  const float dot_raw = fmaf(cl, ca, sl * sa);
  const float dot = fminf(fmaxf(dot_raw, -1.0f + kEps), 1.0f - kEps);
  // evaluation: ln(1 + dot) through MUFU (abs error 3e-7 per circle on terms that sum to O(d)); gradient variants keep log1pf
  const float l1p = FWD_ONLY ? __logf(1.0f + dot) : log1pf(dot);
  acc += logc + kap * l1p;
  if (!FWD_ONLY && p.dlp_dF) {
    // d/dF of kappa log1p(u_hat(F) . m), m = (cos loc, sin loc): kappa / (1 + dot) * (m - dot u_hat) / |F|
    float2 gF = make_float2(0.f, 0.f);
    if (mag2 > 0.f && dot_raw >= -1.0f + kEps && dot_raw <= 1.0f - kEps) {
      const float c = kap / (1.0f + dot) * rsqrtf(mag2);
      gF = make_float2(c * (cl - dot * ca), c * (sl - dot * sa));
    }
    reinterpret_cast<float2*>(p.dlp_dF)[row * p.d + k] = gF;
  }
  if (!FWD_ONLY && p.dlp_dloc) {
    // d dot / d loc = -sin(loc) cos(a) + cos(loc) sin(a); zero where the clamp is active
    const bool inside = (dot_raw >= -1.0f + kEps) && (dot_raw <= 1.0f - kEps);
    const float ddot = inside ? fmaf(cl, sa, -sl * ca) : 0.0f;
    stg_stream1(p.dlp_dloc + row * p.d + k, kap * ddot / (1.0f + dot));
    const float dkv = dlogc + l1p;
    if (ROWK) dk_acc += dkv; else stg_stream1(p.dlp_dkappa + row * p.d + k, dkv);
  }
}

// Element k of the von Mises torus log_prob: kappa cos(a_k - loc_k) - ln(2 pi I0(kappa)) for circles k >= 1 (circle 0 adds
// nothing and gets zero gradients), a_k = angle(F_k), angle(0) = 0.  Evaluated as kappa (cos d - 1) - lnk with
// cos d - 1 = -|u - m|^2 / 2 (u = F_k / |F_k|, m = (cos loc, sin loc)) and lnk = ln 2 pi + log_ive(0, kappa): the two
// kappa-sized halves cancel in closed form instead of in fp32.  d/dloc = kappa sin(a - loc), d/dkappa = cos(a - loc) - A
// = (cos d - 1) + b, d/dF = kappa (m - (u.m) u) / |F|.  ROWK: kap / lnk / b are the row's, else the element's.
template <bool ROWK>
__device__ __forceinline__ void vm_lp_element(const CliffordLogProbParams& p, long long row, long long prow, int k, cplx Fk,
                                              float loc_k, float kap, float lnk, float b, float& acc, float& dk_acc) {
  if (k == 0) {
    if (p.dlp_dF) reinterpret_cast<float2*>(p.dlp_dF)[row * p.d] = make_float2(0.f, 0.f);
    if (p.dlp_dloc) {
      p.dlp_dloc[row * p.d] = 0.f;
      if (!ROWK) p.dlp_dkappa[row * p.d] = 0.f;
    }
    return;
  }
  if (!ROWK) {
    kap = __ldg(p.kappa + prow * p.kappa_row_stride + (long long)k * p.kappa_el_stride);
    const VmRowConsts c = vm_row_consts(kap);
    lnk = c.lnk;
    b = c.b;
  }
  const float mag2 = fmaf(Fk.x, Fk.x, Fk.y * Fk.y);
  float ca = 1.0f, sa = 0.0f;
  if (mag2 > 0.f) {
    const float ri = rsqrtf(mag2);
    ca = Fk.x * ri;
    sa = Fk.y * ri;
  }
  float sl, cl;
  sincosf(loc_k, &sl, &cl);
  const float dc = ca - cl, ds = sa - sl;
  const float cm1 = -0.5f * fmaf(dc, dc, ds * ds);            // cos(a - loc) - 1
  acc += fmaf(kap, cm1, -lnk);
  if (p.dlp_dF) {
    float2 gF = make_float2(0.f, 0.f);
    if (mag2 > 0.f) {
      const float dot = fmaf(cl, ca, sl * sa), c = kap * rsqrtf(mag2);
      gF = make_float2(c * fmaf(-dot, ca, cl), c * fmaf(-dot, sa, sl));
    }
    reinterpret_cast<float2*>(p.dlp_dF)[row * p.d + k] = gF;
  }
  if (p.dlp_dloc) {
    stg_stream1(p.dlp_dloc + row * p.d + k, kap * fmaf(cl, sa, -sl * ca));
    const float dkv = cm1 + b;
    if (ROWK) dk_acc += dkv; else stg_stream1(p.dlp_dkappa + row * p.d + k, dkv);
  }
}

constexpr int kLpConstCache = 256;   // rows per group whose log-normaliser constants are precomputed

// VM: the von Mises torus family (vm_lp_element; row constants (lnk, 1 - A) in place of (log C, dlog C / dkappa)).
template <int LOG2N, bool ROWK, bool FWD_ONLY = false, bool VM = false>
__global__ void __launch_bounds__(FftPlan<LOG2N>::THREADS, (FftPlan<LOG2N>::THREADS <= 128 ? ((FWD_ONLY && LOG2N <= 9) ? 5 : 4) : 1))
clifford_log_prob_kernel(const CliffordLogProbParams p, const cplx* __restrict__ tw) {
  pdl_wait_and_release();
  using Pl = FftPlan<LOG2N>;
  constexpr int d = Pl::N, T = Pl::T, E = Pl::E, G = Pl::GROUPS;
  extern __shared__ cplx smem[];
  const int group = threadIdx.x / T, t = threadIdx.x % T;
  cplx* xch = smem + group * Pl::XCH;
  float* scratch = reinterpret_cast<float*>(smem + G * Pl::XCH) + group * 32;
  float2* ccache = reinterpret_cast<float2*>(reinterpret_cast<float*>(smem + G * Pl::XCH) + G * 32) + group * kLpConstCache;
  float* locs = reinterpret_cast<float*>(reinterpret_cast<float2*>(reinterpret_cast<float*>(smem + G * Pl::XCH) + G * 32) +
                                         G * kLpConstCache) + (size_t)group * d;     // this row's loc, parked for the rolled loop
  const long long stride = (long long)gridDim.x * G;
  const long long first_row = (long long)blockIdx.x * G + group;

  // Prologue: (log C, dlog C/dkappa) of the first kLpConstCache rows of this group, one row per thread (fp64)
  if (ROWK) {
    for (int i = t; i < kLpConstCache; i += T) {
      const long long row = first_row + (long long)i * stride;
      if (row < p.rows) {
        if constexpr (VM) {
          const VmRowConsts c = vm_row_consts(__ldg(p.kappa + (row % p.loc_rows) * p.kappa_row_stride));
          ccache[i] = make_float2(c.lnk, c.b);
        } else {
          const PsConsts c = ps_consts((double)__ldg(p.kappa + (row % p.loc_rows) * p.kappa_row_stride), 0.5);
          ccache[i] = make_float2((float)c.log_norm, (float)c.dlog_norm);
        }
      }
    }
  }
  group_sync<LOG2N>();

  int iter = 0;
  for (long long base = (long long)blockIdx.x * G; base < p.rows; base += stride, ++iter) {
    const long long row = base + group;
    const bool valid = row < p.rows;
    const long long prow = valid ? (row % p.loc_rows) : 0;
    cplx v[E];
    const float2* vz = reinterpret_cast<const float2*>(p.value + (valid ? row : 0) * (2LL * d));
#pragma unroll
    for (int e = 0; e < E; ++e) v[e] = valid ? ldg_stream2(vz + t + e * T) : make_float2(1.f, 0.f);
    float locv[E];
#pragma unroll
    for (int e = 0; e < E; ++e) locv[e] = valid ? ldg_stream1(p.loc + prow * d + t + e * T) : 0.f;   // in flight during the FFT
    fft_run<LOG2N, false>(v, xch, t, tw);
    r2c_untangle<LOG2N>(v, xch, t, tw);        // v[e] = F[k], k = 0..d-1

    const float kap_row = valid ? __ldg(p.kappa + prow * p.kappa_row_stride) : 1.0f;
    float logc = 0.f, dlogc = 0.f;
    if (ROWK) {
      if (iter < kLpConstCache) {
        const float2 c = ccache[iter];
        logc = c.x; dlogc = c.y;
      } else if constexpr (VM) {
        const VmRowConsts c = vm_row_consts(kap_row);
        logc = c.lnk;
        dlogc = c.b;
      } else {
        const PsConsts c = ps_consts((double)kap_row, 0.5);
        logc = (float)c.log_norm;
        dlogc = (float)c.dlog_norm;
      }
    }
    if constexpr (FWD_ONLY && ROWK && !VM) {
      // Evaluation with one concentration per row: the element is ~20 instructions (MUFU sincos / rsqrt / lg2), so it is
      // unrolled over the registers that already hold F[k] and loc[k] -- no round trip through shared memory, no barrier,
      // no branch per bin (angle(0) = 0 by a select); sum_k (log C + kappa l_k) = d log C + kappa sum_k l_k per thread.
      float lsum = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const cplx Fk = v[e];
        const float mag2 = fmaf(Fk.x, Fk.x, Fk.y * Fk.y);
        const float ri = rsqrtf(mag2);
        const float ca = (mag2 > 0.f) ? Fk.x * ri : 1.0f, sa = (mag2 > 0.f) ? Fk.y * ri : 0.0f;
        float sl, cl;
        sincos_any<true>(locv[e], sl, cl);
        const float dot = fminf(fmaxf(fmaf(cl, ca, sl * sa), -1.0f + kEps), 1.0f - kEps);
        lsum += __logf(1.0f + dot);
      }
      const float tot = group_sum<LOG2N>(fmaf(kap_row, lsum, (float)E * logc), scratch, t);
      if (valid && t == 0) p.log_prob[row] = tot;
      continue;
    }
    // F[k] and loc[k] go to this thread's own shared-memory slots so that the (large: accurate sincos, log1p, optional
    // gradient outputs) element routine runs in a rolled loop and the kernel stays inside the instruction cache
    group_sync<LOG2N>();                         // the untangle's partner reads of the exchange buffer are done
#pragma unroll
    for (int e = 0; e < E; ++e) { xch[pad16(t + e * T)] = v[e]; locs[t + e * T] = locv[e]; }
    float acc = 0.f, dk_acc = 0.f;
#pragma unroll 2
    for (int e = 0; e < E; ++e) {
      const int k = t + e * T;
      if constexpr (VM) {
        if (valid) vm_lp_element<ROWK>(p, row, prow, k, xch[pad16(k)], locs[k], kap_row, logc, dlogc, acc, dk_acc);
      } else {
        if (valid) clifford_lp_element<ROWK, FWD_ONLY>(p, row, prow, k, xch[pad16(k)], locs[k], kap_row, logc, dlogc, acc, dk_acc);
      }
    }
    const float tot = group_sum<LOG2N>(acc, scratch, t);
    float dk_tot = 0.f;
    if (!FWD_ONLY && ROWK && p.dlp_dloc) dk_tot = group_sum<LOG2N>(dk_acc, scratch, t);
    if (valid && t == 0) {
      p.log_prob[row] = tot;
      if (ROWK && p.dlp_dkappa) p.dlp_dkappa[row] = dk_tot;
    }
  }
}

// =================================================================================================
// Direct-DFT kernels for lengths the FFT engine does not cover (non power of two, d < 16,
// d > 8192).  One CTA per row (grid-stride), O(n^2) work per row; twiddles from an exact
// (index-reduced) shared-memory table.  Same element functions as the fast kernels.
// =================================================================================================
constexpr int kGenericThreads = 256;

__device__ __forceinline__ float block_sum_256(float v, float* scratch) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kGenericThreads / 32; ++i) s += scratch[i];
  return s;
}

// tw[m] = (cos(2 pi m / n), sin(2 pi m / n)), m in [0, n)
__device__ __forceinline__ void fill_twiddles(cplx* tw, int n) {
  for (int m = threadIdx.x; m < n; m += blockDim.x) {
    double s, c;
    sincospi(2.0 * (double)m / (double)n, &s, &c);
    tw[m] = make_float2((float)c, (float)s);
  }
}

// Output length n (any n >= 2), nph = (n-1)/2 free phases at bins 1..nph; DC = 1 and, for even n,
// Nyquist = 1.  For the torus n = 2d and nph = d-1.
// smem: tw[n] cplx, X[nph+1] cplx
template <int MODE, bool ROWK>
__global__ void __launch_bounds__(kGenericThreads)
clifford_fwd_generic_kernel(const CliffordFwdParams p) {
  extern __shared__ cplx smem[];
  const int n = p.n, nph = (n - 1) / 2;
  cplx* tw = smem;
  cplx* X = smem + n;
  constexpr bool PS = (MODE == kPsInjected || MODE == kPsRng);
  fill_twiddles(tw, n);
  if constexpr (MODE == kVonMisesRng)
    vm_fwd_row_entropies(p, (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);
  for (long long row = blockIdx.x; row < p.rows; row += gridDim.x) {
    const long long prow = row % p.loc_rows;
    float kap_row = 1.0f;
    if (PS) kap_row = fwd_row_kappa(p, prow);
    HalfAngle gm(kap_row + kEps);
    __syncthreads();
    const RowSrc src = global_row_src(p, row, prow);
    for (int k = 1 + threadIdx.x; k <= nph; k += blockDim.x) {
      cplx x;
      float tp_unused;
      if (!clifford_phasor<MODE, ROWK>(p, src, row, prow, k, gm, x)) x = clifford_phasor_retry<ROWK>(p, src, row, prow, k, gm, tp_unused);
      X[k] = x;
    }
    float dc = 1.0f, nyq = 1.0f;
    if (MODE == kSpectrum) {             // X_0 = 2 scale Re H_0 (so that the common factor 2 below halves it), X_d = 0
      dc = p.phase_scale * reinterpret_cast<const float2*>(src.phases)[0].x;
      nyq = 0.0f;
    }
    __syncthreads();
    const float inv_n = 1.0f / (float)n;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      double acc = 0.0;
      int m = 0;
      for (int k = 1; k <= nph; ++k) {
        m += j;
        if (m >= n) m -= n;
        const cplx w = tw[m], x = X[k];
        acc += (double)(x.x * w.x - x.y * w.y);      // Re(X_k e^{+2 pi i jk/n})
      }
      float base = (MODE == kSpectrum) ? 2.0f * dc : dc;
      if ((n & 1) == 0) base += (j & 1) ? -nyq : nyq;
      p.z[row * n + j] = inv_n * (base + 2.0f * (float)acc);
    }
    if (PS && ROWK && threadIdx.x == 0 && (p.entropy || p.kl || p.dentropy)) clifford_row_entropy(p, row, kap_row);
  }
  if (MODE == kPsRng || MODE == kUniformRng || MODE == kUnitaryRng || MODE == kVonMisesRng) rng_launch_done(p.key);
}

// smem: tw[n] cplx, g[n] float, scratch[32] float.  VM: the von Mises torus family (vm_bwd_element).
template <bool ROWK, bool VM = false>
__global__ void __launch_bounds__(kGenericThreads)
clifford_bwd_generic_kernel(const CliffordBwdParams p) {
  extern __shared__ cplx smem[];
  const int d = p.d, n = 2 * d;
  cplx* tw = smem;
  float* g = reinterpret_cast<float*>(smem + n);
  float* scratch = g + n;
  fill_twiddles(tw, n);
  for (long long row = blockIdx.x; row < p.rows; row += gridDim.x) {
    const long long prow = row % p.loc_rows;
    __syncthreads();
    for (int j = threadIdx.x; j < n; j += blockDim.x) g[j] = p.grad_z[row * n + j];
    __syncthreads();
    const float kap_raw = __ldg(p.kappa + prow * p.kappa_row_stride);
    const float kap_row = head_kappa(p.head, kap_raw);
    BetaGradRow bc(0.5f + (kap_row + kEps), 0.5f);
    float vm_b = 1.0f;
    if constexpr (VM) { if (ROWK) vm_b = vm_row_consts(kap_row).b; }
    BwdRowSrc gsrc;
    gsrc.loc = p.loc + prow * d;
    gsrc.tps = p.tp_signed ? p.tp_signed + row * d : nullptr;
    gsrc.tprime = p.tprime ? p.tprime + row * d : nullptr;
    gsrc.gnoise = p.gnoise ? p.gnoise + row * d : nullptr;
    float dk_sum = 0.f;
    for (int k = threadIdx.x; k < d; k += blockDim.x) {
      if (k == 0) {
        p.dloc[row * d] = 0.f;
        if (!ROWK) p.dkappa[row * d] = 0.f;
        continue;
      }
      double gr = 0.0, gi = 0.0;
      int m = 0;
      for (int j = 0; j < n; ++j) {            // G_k = sum_j g_j e^{-2 pi i jk/n}
        const cplx w = tw[m];
        gr += (double)(g[j] * w.x);
        gi -= (double)(g[j] * w.y);
        m += k;
        if (m >= n) m -= n;
      }
      float dk = 0.f;
      if constexpr (VM) dk = vm_bwd_element<ROWK>(p, gsrc, row, prow, k, make_float2((float)gr, (float)gi), kap_row, vm_b, 1.0f / (float)d);
      else clifford_bwd_element<ROWK>(p, gsrc, row, prow, k, make_float2((float)gr, (float)gi), bc, 1.0f / (float)d, dk);
      dk_sum += dk;
    }
    if (ROWK) {
      const float tot = block_sum_256(dk_sum, scratch);
      if (threadIdx.x == 0) p.dkappa[row] = tot * head_dkappa(p.head, kap_raw);
    }
  }
}

template <bool ROWK, bool VM = false>
__global__ void __launch_bounds__(kGenericThreads)
clifford_log_prob_generic_kernel(const CliffordLogProbParams p) {
  extern __shared__ cplx smem[];
  const int d = p.d, n = 2 * d;
  cplx* tw = smem;
  float* g = reinterpret_cast<float*>(smem + n);
  float* scratch = g + n;
  fill_twiddles(tw, n);
  for (long long row = blockIdx.x; row < p.rows; row += gridDim.x) {
    const long long prow = row % p.loc_rows;
    __syncthreads();
    for (int j = threadIdx.x; j < n; j += blockDim.x) g[j] = p.value[row * n + j];
    __syncthreads();
    const float kap_row = __ldg(p.kappa + prow * p.kappa_row_stride);
    float logc = 0.f, dlogc = 0.f;
    if constexpr (VM) {
      if (ROWK) {
        const VmRowConsts c = vm_row_consts(kap_row);
        logc = c.lnk;
        dlogc = c.b;
      }
    } else if (ROWK) {
      const PsConsts c = ps_consts((double)kap_row, 0.5);
      logc = (float)c.log_norm;
      dlogc = (float)c.dlog_norm;
    }
    float acc = 0.f, dk_acc = 0.f;
    for (int k = threadIdx.x; k < d; k += blockDim.x) {
      double fr = 0.0, fi = 0.0;
      int m = 0;
      for (int j = 0; j < n; ++j) {
        const cplx w = tw[m];
        fr += (double)(g[j] * w.x);
        fi -= (double)(g[j] * w.y);
        m += k;
        if (m >= n) m -= n;
      }
      if (k == 0) fi = 0.0;
      if constexpr (VM)
        vm_lp_element<ROWK>(p, row, prow, k, make_float2((float)fr, (float)fi), p.loc[prow * d + k], kap_row, logc, dlogc,
                            acc, dk_acc);
      else
        clifford_lp_element<ROWK>(p, row, prow, k, make_float2((float)fr, (float)fi), p.loc[prow * d + k], kap_row, logc, dlogc,
                                  acc, dk_acc);
    }
    const float tot = block_sum_256(acc, scratch);
    float dk_tot = 0.f;
    if (ROWK && p.dlp_dloc) dk_tot = block_sum_256(dk_acc, scratch);
    if (threadIdx.x == 0) {
      p.log_prob[row] = tot;
      if (ROWK && p.dlp_dkappa) p.dlp_dkappa[row] = dk_tot;
    }
  }
}

// Row entropy / KL for an arbitrary (rows, d) concentration tensor (strided): sum over k >= 1.
// One warp per row.  Also the elementwise derivative dH/dkappa when requested.
struct EntropyParams {
  const float* kappa;
  long long kappa_row_stride;
  int kappa_el_stride;
  float* entropy;      // (rows) optional
  float* kl;           // (rows) optional
  float* dentropy;     // optional; el_stride == 0: (rows) = (d-1) H'(kappa); else (rows, d) with [.,0] = 0
  long long rows;
  int d;
  double half_dm1;     // (sphere dim - 1)/2 : 0.5 for the torus circles
  int skip_first;      // 1: torus (sum over k >= 1, kl adds (d-1) ln 2 pi); 0: plain per-row PowerSpherical
  double prior_entropy;   // added to -H for kl when skip_first == 0
};

static __global__ void ps_entropy_kernel(const EntropyParams p) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < p.rows; row += nwarps) {
    const float* kr = p.kappa + row * p.kappa_row_stride;
    if (p.kappa_el_stride == 0 || !p.skip_first) {
      if (lane == 0) {
        const PsConsts c = ps_consts((double)kr[0], p.half_dm1);
        const double mult = p.skip_first ? (double)(p.d - 1) : 1.0;
        const double ent = mult * c.entropy;
        if (p.entropy) p.entropy[row] = (float)ent;
        if (p.kl) p.kl[row] = (float)((p.skip_first ? mult * 1.83787706640934548356 : p.prior_entropy) - ent);
        if (p.dentropy) p.dentropy[row] = (float)(mult * c.dentropy);
      }
    } else {
      double acc = 0.0;
      for (int k = lane; k < p.d; k += 32) {
        if (k == 0) {
          if (p.dentropy) p.dentropy[row * p.d] = 0.f;
          continue;
        }
        const PsConsts c = ps_consts((double)kr[(long long)k * p.kappa_el_stride], p.half_dm1);
        acc += c.entropy;
        if (p.dentropy) p.dentropy[row * p.d + k] = (float)c.dentropy;
      }
      acc = warp_sum(acc);
      if (lane == 0) {
        if (p.entropy) p.entropy[row] = (float)acc;
        if (p.kl) p.kl[row] = (float)((double)(p.d - 1) * 1.83787706640934548356 - acc);
      }
    }
  }
}

// One warp per row; kappa addressed like the samplers' (el_stride 0: one concentration per row).
static __global__ void vm_entropy_kernel(const EntropyParams p) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < p.rows; row += nwarps) {
    const float* kr = p.kappa + row * p.kappa_row_stride;
    if (p.kappa_el_stride == 0) {
      if (lane == 0) {
        const VmEntropy e = vm_circle_entropy(kr[0]);
        if (p.entropy) p.entropy[row] = (float)(p.d - 1) * e.h;
        if (p.dentropy) p.dentropy[row] = (float)(p.d - 1) * e.dh;
      }
    } else {
      float acc = 0.f;
      for (int k = lane; k < p.d; k += 32) {
        if (k == 0) {
          if (p.dentropy) p.dentropy[row * p.d] = 0.f;
          continue;
        }
        const VmEntropy e = vm_circle_entropy(kr[(long long)k * p.kappa_el_stride]);
        acc += e.h;
        if (p.dentropy) p.dentropy[row * p.d + k] = e.dh;
      }
      acc = warp_sum(acc);
      if (lane == 0 && p.entropy) p.entropy[row] = acc;
    }
  }
}

}  // namespace cvb
