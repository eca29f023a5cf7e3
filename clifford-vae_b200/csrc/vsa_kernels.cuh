// FFT-domain VSA kernels: bind / unbind fused as FFT(a), FFT(b) -> pointwise op -> inverse FFT in one
// kernel, one HBM round trip per vector pair (12 d bytes); plus the streaming helpers.
// Reference semantics: utils/vsa.py:43-72.
#pragma once
#include "fft_core.cuh"
#include "tma.cuh"

namespace cvb {

enum BindMode : int {
  kBindMul = 0,       // irfft(A * B)              bind (vsa.py:43-46)
  kBindMulConj = 1,   // irfft(A * conj(B))        unbind "inv"/"*" (bind with invert(b), vsa.py:56-64); bind backward
  kBindDiv = 2,       // irfft(A / (B + 1e-12))    unbind "dagger"/"deconv" (vsa.py:65-70)
  kBindDivConj = 3,   // irfft(A / conj(B + 1e-12))     d/d(ab) of the deconv unbind
  kBindNegMulConj = 4,   // -irfft(A * conj(B))         d/db of the deconv unbind (A = grad_ab, B = out)
};

struct BindParams {
  const float* a;      // row r at a + (r % a_rows) * d
  const float* b;
  float* out;          // (rows, d)
  long long rows;
  long long a_rows, b_rows;   // broadcasting: operand row = r % operand_rows
  int* sched;                 // dynamic row schedule counters (see clifford_kernels.cuh); null = static
};

__device__ __forceinline__ cplx bind_op(int mode, cplx a, cplx b) {
  if (mode == kBindMul) return cmul(a, b);
  if (mode == kBindMulConj) return cmulc(a, b);
  if (mode == kBindNegMulConj) { const cplx q = cmulc(a, b); return make_float2(-q.x, -q.y); }
  // a / (b + eps) (or its conjugated denominator): complex division
  const cplx be = make_float2(b.x + 1e-12f, mode == kBindDivConj ? -b.y : b.y);
  const float inv = 1.0f / fmaf(be.x, be.x, be.y * be.y);
  const cplx q = cmulc(a, be);
  return make_float2(q.x * inv, q.y * inv);
}

// bind_op on operands that both carry a factor 2 (A' = 2A, B' = 2B): A'B' = 4AB, A'/(B' + 2 eps) = A/(B + eps)
__device__ __forceinline__ cplx bind_op_unscaled(int mode, cplx a, cplx b) {
  if (mode == kBindMul) return cmul(a, b);
  if (mode == kBindMulConj) return cmulc(a, b);
  if (mode == kBindNegMulConj) { const cplx q = cmulc(a, b); return make_float2(-q.x, -q.y); }
  const cplx be = make_float2(b.x + 2e-12f, mode == kBindDivConj ? -b.y : b.y);
  const float inv = 1.0f / fmaf(be.x, be.x, be.y * be.y);
  const cplx q = cmulc(a, be);
  return make_float2(q.x * inv, q.y * inv);
}

// LOG2N below is log2 of the COMPLEX half length: d = 2 * 2^LOG2N.

// ---- production bind kernel ------------------------------------------------------------------------
// Z_a = FFT(a packed as N complex) is parked in shared memory, Z_b = FFT(b) stays in registers; one
// partner exchange then gives every thread Z_a[k], Z_a[N-k], Z_b[k], Z_b[N-k], from which it forms the
// real-FFT bins A, B at k and N-k, applies the pointwise op, and re-packs the Hermitian product for
// the inverse half-length FFT -- the two R2C untangles and the C2R pre-processing of the textbook
// pipeline collapse into one exchange.  Only one 16-point register array is live (<= 128 registers,
// 4 CTAs per SM for d <= 4096).  STAGED (1: a only, 2: a and b): rows arrive through cp.async.bulk (TMA) + mbarrier so the
// next row's HBM read overlaps this row's passes; otherwise plain coalesced 64-bit loads.
template <int LOG2N, int STAGED>
constexpr size_t bind_v3_smem_bytes() {
  using Pl = WideFftPlan<LOG2N>;
  return (sizeof(cplx) * (Pl::XCH + Pl::N + (STAGED == 2 ? Pl::N : 0)) + 3 * sizeof(uint64_t)) * Pl::GROUPS;
}

// Bins k and kp = N-k of the product spectrum, re-packed for the inverse half-length transform: from the parked
// Z_a (park[]), the exchanged Z_b (xch[], padded layout) and this thread's own zb = Z_b[k].  V[k] = c (s + d),
// V[N-k] = c conj(s - d).
template <int LOG2N, int MODE>
__device__ __forceinline__ void bind_pair(const cplx* park, const cplx* xch, const cplx* __restrict__ tw, int k, int kp,
                                          cplx zb, cplx& vk, cplx& vkp) {
  constexpr int N = 1 << LOG2N;
  constexpr float scale = 1.0f / (2.0f * N);
  constexpr float fold = (MODE == kBindDiv || MODE == kBindDivConj) ? scale : 0.25f * scale;
  const cplx za = park[k], zap = cconj(park[kp]);
  // self-paired bins (k = 0: DC / Nyquist, k = N/2) pair the thread's own value; only upper-half bins are exchanged
  const cplx zbp = cconj(kp == k ? zb : xch[pad16(kp)]);
  const cplx w = __ldg(&tw[twiddle_offset(LOG2N) + k]);    // exp(-2 pi i k / n)
  // bins k and N-k of the real FFTs (X[N-k] uses W^(N-k) = -conj(W^k)); factor 1/2 each
  const cplx sa = cadd(za, zap), da = cmul_mi(cmul(w, csub(za, zap)));
  const cplx sb = cadd(zb, zbp), db = cmul_mi(cmul(w, csub(zb, zbp)));
  // A = (sa +- da)/2, B = (sb +- db)/2: the halves are folded into one final constant -- the bilinear modes
  // pick up 1/4; for the quotient modes they cancel (only the 1e-12 regulariser has to be doubled to match)
  const cplx Ak = cadd(sa, da), Akp = cconj(csub(sa, da));
  const cplx Bk = cadd(sb, db), Bkp = cconj(csub(sb, db));
  const cplx Pk = bind_op_unscaled(MODE, Ak, Bk), Pkpc = cconj(bind_op_unscaled(MODE, Akp, Bkp));
  const cplx s = cadd(Pk, Pkpc), d = cmul_i(cmul(cconj(w), csub(Pk, Pkpc)));
  vk = cadd_scaled(s, d, fold);
  vkp = cconj(cscale(csub(s, d), fold));
}

// resident CTAs per SM requested for the 128-thread plans of 16 points per thread
constexpr int kBindMinBlocks = 4;
template <int LOG2N, int MODE, int STAGED>
__global__ void __launch_bounds__(WideFftPlan<LOG2N>::THREADS, (WideFftPlan<LOG2N>::THREADS <= 128 ? (WideFftPlan<LOG2N>::E > 16 ? 2 : kBindMinBlocks) : ((WideFftPlan<LOG2N>::THREADS <= 256 && WideFftPlan<LOG2N>::E <= 16) ? 2 : 1)))
bind_v3_kernel(const BindParams p, const cplx* __restrict__ tw) {
  pdl_wait_and_release();
  using Pl = WideFftPlan<LOG2N>;
  constexpr int N = Pl::N, T = Pl::T, E = Pl::E, G = Pl::GROUPS;
  constexpr uint32_t kRowBytes = 2u * N * sizeof(float);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int group = threadIdx.x / T, t = threadIdx.x % T;
  // layout: [G x park/stage_a][G x stage_b (STAGED)][G x xch][G x 2 mbarriers]
  cplx* park = reinterpret_cast<cplx*>(smem_raw) + (size_t)group * N;
  cplx* stage_b = reinterpret_cast<cplx*>(smem_raw) + (size_t)(G + group) * N;
  cplx* xch = reinterpret_cast<cplx*>(smem_raw) + (size_t)(STAGED == 2 ? 2 : 1) * G * N + (size_t)group * Pl::XCH;
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<cplx*>(smem_raw) + (size_t)(STAGED == 2 ? 2 : 1) * G * N + (size_t)G * Pl::XCH) + 3 * group;
  int* next_slot = reinterpret_cast<int*>(&bars[2]);
  const long long stride = (long long)gridDim.x * G;
  const long long row0 = (long long)blockIdx.x * G + group;
  constexpr float scale = 1.0f / (2.0f * N);
  const bool dynamic = (T >= 32) && p.sched != nullptr;

  if (STAGED) {
    if (t == 0) {
      mbar_init(&bars[0], 1);
      mbar_init(&bars[1], 1);
      mbar_init_fence();
    }
    __syncthreads();
    if (t == 0 && row0 < p.rows) {
      mbar_expect_tx(&bars[0], kRowBytes);
      tma_load_1d(park, p.a + (row0 % p.a_rows) * (2LL * N), kRowBytes, &bars[0]);
      if (STAGED == 2) {
        mbar_expect_tx(&bars[1], kRowBytes);
        tma_load_1d(stage_b, p.b + (row0 % p.b_rows) * (2LL * N), kRowBytes, &bars[1]);
      }
    }
  }

  uint32_t parity = 0;
  long long row = row0;
  const long long loop_end = dynamic ? p.rows : p.rows + (long long)group;    // static: trip counts uniform over the CTA
  for (; row < loop_end; parity ^= 1u) {
    const bool valid = row < p.rows;
    if (dynamic && t == 0) *next_slot = atomicAdd(p.sched, 1);
    cplx v[E];
    // ---- a -> Z_a, parked
    if (STAGED) {
      if (valid) mbar_wait(&bars[0], parity);
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = valid ? park[t + e * T] : make_float2(0.f, 0.f);
    } else {
      const float2* ar = reinterpret_cast<const float2*>(p.a + (valid ? row % p.a_rows : 0) * (2LL * N));
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = valid ? ldg_stream2(ar + t + e * T) : make_float2(0.f, 0.f);
    }
    fft_run_p<Pl, false>(v, xch, t, tw);      // (STAGED: its barriers order every thread's stage read before the park write)
    const long long next_row = dynamic ? (long long)*next_slot + stride : row + stride;   // visible after the barriers above
    const bool next_valid = next_row < p.rows;
#pragma unroll
    for (int e = 0; e < E; ++e) park[t + e * T] = v[e];
    // ---- b -> Z_b in registers
    if (STAGED == 2) {
      if (valid) mbar_wait(&bars[1], parity);
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = valid ? stage_b[t + e * T] : make_float2(1.f, 0.f);
    } else {
      const float2* br = reinterpret_cast<const float2*>(p.b + (valid ? row % p.b_rows : 0) * (2LL * N));
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = valid ? ldg_stream2(br + t + e * T) : make_float2(1.f, 0.f);
    }
    fft_run_p<Pl, false>(v, xch, t, tw);
    if (STAGED == 2 && t == 0 && next_valid) {   // every thread has read stage_b (barriers inside fft_run)
      mbar_expect_tx(&bars[1], kRowBytes);
      tma_load_1d(stage_b, p.b + (next_row % p.b_rows) * (2LL * N), kRowBytes, &bars[1]);
    }
    // ---- one partner exchange: untangle a and b, pointwise op, re-pack for the inverse transform.
    // Bins k and N-k share every intermediate (V[k] = c (s + d), V[N-k] = c conj(s - d)), so each pair is formed ONCE,
    // by the thread that owns k < N/2 (its points e < E/2); the partner value V[N-k] goes back through the parked row
    // (the slot this thread just consumed), and every thread re-reads its upper-half points after one barrier.
    group_sync_p<Pl>();
#pragma unroll
    for (int e = E / 2; e < E; ++e) xch[pad16(t + e * T)] = v[e];      // partners only ever read bins > N/2
    group_sync_p<Pl>();
    auto pair = [&](int k, int kp, cplx zb, cplx& vk, cplx& vkp) { bind_pair<LOG2N, MODE>(park, xch, tw, k, kp, zb, vk, vkp); };
#pragma unroll
    for (int e = 0; e < E / 2; ++e) {
      const int k = t + e * T, kp = (N - k) & (N - 1);
      cplx vkp;
      pair(k, kp, v[e], v[e], vkp);
      if (kp != k) park[kp] = vkp;               // k = 0 pairs the DC / Nyquist bins inside one slot
    }
    if (t == 0) {                                // k = N/2 is its own partner
      cplx vk, vkp;
      pair(N / 2, N / 2, v[E / 2], vk, vkp);
      park[N / 2] = vk;
    }
    group_sync_p<Pl>();
#pragma unroll
    for (int e = E / 2; e < E; ++e) v[e] = park[t + e * T];
    if (STAGED) {
      fence_proxy_async();                       // parked-spectrum accesses before the next TMA write
      group_sync_p<Pl>();
      if (t == 0 && next_valid) {
        mbar_expect_tx(&bars[0], kRowBytes);
        tma_load_1d(park, p.a + (next_row % p.a_rows) * (2LL * N), kRowBytes, &bars[0]);
      }
    }
    fft_run_p<Pl, true>(v, xch, t, tw);        // begins with a barrier: partner reads are complete
    if (valid) {
      float2* o = reinterpret_cast<float2*>(p.out + row * (2LL * N));
#pragma unroll
      for (int e = 0; e < E; ++e) stg_stream2(o + t + e * T, v[e]);
    }
    row = next_row;
  }
  if (dynamic && t == 0) {
    if (atomicAdd(p.sched + 1, 1) == (int)stride - 1) { p.sched[0] = 0; p.sched[1] = 0; }
  }
}

// ---- any-length bind / unbind("inv") through the power-of-two kernel's machinery -----------------------------------
// A circular convolution of length n is the linear convolution folded once: out[i] = c[i] + c[i + n], c = a * b zero-
// padded to M >= 2n (power of two); the circular correlation of unbind("inv") folds the negative lags,
// out[i] = c[i] + c[M + i - n].  Rows of any length n (odd, 513, 144, 484 ... -- the reference's PowerSpherical / vMF
// latents and heat-map dimensions) therefore cost one pass of the fused FFT pipeline at M instead of an O(n^2) direct
// DFT.  Rows are only 4-byte aligned: scalar coalesced loads / stores.  LOG2N = log2(M / 2).
template <int LOG2N>
constexpr size_t bind_pad_smem_bytes() {
  using Pl = WideFftPlan<LOG2N>;
  return sizeof(cplx) * (Pl::XCH + Pl::N) * Pl::GROUPS;
}

template <int LOG2N, int MODE>
__global__ void __launch_bounds__(WideFftPlan<LOG2N>::THREADS, (WideFftPlan<LOG2N>::THREADS <= 128 ? (WideFftPlan<LOG2N>::E > 16 ? 2 : 4) : ((WideFftPlan<LOG2N>::THREADS <= 256 && WideFftPlan<LOG2N>::E <= 16) ? 2 : 1)))
bind_pad_kernel(const BindParams p, int n, const cplx* __restrict__ tw) {
  using Pl = WideFftPlan<LOG2N>;
  constexpr int N = Pl::N, T = Pl::T, E = Pl::E, G = Pl::GROUPS, M = 2 * N;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int group = threadIdx.x / T, t = threadIdx.x % T;
  cplx* park = reinterpret_cast<cplx*>(smem_raw) + (size_t)group * N;
  cplx* xch = reinterpret_cast<cplx*>(smem_raw) + (size_t)G * N + (size_t)group * Pl::XCH;
  const long long stride = (long long)gridDim.x * G;
  for (long long base = (long long)blockIdx.x * G; base < p.rows; base += stride) {   // trip counts uniform over the CTA
    const long long row = base + group;
    const bool valid = row < p.rows;
    cplx v[E];
    auto load_padded = [&](const float* src) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int i0 = 2 * (t + e * T);
        v[e] = make_float2((valid && i0 < n) ? ldg_stream1(src + i0) : 0.0f, (valid && i0 + 1 < n) ? ldg_stream1(src + i0 + 1) : 0.0f);
      }
    };
    load_padded(p.a + (valid ? row % p.a_rows : 0) * (long long)n);
    fft_run_p<Pl, false>(v, xch, t, tw);
#pragma unroll
    for (int e = 0; e < E; ++e) park[t + e * T] = v[e];
    load_padded(p.b + (valid ? row % p.b_rows : 0) * (long long)n);
    fft_run_p<Pl, false>(v, xch, t, tw);
    group_sync_p<Pl>();
#pragma unroll
    for (int e = E / 2; e < E; ++e) xch[pad16(t + e * T)] = v[e];
    group_sync_p<Pl>();
#pragma unroll
    for (int e = 0; e < E / 2; ++e) {
      const int k = t + e * T, kp = (N - k) & (N - 1);
      cplx vkp;
      bind_pair<LOG2N, MODE>(park, xch, tw, k, kp, v[e], v[e], vkp);
      if (kp != k) park[kp] = vkp;
    }
    if (t == 0) {
      cplx vk, vkp;
      bind_pair<LOG2N, MODE>(park, xch, tw, N / 2, N / 2, v[E / 2], vk, vkp);
      park[N / 2] = vk;
    }
    group_sync_p<Pl>();
#pragma unroll
    for (int e = E / 2; e < E; ++e) v[e] = park[t + e * T];
    fft_run_p<Pl, true>(v, xch, t, tw);
    // fold: the M real samples c[2m], c[2m+1] go to the parked buffer (as floats), then out[i] = c[i] + c[partner(i)]
    group_sync_p<Pl>();
#pragma unroll
    for (int e = 0; e < E; ++e) park[t + e * T] = v[e];
    group_sync_p<Pl>();
    if (valid) {
      const float* c = reinterpret_cast<const float*>(park);
      float* o = p.out + row * (long long)n;
      for (int i = t; i < n; i += T) {
        const int j = (MODE == kBindMul) ? i + n : M + i - n;
        stg_stream1(o + i, c[i] + c[j]);          // (the NegMulConj sign is already in the product spectrum)
      }
    }
    group_sync_p<Pl>();            // the parked samples are consumed before the next row parks its spectrum
  }
}

// ---- fused binding-depth chain (BASELINE config 5) --------------------------------------------------
// reference scripts/binding_depth_heatmap.py:25-35: bound = x0 (*) y1 (*) ... (*) ym, then unbind ym ... y1
// with the "inv" method, then cos(recovered, x0).  In the frequency domain the chain is X0 * prod_j |Y_j|^2,
// and by Parseval the cosine needs no inverse transform:
//     cos = sum_k w_k |X0_k|^2 P_k / sqrt(sum_k w_k |X0_k|^2 P_k^2 * sum_k w_k |X0_k|^2),   P_k = prod_j |Y_jk|^2,
// with Hermitian weights w_k = 1 for k in {0, N}, 2 otherwise.  One trial = (m+1) forward half-length FFTs,
// 4 d (m+1) bytes read and 4 bytes written, instead of 2m fused bind launches (24 m d bytes).
template <int LOG2N>
__global__ void __launch_bounds__(FftPlan<LOG2N>::THREADS, (FftPlan<LOG2N>::THREADS <= 128 ? 4 : (FftPlan<LOG2N>::THREADS <= 256 ? 2 : 1)))
depth_chain_kernel(const float* __restrict__ vecs, float* __restrict__ out, long long trials, int mp1,
                   const cplx* __restrict__ tw) {
  using Pl = FftPlan<LOG2N>;
  constexpr int N = Pl::N, T = Pl::T, E = Pl::E, G = Pl::GROUPS;
  extern __shared__ cplx smem[];
  const int group = threadIdx.x / T, t = threadIdx.x % T;
  cplx* xch = smem + group * Pl::XCH;
  float* scratch = reinterpret_cast<float*>(smem + G * Pl::XCH) + group * 32;
  for (long long base = (long long)blockIdx.x * G; base < trials; base += (long long)gridDim.x * G) {
    const long long trial = base + group;
    const bool valid = trial < trials;
    float x2[E], P[E];            // |X0_k|^2 and the running product for this thread's bins
    float x2_nyq = 0.f, P_nyq = 1.f;
#pragma unroll
    for (int e = 0; e < E; ++e) { x2[e] = 0.f; P[e] = 1.f; }
    for (int j = 0; j < mp1; ++j) {
      const float2* r = reinterpret_cast<const float2*>(vecs + ((valid ? trial : 0) * mp1 + j) * (2LL * N));
      cplx v[E];
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = valid ? ldg_stream2(r + t + e * T) : make_float2(0.f, 0.f);
      fft_run<LOG2N, false>(v, xch, t, tw);
      const float nyq = r2c_untangle<LOG2N>(v, xch, t, tw);
      if (j == 0) {
#pragma unroll
        for (int e = 0; e < E; ++e) x2[e] = fmaf(v[e].x, v[e].x, v[e].y * v[e].y);
        x2_nyq = nyq * nyq;
      } else {
#pragma unroll
        for (int e = 0; e < E; ++e) P[e] *= fmaf(v[e].x, v[e].x, v[e].y * v[e].y);
        P_nyq *= nyq * nyq;
      }
    }
    float num = 0.f, rr = 0.f, xx = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const float w = (t + e * T == 0) ? 1.0f : 2.0f;
      const float a = w * x2[e] * P[e];
      num += a; rr += a * P[e]; xx += w * x2[e];
    }
    if (t == 0) { const float a = x2_nyq * P_nyq; num += a; rr += a * P_nyq; xx += x2_nyq; }
    num = group_sum<LOG2N>(num, scratch, t);
    rr = group_sum<LOG2N>(rr, scratch, t);
    xx = group_sum<LOG2N>(xx, scratch, t);
    if (valid && t == 0) {
      // time-domain norms are sqrt(sum / n); the 1/n cancels; clamp like F.cosine_similarity (eps 1e-8 on each norm)
      const float inv_n = 1.0f / (2.0f * N);
      const float nr = fmaxf(sqrtf(rr * inv_n), 1e-8f), nx = fmaxf(sqrtf(xx * inv_n), 1e-8f);
      out[trial] = (num * inv_n) / (nr * nx);
    }
  }
}

// ---- any-length bind (direct DFT, O(d^2) per pair): covers odd / non power-of-two d -----------
// smem: tw[d] cplx, a[d], b[d] float, P[d/2+1] cplx
template <int MODE>
__global__ void __launch_bounds__(256)
bind_generic_kernel(const BindParams p, int d) {
  extern __shared__ cplx smem[];
  cplx* tw = smem;
  float* sa = reinterpret_cast<float*>(smem + d);
  float* sb = sa + d;
  cplx* P = reinterpret_cast<cplx*>(sb + d);   // 4d floats from the base: 8-byte aligned for any d
  const int nh = d / 2;                     // bins 0..nh
  for (int m = threadIdx.x; m < d; m += blockDim.x) {
    double s, c;
    sincospi(2.0 * (double)m / (double)d, &s, &c);
    tw[m] = make_float2((float)c, (float)s);
  }
  for (long long row = blockIdx.x; row < p.rows; row += gridDim.x) {
    const float* ar = p.a + (row % p.a_rows) * (long long)d;
    const float* br = p.b + (row % p.b_rows) * (long long)d;
    __syncthreads();
    for (int j = threadIdx.x; j < d; j += blockDim.x) { sa[j] = ar[j]; sb[j] = br[j]; }
    __syncthreads();
    for (int k = threadIdx.x; k <= nh; k += blockDim.x) {
      double are = 0, aim = 0, bre = 0, bim = 0;
      int m = 0;
      for (int j = 0; j < d; ++j) {
        const cplx w = tw[m];
        are += (double)(sa[j] * w.x); aim -= (double)(sa[j] * w.y);
        bre += (double)(sb[j] * w.x); bim -= (double)(sb[j] * w.y);
        m += k;
        if (m >= d) m -= d;
      }
      if (k == 0 || 2 * k == d) { aim = 0; bim = 0; }
      P[k] = bind_op(MODE, make_float2((float)are, (float)aim), make_float2((float)bre, (float)bim));
    }
    __syncthreads();
    const float inv_d = 1.0f / (float)d;
    const int kmax = (d - 1) / 2;
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
      double acc = 0.0;
      int m = 0;
      for (int k = 1; k <= kmax; ++k) {
        m += j;
        if (m >= d) m -= d;
        const cplx w = tw[m], x = P[k];
        acc += (double)(x.x * w.x - x.y * w.y);
      }
      float base = P[0].x;
      if ((d & 1) == 0) base += (j & 1) ? -P[nh].x : P[nh].x;
      p.out[row * (long long)d + j] = inv_d * (base + 2.0f * (float)acc);
    }
  }
}

// ---- short vectors of any length (d <= 256): a TILE of RT pairs per CTA ----------------------------------------------
// The reference's default MNIST latents are bound / unbound at d = 2 z_dim (Clifford: 4 .. 80) or z_dim + 1 (vMF:
// 3 .. 41) (mnist/mnist_clifpws.py:235-236,713-719); one 256-thread CTA per pair (bind_generic_kernel) idles most of its
// threads there.  Same scheme as clifford_small.cuh: operands parked as g[j][r], one (4 pairs, bin k) item per thread
// for the two forward real DFTs (packed FMAs, exact index-reduced twiddles, 128-bit broadcast loads), the pointwise op,
// then one (4 pairs, output j) item per thread for the inverse, outputs j and d - j together (shared cos, negated sin).
// fp32 accumulation (<= 256 terms).
constexpr int kBindSmallMaxD = 256;
constexpr int kBindSmallThreads = 128;
inline size_t bind_small_smem(int d, int rt) {
  return sizeof(cplx) * (size_t)((d + 1) & ~1) + 2 * sizeof(float) * (size_t)d * (rt + 4) + sizeof(cplx) * (size_t)(d / 2 + 1) * (rt + 2);
}
template <int MODE>
__global__ void __launch_bounds__(kBindSmallThreads)
bind_small_kernel(const BindParams p, const int d, const int RT) {
  extern __shared__ __align__(16) unsigned char smem_bs[];
  const int GP = RT + 4, XP = RT + 2, nh = d / 2, kmax = (d - 1) / 2;
  cplx* tw = reinterpret_cast<cplx*>(smem_bs);
  float* ga = reinterpret_cast<float*>(tw + ((d + 1) & ~1));
  float* gb = ga + (size_t)d * GP;
  cplx* P = reinterpret_cast<cplx*>(gb + (size_t)d * GP);
  for (int m = threadIdx.x; m < d; m += blockDim.x) {
    double sn, cs;
    sincospi(2.0 * (double)m / (double)d, &sn, &cs);
    tw[m] = make_float2((float)cs, (float)sn);
  }
  const long long tiles = (p.rows + RT - 1) / RT;
  const float inv_d = 1.0f / (float)d;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long row0 = tile * RT;
    __syncthreads();
    for (int i = threadIdx.x; i < RT * d; i += kBindSmallThreads) {
      const int r = i / d, j = i - r * d;
      const long long row = row0 + r;
      const bool in = row < p.rows;
      ga[j * GP + r] = in ? __ldg(p.a + (row % p.a_rows) * (long long)d + j) : 0.0f;
      gb[j * GP + r] = in ? __ldg(p.b + (row % p.b_rows) * (long long)d + j) : 0.0f;
    }
    __syncthreads();
    // forward: A_k, B_k = sum_j x_j e^{-2 pi i jk/d}, k = 0 .. d/2, then the pointwise op
    for (int i = threadIdx.x; i < (RT / 4) * (nh + 1); i += kBindSmallThreads) {
      const int q = i / (nh + 1), k = i - q * (nh + 1);
      float2 aa[4], bb[4];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) { aa[rr] = make_float2(0.f, 0.f); bb[rr] = make_float2(0.f, 0.f); }
      int m = 0;
      for (int j = 0; j < d; ++j) {
        const cplx w = make_float2(tw[m].x, -tw[m].y);
        const float4 a4 = *reinterpret_cast<const float4*>(ga + j * GP + 4 * q);
        const float4 b4 = *reinterpret_cast<const float4*>(gb + j * GP + 4 * q);
        aa[0] = __ffma2_rn(make_float2(a4.x, a4.x), w, aa[0]); bb[0] = __ffma2_rn(make_float2(b4.x, b4.x), w, bb[0]);
        aa[1] = __ffma2_rn(make_float2(a4.y, a4.y), w, aa[1]); bb[1] = __ffma2_rn(make_float2(b4.y, b4.y), w, bb[1]);
        aa[2] = __ffma2_rn(make_float2(a4.z, a4.z), w, aa[2]); bb[2] = __ffma2_rn(make_float2(b4.z, b4.z), w, bb[2]);
        aa[3] = __ffma2_rn(make_float2(a4.w, a4.w), w, aa[3]); bb[3] = __ffma2_rn(make_float2(b4.w, b4.w), w, bb[3]);
        m += k;
        if (m >= d) m -= d;
      }
      const bool real_bin = (k == 0) || (2 * k == d);
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        if (real_bin) { aa[rr].y = 0.f; bb[rr].y = 0.f; }
        P[k * XP + 4 * q + rr] = bind_op(MODE, aa[rr], bb[rr]);
      }
    }
    __syncthreads();
    // inverse: out_j = (1/d) (P_0 + (-1)^j P_{d/2} + 2 sum_k (Re P_k cos(2 pi jk/d) - Im P_k sin(2 pi jk/d))); out_{d-j}: + Im P_k sin
    for (int i = threadIdx.x; i < (RT / 4) * (nh + 1); i += kBindSmallThreads) {
      const int q = i / (nh + 1), j = i - q * (nh + 1);
      float2 acc[4];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) acc[rr] = make_float2(0.f, 0.f);
      int m = 0;
      const cplx* pq = P + 4 * q;
      for (int k = 1; k <= kmax; ++k) {
        m += j;
        if (m >= d) m -= d;
        const cplx w = tw[m];
        const float4 x01 = *reinterpret_cast<const float4*>(pq + k * XP);
        const float4 x23 = *reinterpret_cast<const float4*>(pq + k * XP + 2);
        acc[0] = __ffma2_rn(make_float2(x01.x, x01.y), w, acc[0]);
        acc[1] = __ffma2_rn(make_float2(x01.z, x01.w), w, acc[1]);
        acc[2] = __ffma2_rn(make_float2(x23.x, x23.y), w, acc[2]);
        acc[3] = __ffma2_rn(make_float2(x23.z, x23.w), w, acc[3]);
      }
      const bool mirror = (j != 0) && (2 * j != d);
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const long long row = row0 + 4 * q + rr;
        if (row < p.rows) {
          float base = pq[rr].x;
          if ((d & 1) == 0) base += (j & 1) ? -pq[nh * XP + rr].x : pq[nh * XP + rr].x;
          p.out[row * (long long)d + j] = inv_d * (base + 2.0f * (acc[rr].x - acc[rr].y));
          if (mirror) p.out[row * (long long)d + (d - j)] = inv_d * (base + 2.0f * (acc[rr].x + acc[rr].y));
        }
      }
    }
  }
}

// ---- elementwise / reduction VSA helpers --------------------------------------------------------
// invert (vsa.py:49-53): out[r, j] = a[r, (d - j) mod d]
// one warp per row: no per-element 64-bit division
static __global__ void __launch_bounds__(256)
invert_kernel(const float* __restrict__ a, float* __restrict__ out, long long rows, int d) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < rows; row += nwarps) {
    const float* ar = a + row * (long long)d;
    float* orow = out + row * (long long)d;
#pragma unroll 4
    for (int j = lane; j < d; j += 32) stg_stream1(orow + j, ldg_stream1(ar + (j == 0 ? 0 : d - j)));
  }
}

// permute (vsa.py:82-84): out[r, j] = v[r, perm[j]];  unpermute (:87-90): out[r, perm[j]] = v[r, j]
static __global__ void permute_kernel(const float* __restrict__ v, const long long* __restrict__ perm, float* __restrict__ out,
                               long long rows, int d, int inverse) {
  // one CTA per row: the 256 threads gather from the same (L1-resident) row; no per-element 64-bit division
  for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
    const float* vr = v + row * (long long)d;
    float* orow = out + row * (long long)d;
#pragma unroll 4
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
      const int pj = (int)__ldg(perm + j);
      if (inverse) orow[pj] = vr[j];
      else orow[j] = vr[pj];
    }
  }
}

// bundle (vsa.py:75-79), stage 1: partial column sums of a (k, d) stack over row chunks.
// grid = (ceil(d / 128), chunks); partial[(chunk, j)].
static __global__ void __launch_bounds__(128)
bundle_partial_kernel(const float* __restrict__ v, float* __restrict__ partial, long long k, int d,
                      long long rows_per_chunk) {
  const int j = blockIdx.x * 128 + threadIdx.x;
  const long long r0 = (long long)blockIdx.y * rows_per_chunk;
  long long r1 = r0 + rows_per_chunk;
  if (r1 > k) r1 = k;
  if (j >= d) return;
  float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
  long long r = r0;
  for (; r + 3 < r1; r += 4) {
    acc0 += ldg_stream1(v + r * d + j);
    acc1 += ldg_stream1(v + (r + 1) * d + j);
    acc2 += ldg_stream1(v + (r + 2) * d + j);
    acc3 += ldg_stream1(v + (r + 3) * d + j);
  }
  for (; r < r1; ++r) acc0 += ldg_stream1(v + r * d + j);
  partial[(long long)blockIdx.y * d + j] = (acc0 + acc1) + (acc2 + acc3);
}
// stage 2: out[j] = scale * sum_chunks partial
static __global__ void bundle_final_kernel(const float* __restrict__ partial, float* __restrict__ out, int chunks, int d,
                                    float scale) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d) return;
  float acc = 0.f;
  for (int c = 0; c < chunks; ++c) acc += partial[(long long)c * d + j];
  out[j] = acc * scale;
}

// similarity (vsa.py:93-96): cosine with each norm clamped at 1e-8.  One warp per output row;
// operand row = r % operand_rows (broadcast).  Optional backward outputs handled by cosine_bwd_kernel.
static __global__ void __launch_bounds__(256)
cosine_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long rows,
              long long a_rows, long long b_rows, int d) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < rows; row += nwarps) {
    const float* ar = a + (row % a_rows) * (long long)d;
    const float* br = b + (row % b_rows) * (long long)d;
    float ab = 0.f, aa = 0.f, bb = 0.f;
    if ((d & 3) == 0) {
      const float4* a4 = reinterpret_cast<const float4*>(ar);
      const float4* b4 = reinterpret_cast<const float4*>(br);
#pragma unroll 4
      for (int i = lane; i < d / 4; i += 32) {
        const float4 x = __ldg(a4 + i), y = __ldg(b4 + i);
        ab += x.x * y.x + x.y * y.y + x.z * y.z + x.w * y.w;
        aa += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
        bb += y.x * y.x + y.y * y.y + y.z * y.z + y.w * y.w;
      }
    } else {
      for (int i = lane; i < d; i += 32) {
        const float x = ar[i], y = br[i];
        ab += x * y; aa += x * x; bb += y * y;
      }
    }
    ab = warp_sum(ab); aa = warp_sum(aa); bb = warp_sum(bb);
    if (lane == 0) out[row] = ab / (fmaxf(sqrtf(aa), 1e-8f) * fmaxf(sqrtf(bb), 1e-8f));
  }
}

// d cos / d a = g (b / (|a||b|) - cos a / |a|^2), same for b; per expanded row (caller reduces broadcasts)
static __global__ void __launch_bounds__(256)
cosine_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ gout,
                  float* __restrict__ da, float* __restrict__ db, long long rows, long long a_rows, long long b_rows,
                  int d) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < rows; row += nwarps) {
    const float* ar = a + (row % a_rows) * (long long)d;
    const float* br = b + (row % b_rows) * (long long)d;
    float ab = 0.f, aa = 0.f, bb = 0.f;
    for (int i = lane; i < d; i += 32) {
      const float x = ar[i], y = br[i];
      ab += x * y; aa += x * x; bb += y * y;
    }
    ab = warp_sum(ab); aa = warp_sum(aa); bb = warp_sum(bb);
    const float na = sqrtf(aa), nb = sqrtf(bb);
    const float ca = fmaxf(na, 1e-8f), cb = fmaxf(nb, 1e-8f);
    const float g = gout[row];
    const float inv = 1.0f / (ca * cb);
    const float cosv = ab * inv;
    // derivative of the clamped norms: d max(|a|, eps) / da = a/|a| when |a| > eps else 0
    const float ka = (na > 1e-8f) ? cosv / (ca * na) : 0.f;
    const float kb = (nb > 1e-8f) ? cosv / (cb * nb) : 0.f;
    for (int i = lane; i < d; i += 32) {
      const float x = ar[i], y = br[i];
      if (da) da[row * (long long)d + i] = g * (y * inv - ka * x);
      if (db) db[row * (long long)d + i] = g * (x * inv - kb * y);
    }
  }
}

// normalize_vectors (vsa.py:39-40): x / max(||x||, 1e-12); backward dx = (g - y (y.g)) / max(||x||, eps)
static __global__ void __launch_bounds__(256)
normalize_kernel(const float* __restrict__ x, float* __restrict__ out, long long rows, int d, int vec4) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < rows; row += nwarps) {
    const float* xr = x + row * (long long)d;
    float* orow = out + row * (long long)d;
    float ss = 0.f;
    if (vec4) {
      // rows are 16-byte aligned and d % 4 == 0: 128-bit accesses (the second pass hits L1 / L2)
      const float4* x4 = reinterpret_cast<const float4*>(xr);
      float4* o4 = reinterpret_cast<float4*>(orow);
      const int d4 = d >> 2;
#pragma unroll 4
      for (int i = lane; i < d4; i += 32) { const float4 v = x4[i]; ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w; }
      ss = warp_sum(ss);
      const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
#pragma unroll 4
      for (int i = lane; i < d4; i += 32) { const float4 v = x4[i]; o4[i] = make_float4(v.x * inv, v.y * inv, v.z * inv, v.w * inv); }
      continue;
    }
    for (int i = lane; i < d; i += 32) { const float v = xr[i]; ss += v * v; }
    ss = warp_sum(ss);
    const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
    for (int i = lane; i < d; i += 32) orow[i] = xr[i] * inv;
  }
}
static __global__ void __launch_bounds__(256)
normalize_bwd_kernel(const float* __restrict__ x, const float* __restrict__ gout, float* __restrict__ dx,
                     long long rows, int d) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < rows; row += nwarps) {
    const float* xr = x + row * (long long)d;
    const float* gr = gout + row * (long long)d;
    float ss = 0.f, xg = 0.f;
    for (int i = lane; i < d; i += 32) { const float v = xr[i]; ss += v * v; xg += v * gr[i]; }
    ss = warp_sum(ss); xg = warp_sum(xg);
    const float nrm = sqrtf(ss);
    const float inv = 1.0f / fmaxf(nrm, 1e-12f);
    const float k = (nrm > 1e-12f) ? xg * inv * inv * inv : 0.f;     // (y.g)/max(|x|) * 1/|x|
    for (int i = lane; i < d; i += 32) dx[row * (long long)d + i] = gr[i] * inv - k * xr[i];
  }
}

}  // namespace cvb
