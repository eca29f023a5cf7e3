// Clifford-torus kernels for SHORT rows of any length: n = output length <= 512 (d <= 256 circles), power of two or not.
// This is where the reference's default MNIST latents live (d in {2, 5, 10, 20, 40}, mnist/mnist_clifpws.py:713-719)
// and the per-token latents of cnn/cliffordar_model.py (D = 16).  At these sizes an FFT has nothing to factor and one
// row cannot fill a CTA, so the direct-DFT kernels of clifford_kernels.cuh (one 256-thread CTA per row) idle most of
// their threads.  Here a CTA owns a TILE of RT rows (RT = 4 .. 32, chosen by the launcher from the batch size):
//
//   forward   phase 1: one (row, bin) item per thread -> phasor (same element functions and Philox indexing as the other
//                      kernels) -> X[bin][row] in shared memory
//             phase 2: one (4 rows, output j) item per thread: the length-(d-1) real DFT sums for outputs j AND n-j
//                      (they share cos, negate sin) as packed FMAs (c_k cos, s_k sin), twiddles from an exact
//                      index-reduced table, the four rows' bins by two 128-bit broadcast loads
//   backward  G_k = sum_j g_j e^{-2 pi i jk/n} the same way (4 rows per item), then the shared element routine
//   log_prob  F_k likewise, then the shared element routine.
//
// fp32 accumulation: the sums have <= 511 terms (the long-row direct-DFT kernels keep fp64).  Power-of-two d >= 16 never
// comes here (the FFT engine is faster from d = 16 up); the tile shrinks with n so that a CTA stays within 48 KB.
#pragma once
#include "clifford_kernels.cuh"

namespace cvb {

constexpr int kSmallMaxN = 512;
constexpr int kSmallThreads = 128;
constexpr int kSmallMaxRows = 32;

__host__ __device__ __forceinline__ constexpr int small_pitch_c(int rt) { return rt + 2; }   // complex pitch: 16-byte aligned rows of 4
__host__ __device__ __forceinline__ constexpr int small_pitch_f(int rt) { return rt + 4; }   // float pitch:   16-byte aligned rows of 4

// rows per tile: as large as keeps >= 2 tiles per SM in flight (small batches stay spread over the SMs) and the tile's
// shared memory (smem_of(rt)) within 48 KB
template <class SmemOf>
inline int small_rows_per_tile(long long rows, int sms, SmemOf smem_of) {
  int rt = kSmallMaxRows;
  while (rt > 4 && ((rows + rt - 1) / rt < 2LL * sms || smem_of(rt) > 48 * 1024)) rt >>= 1;
  return rt;
}

inline size_t clifford_fwd_small_smem(int n, int rt) {
  const int nph = (n - 1) / 2;
  return sizeof(cplx) * (size_t)((n + 1) & ~1) + sizeof(cplx) * (size_t)(nph + 1) * small_pitch_c(rt);
}

template <int MODE, bool ROWK>
__global__ void __launch_bounds__(kSmallThreads)
clifford_fwd_small_kernel(const CliffordFwdParams p, const int RT) {
  extern __shared__ __align__(16) unsigned char smem_small[];
  const int n = p.n, nph = (n - 1) / 2, J = n / 2 + 1;       // outputs j = 0 .. floor(n/2) (and their mirrors n - j)
  const int XP = small_pitch_c(RT);
  cplx* tw = reinterpret_cast<cplx*>(smem_small);
  cplx* X = tw + ((n + 1) & ~1);                             // [k = 0 .. nph][r]; slot k = 0 holds (dc, nyquist)
  constexpr bool PS = (MODE == kPsInjected || MODE == kPsRng);
  fill_twiddles(tw, n);
  if constexpr (MODE == kVonMisesRng)
    vm_fwd_row_entropies(p, (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);
  const long long tiles = (p.rows + RT - 1) / RT;
  const float inv_n = 1.0f / (float)n;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long row0 = tile * RT;
    __syncthreads();                                         // twiddles visible / the previous tile's readers are done
    // phase 1: phasors.  Items (r, k) with k fastest: injected draws and loc are read coalesced along the row.
    for (int i = threadIdx.x; i < RT * (nph + 1); i += kSmallThreads) {
      const int r = i / (nph + 1), k = i - r * (nph + 1);
      const long long row = row0 + r;
      cplx x = make_float2(0.f, 0.f);
      if (row < p.rows) {
        const long long prow = row % p.loc_rows;
        const RowSrc src = global_row_src(p, row, prow);
        if (k == 0) {
          x = make_float2(1.0f, 1.0f);
          if (MODE == kSpectrum) x = make_float2(p.phase_scale * reinterpret_cast<const float2*>(src.phases)[0].x, 0.0f);
        } else {
          float kap_row = 1.0f;
          if (PS) kap_row = fwd_row_kappa(p, prow);
          HalfAngle gm(kap_row + kEps);
          float tp_unused;
          if (!clifford_phasor<MODE, ROWK>(p, src, row, prow, k, gm, x)) x = clifford_phasor_retry<ROWK>(p, src, row, prow, k, gm, tp_unused);
        }
      }
      X[k * XP + r] = x;
    }
    if (PS && ROWK && (p.entropy || p.kl || p.dentropy)) {
      for (int r = threadIdx.x; r < RT; r += kSmallThreads)
        if (row0 + r < p.rows) clifford_row_entropy(p, row0 + r, fwd_row_kappa(p, (row0 + r) % p.loc_rows));
    }
    __syncthreads();
    // phase 2: z_j = (1/n) (dc + (-1)^j nyq + 2 sum_k (c_k cos(2 pi jk/n) - s_k sin(2 pi jk/n))), z_{n-j} with + s_k sin
    for (int i = threadIdx.x; i < (RT / 4) * J; i += kSmallThreads) {
      const int q = i / J, j = i - q * J;
      float2 acc[4];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) acc[rr] = make_float2(0.f, 0.f);
      int m = 0;
      const cplx* xq = X + 4 * q;
      for (int k = 1; k <= nph; ++k) {
        m += j;
        if (m >= n) m -= n;
        const cplx w = tw[m];
        const float4 x01 = *reinterpret_cast<const float4*>(xq + k * XP);
        const float4 x23 = *reinterpret_cast<const float4*>(xq + k * XP + 2);
        acc[0] = __ffma2_rn(make_float2(x01.x, x01.y), w, acc[0]);     // (sum c cos, sum s sin)
        acc[1] = __ffma2_rn(make_float2(x01.z, x01.w), w, acc[1]);
        acc[2] = __ffma2_rn(make_float2(x23.x, x23.y), w, acc[2]);
        acc[3] = __ffma2_rn(make_float2(x23.z, x23.w), w, acc[3]);
      }
      const float4 h01 = *reinterpret_cast<const float4*>(xq), h23 = *reinterpret_cast<const float4*>(xq + 2);
      const cplx head[4] = {make_float2(h01.x, h01.y), make_float2(h01.z, h01.w), make_float2(h23.x, h23.y), make_float2(h23.z, h23.w)};
      const bool mirror = (j != 0) && (2 * j != n);
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const long long row = row0 + 4 * q + rr;
        if (row < p.rows) {
          float base = (MODE == kSpectrum) ? 2.0f * head[rr].x : head[rr].x;
          if ((n & 1) == 0) base += (j & 1) ? -head[rr].y : head[rr].y;
          p.z[row * n + j] = inv_n * (base + 2.0f * (acc[rr].x - acc[rr].y));
          if (mirror) p.z[row * n + (n - j)] = inv_n * (base + 2.0f * (acc[rr].x + acc[rr].y));
        }
      }
    }
  }
  if (MODE == kPsRng || MODE == kUniformRng || MODE == kUnitaryRng || MODE == kVonMisesRng) rng_launch_done(p.key);
}

// ---- backward ----------------------------------------------------------------------------------------------------
// smem: tw[n] | g[n][RT+4] floats | G[d][RT+2] cplx | per-row Beta-gradient constants RT x 8 floats | dk partials [TPR][RT]
constexpr int kSmallRowConst = 8;
inline size_t clifford_bwd_small_smem(int d, int rt) {
  const int n = 2 * d;
  return sizeof(cplx) * (size_t)n + sizeof(float) * (size_t)n * small_pitch_f(rt) + sizeof(cplx) * (size_t)d * small_pitch_c(rt) +
         sizeof(float) * (size_t)rt * kSmallRowConst + sizeof(float) * (size_t)kSmallThreads;
}

// Row constants of the implicit Beta gradient for short rows: the seven scalars of BetaGradConsts (two digammas, two
// logs), built by ONE thread per row -- a tile's rows in parallel lanes -- and the plain piecewise form per element.
// (The long-row kernels expand every branch into row polynomials with a warp per row, beta_row_build: ~600 issue slots
// per row, which a row of <= 63 elements cannot amortise -- measured 0.104 ms vs 0.023 ms per 65536 rows at d = 2.)
struct BetaGradPlain {
  BetaGradConsts c;
  __device__ __forceinline__ explicit BetaGradPlain(const float* v) : c(v, 0) {}
  __device__ __forceinline__ float grad(float x) const { return dirichlet_grad_one<false>(x, c); }
};

// Load RT rows of length n into g[j][r] and transform: S[k][r] = sum_j g_j e^{-2 pi i jk/n} for k = k0 .. d-1.
__device__ __forceinline__ void small_rows_dft(const float* __restrict__ src, long long row0, long long rows, int n, int d, int RT,
                                               int k0, const cplx* tw, float* g, cplx* S) {
  const int GP = small_pitch_f(RT), XP = small_pitch_c(RT);
  for (int i = threadIdx.x; i < RT * n; i += kSmallThreads) {
    const int r = i / n, j = i - r * n;
    g[j * GP + r] = (row0 + r < rows) ? ldg_stream1(src + (row0 + r) * n + j) : 0.0f;
  }
  __syncthreads();
  const int K = d - k0;
  for (int i = threadIdx.x; i < (RT / 4) * K; i += kSmallThreads) {
    const int q = i / K, k = k0 + (i - q * K);
    float2 acc[4];
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) acc[rr] = make_float2(0.f, 0.f);
    int m = 0;
    const float* gq = g + 4 * q;
    for (int j = 0; j < n; ++j) {
      const cplx w = make_float2(tw[m].x, -tw[m].y);                  // e^{-2 pi i jk/n}
      const float4 g4 = *reinterpret_cast<const float4*>(gq + j * GP);
      acc[0] = __ffma2_rn(make_float2(g4.x, g4.x), w, acc[0]);
      acc[1] = __ffma2_rn(make_float2(g4.y, g4.y), w, acc[1]);
      acc[2] = __ffma2_rn(make_float2(g4.z, g4.z), w, acc[2]);
      acc[3] = __ffma2_rn(make_float2(g4.w, g4.w), w, acc[3]);
      m += k;
      if (m >= n) m -= n;
    }
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) S[k * XP + 4 * q + rr] = acc[rr];
  }
  __syncthreads();
}

// VM: the von Mises torus family (saved offsets phi in tp_signed; row constant 1 - A(kappa) in rowconst[0]).
template <bool ROWK, bool VM = false>
__global__ void __launch_bounds__(kSmallThreads)
clifford_bwd_small_kernel(const CliffordBwdParams p, const int RT) {
  extern __shared__ __align__(16) unsigned char smem_small[];
  const int d = p.d, n = 2 * d;
  const int XP = small_pitch_c(RT);
  cplx* tw = reinterpret_cast<cplx*>(smem_small);
  float* g = reinterpret_cast<float*>(tw + n);
  cplx* G = reinterpret_cast<cplx*>(g + (size_t)n * small_pitch_f(RT));
  float* rowconst = reinterpret_cast<float*>(G + (size_t)d * XP);
  float* dkp = rowconst + (size_t)RT * kSmallRowConst;
  fill_twiddles(tw, n);
  const long long tiles = (p.rows + RT - 1) / RT;
  const int TPR = kSmallThreads / RT;                                // threads per row in the element phase
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long row0 = tile * RT;
    __syncthreads();
    // row constants of the Beta gradient: one thread per row (published by the barriers of the DFT)
    if (ROWK) {
      for (int r = threadIdx.x; r < RT; r += kSmallThreads) {
        if (row0 + r < p.rows) {
          const float kap = head_kappa(p.head, __ldg(p.kappa + ((row0 + r) % p.loc_rows) * p.kappa_row_stride));
          float* o = rowconst + r * kSmallRowConst;
          if constexpr (VM) {
            o[0] = vm_row_consts(kap).b;
          } else {
            const BetaGradConsts c(0.5f + (kap + kEps), 0.5f);
            o[0] = c.alpha; o[1] = c.beta; o[2] = c.total; o[3] = c.psi_alpha; o[4] = c.psi_total; o[5] = c.log_alpha; o[6] = c.log_total;
          }
        }
      }
    }
    small_rows_dft(p.grad_z, row0, p.rows, n, d, RT, 1, tw, g, G);
    // element phase: thread (r = tid % RT, kk = tid / RT) walks bins kk, kk + TPR, ... of its row
    const int r = threadIdx.x % RT, kk = threadIdx.x / RT;
    const long long row = row0 + r;
    float dk_sum = 0.f;
    if (row < p.rows) {
      const long long prow = row % p.loc_rows;
      BwdRowSrc src;
      src.loc = p.loc + prow * d;
      src.tps = p.tp_signed ? p.tp_signed + row * d : nullptr;
      src.tprime = p.tprime ? p.tprime + row * d : nullptr;
      src.gnoise = p.gnoise ? p.gnoise + row * d : nullptr;
      BetaGradPlain bc(rowconst + r * kSmallRowConst);               // (unused values when !ROWK)
      for (int k = kk; k < d; k += TPR) {
        if (k == 0) {
          p.dloc[row * d] = 0.f;
          if (!ROWK) p.dkappa[row * d] = 0.f;
          continue;
        }
        float dk = 0.f;
        if constexpr (VM)
          dk = vm_bwd_element<ROWK>(p, src, row, prow, k, G[k * XP + r], __ldg(p.kappa + prow * p.kappa_row_stride),
                                    rowconst[r * kSmallRowConst], 1.0f / (float)d);
        else clifford_bwd_element<ROWK>(p, src, row, prow, k, G[k * XP + r], bc, 1.0f / (float)d, dk);
        dk_sum += dk;
      }
    }
    if (ROWK) {
      dkp[kk * RT + r] = dk_sum;
      __syncthreads();
      if (kk == 0 && row < p.rows) {
        float tot = 0.f;
        for (int i = 0; i < TPR; ++i) tot += dkp[i * RT + r];
        p.dkappa[row] = tot * head_dkappa(p.head, __ldg(p.kappa + (row % p.loc_rows) * p.kappa_row_stride));
      }
    }
  }
}

// ---- log_prob ----------------------------------------------------------------------------------------------------
// smem: tw[n] | g[n][RT+4] floats | F[d][RT+2] cplx | partial sums 2 x [TPR][RT] | (logC, dlogC) per row
inline size_t clifford_lp_small_smem(int d, int rt) {
  const int n = 2 * d;
  return sizeof(cplx) * (size_t)n + sizeof(float) * (size_t)n * small_pitch_f(rt) + sizeof(cplx) * (size_t)d * small_pitch_c(rt) +
         sizeof(float) * 2 * (size_t)kSmallThreads + sizeof(float2) * (size_t)rt;
}

// VM: the von Mises torus family (vm_lp_element; consts[r] = (lnk, 1 - A)).
template <bool ROWK, bool VM = false>
__global__ void __launch_bounds__(kSmallThreads)
clifford_lp_small_kernel(const CliffordLogProbParams p, const int RT) {
  extern __shared__ __align__(16) unsigned char smem_small[];
  const int d = p.d, n = 2 * d;
  const int XP = small_pitch_c(RT);
  cplx* tw = reinterpret_cast<cplx*>(smem_small);
  float* g = reinterpret_cast<float*>(tw + n);
  cplx* F = reinterpret_cast<cplx*>(g + (size_t)n * small_pitch_f(RT));
  float* part = reinterpret_cast<float*>(F + (size_t)d * XP);
  float2* consts = reinterpret_cast<float2*>(part + 2 * kSmallThreads);
  fill_twiddles(tw, n);
  const long long tiles = (p.rows + RT - 1) / RT;
  const int TPR = kSmallThreads / RT;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long row0 = tile * RT;
    __syncthreads();
    if (ROWK) {
      for (int r = threadIdx.x; r < RT; r += kSmallThreads) {
        if (row0 + r < p.rows) {
          if constexpr (VM) {
            const VmRowConsts c = vm_row_consts(__ldg(p.kappa + ((row0 + r) % p.loc_rows) * p.kappa_row_stride));
            consts[r] = make_float2(c.lnk, c.b);
          } else {
            const PsConsts c = ps_consts((double)__ldg(p.kappa + ((row0 + r) % p.loc_rows) * p.kappa_row_stride), 0.5);
            consts[r] = make_float2((float)c.log_norm, (float)c.dlog_norm);
          }
        }
      }
    }
    small_rows_dft(p.value, row0, p.rows, n, d, RT, 0, tw, g, F);
    const int r = threadIdx.x % RT, kk = threadIdx.x / RT;
    const long long row = row0 + r;
    float acc = 0.f, dk_acc = 0.f;
    if (row < p.rows) {
      const long long prow = row % p.loc_rows;
      const float kap_row = __ldg(p.kappa + prow * p.kappa_row_stride);
      const float2 c = ROWK ? consts[r] : make_float2(0.f, 0.f);
      for (int k = kk; k < d; k += TPR) {
        cplx Fk = F[k * XP + r];
        if (k == 0) Fk.y = 0.0f;
        if constexpr (VM) vm_lp_element<ROWK>(p, row, prow, k, Fk, __ldg(p.loc + prow * d + k), kap_row, c.x, c.y, acc, dk_acc);
        else clifford_lp_element<ROWK>(p, row, prow, k, Fk, __ldg(p.loc + prow * d + k), kap_row, c.x, c.y, acc, dk_acc);
      }
    }
    part[kk * RT + r] = acc;
    part[kSmallThreads + kk * RT + r] = dk_acc;
    __syncthreads();
    if (kk == 0 && row < p.rows) {
      float tot = 0.f, dk_tot = 0.f;
      for (int i = 0; i < TPR; ++i) { tot += part[i * RT + r]; dk_tot += part[kSmallThreads + i * RT + r]; }
      p.log_prob[row] = tot;
      if (ROWK && p.dlp_dkappa) p.dlp_dkappa[row] = dk_tot;
    }
  }
}

}  // namespace cvb
