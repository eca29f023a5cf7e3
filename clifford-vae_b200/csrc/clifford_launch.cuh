// The size dispatch shared by the Clifford forward, backward and log_prob entry points (api_clifford_*.cu): which kernel
// serves a call follows from its row shape and pointer alignment alone.
#pragma once
#include "launch.cuh"
#include "clifford_small.cuh"

namespace cvb {

// In order:
//  - fft(std::integral_constant<int, log2 d>): the FFT engine, for power-of-two d in [16, 8192] with n = 2d and 8-byte
//    aligned output (or gradient) rows `out`;
//  - short rows (n <= kSmallMaxN): the row-tile kernel `small`, a tile of rows per CTA, small_smem(rows per tile) bytes;
//  - any other length: the direct-DFT kernel `generic`, one row per CTA, generic_smem bytes.
// `what` names the operation in error messages.
template <typename P, typename Fft, typename SmallKernel, typename SmallSmem, typename GenericKernel>
int dispatch_clifford(const char* what, const P& p, int n, const void* out, Fft fft, SmallKernel small, SmallSmem small_smem,
                      GenericKernel generic, size_t generic_smem, cudaStream_t st) {
  if (is_pow2(p.d) && p.d >= 16 && p.d <= 8192 && n == 2 * p.d && aligned(out, 8)) return with_int<4, 13>(ilog2(p.d), fft);
  if (n <= kSmallMaxN) {
    const int rt = small_rows_per_tile(p.rows, sm_count(), small_smem);
    return launch_persistent(small, what, kSmallThreads, small_smem(rt), (p.rows + rt - 1) / rt, st, p, rt);
  }
  CVB_REQUIRE(generic_smem <= kGenericSmemLimit, kUnsupported, "%s: length n=%d too large for the direct-DFT path", what, n);
  return launch_persistent(generic, what, kGenericThreads, generic_smem, p.rows, st, p);
}

// Whether the power-spherical draws a device-RNG forward saves for its backward (tp_signed) depend on the kernel tier.
// With one concentration per row and a power-of-two d in [512, 8192] the FFT engine saves the signed table coordinate
// of table-sampled rows (clifford_saves_table_coord); the row-tile and direct-DFT kernels save and read copysign(t', s).
// dispatch_clifford picks the tier from the alignment of z (forward) and grad_z (backward), so at these lengths both
// must be 8-byte aligned: otherwise one of the two calls would read the other's format as its own.
static_assert(clifford_saves_table_coord<9>() && !clifford_saves_table_coord<8>(), "table coordinates from d = 512 up");
inline bool ps_saved_draws_need_fft(int d, bool rowk) { return rowk && is_pow2(d) && d >= 512 && d <= 8192; }

}  // namespace cvb
