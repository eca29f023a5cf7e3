// C ABI entry points for the VSA / HRR kernels (include/clifford_b200.h).
#include "launch.cuh"
#include "vsa_kernels.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

extern "C" int cvb_internal_bind_a(const cvb::BindParams* p, int d, int mode, void* stream);
extern "C" int cvb_internal_bind_b(const cvb::BindParams* p, int d, int mode, void* stream);
extern "C" int cvb_internal_unitary(float* out, long long n, int d, float eps, unsigned long long seed,
                                    unsigned long long offset, void* stream);

namespace {

__global__ void normal_fill_kernel(float* out, long long total, float scale, PhiloxKey key) {
  // each Philox call yields 4 normals
  const long long nvec = (total + 3) / 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    const uint4 r = philox_draw(key, (uint64_t)i, 0);
    const float2 n01 = box_muller(r.x, r.y), n23 = box_muller(r.z, r.w);
    const float v[4] = {n01.x * scale, n01.y * scale, n23.x * scale, n23.y * scale};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * i + j < total) out[4 * i + j] = v[j];
  }
  rng_launch_done(key);
}

inline int ew_grid(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = (long long)sm_count() * 16;
  return (int)(b < cap ? (b < 1 ? 1 : b) : cap);
}

}  // namespace

extern "C" {

int cvb_vsa_bind(const float* a, const float* b, float* out, long long rows, long long a_rows, long long b_rows, int d,
                 int mode, void* stream) {
  CVB_REQUIRE(a && b && out, kBadArgument, "cvb_vsa_bind: null pointer");
  CVB_REQUIRE(rows > 0 && a_rows > 0 && b_rows > 0 && d >= 1, kBadArgument, "cvb_vsa_bind: bad sizes");
  BindParams p{a, b, out, rows, a_rows, b_rows, nullptr};
  if (mode == CVB_BIND_MUL || mode == CVB_BIND_MUL_CONJ) return cvb_internal_bind_a(&p, d, mode, stream);
  if (mode == CVB_BIND_DIV || mode == CVB_BIND_DIV_CONJ || mode == CVB_BIND_NEG_MUL_CONJ) return cvb_internal_bind_b(&p, d, mode, stream);
  set_last_error("cvb_vsa_bind: unknown mode %d", mode);
  return kBadArgument;
}

int cvb_vsa_depth_chain_cosine(const float* vecs, float* out, long long trials, int m_plus_1, int d, void* stream) {
  CVB_REQUIRE(vecs && out && trials > 0 && m_plus_1 >= 1, kBadArgument, "cvb_vsa_depth_chain_cosine: bad arguments");
  CVB_REQUIRE(is_pow2(d) && d >= 32 && d <= 16384 && aligned(vecs, 8), kUnsupported,
              "cvb_vsa_depth_chain_cosine: d=%d must be a power of two in [32, 16384] (use bind/unbind otherwise)", d);
  return with_int<4, 13>(ilog2(d) - 1, [&](auto L) -> int {
    using Pl = FftPlan<decltype(L)::value>;
    const cplx* tw = device_twiddles();
    if (!tw) return kCudaError;
    return launch_persistent(depth_chain_kernel<decltype(L)::value>, "depth_chain_kernel", Pl::THREADS,
                             sizeof(cplx) * Pl::XCH * Pl::GROUPS + sizeof(float) * 32 * Pl::GROUPS,
                             (trials + Pl::GROUPS - 1) / Pl::GROUPS, (cudaStream_t)stream, vecs, out, trials, m_plus_1, tw);
  });
}

int cvb_vsa_invert(const float* a, float* out, long long rows, int d, void* stream) {
  CVB_REQUIRE(a && out && rows > 0 && d >= 1, kBadArgument, "cvb_vsa_invert: bad arguments");
  invert_kernel<<<ew_grid(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(a, out, rows, d);
  return check_launch("invert_kernel");
}

int cvb_vsa_permute(const float* v, const long long* perm, float* out, long long rows, int d, int inverse, void* stream) {
  CVB_REQUIRE(v && perm && out && rows > 0 && d >= 1, kBadArgument, "cvb_vsa_permute: bad arguments");
  permute_kernel<<<ew_grid(rows * 256, 256), 256, 0, (cudaStream_t)stream>>>(v, perm, out, rows, d, inverse);
  return check_launch("permute_kernel");
}

static int bundle_chunks(long long k, int d) {
  const long long col_blocks = (d + 127) / 128;
  long long want = ((long long)sm_count() * 8 + col_blocks - 1) / col_blocks;   // ~8 CTAs per SM in total
  if (want > (k + 7) / 8) want = (k + 7) / 8;                                     // at least 8 rows per chunk
  if (want < 1) want = 1;
  if (want > 65535) want = 65535;
  return (int)want;
}

long long cvb_vsa_bundle_workspace_bytes(long long k, int d) {
  if (k <= 0 || d <= 0) return 0;
  return (long long)bundle_chunks(k, d) * d * (long long)sizeof(float);
}

int cvb_vsa_bundle(const float* v, float* out, long long k, int d, float scale, void* workspace, void* stream) {
  CVB_REQUIRE(v && out && workspace && k > 0 && d >= 1, kBadArgument, "cvb_vsa_bundle: bad arguments");
  const int chunks = bundle_chunks(k, d);
  const long long rpc = (k + chunks - 1) / chunks;
  dim3 grid((d + 127) / 128, chunks);
  bundle_partial_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(v, (float*)workspace, k, d, rpc);
  if (int rc = check_launch("bundle_partial_kernel")) return rc;
  bundle_final_kernel<<<(d + 255) / 256, 256, 0, (cudaStream_t)stream>>>((const float*)workspace, out, chunks, d, scale);
  return check_launch("bundle_final_kernel");
}

int cvb_vsa_cosine(const float* a, const float* b, float* out, long long rows, long long a_rows, long long b_rows, int d,
                   void* stream) {
  CVB_REQUIRE(a && b && out && rows > 0 && a_rows > 0 && b_rows > 0 && d >= 1, kBadArgument, "cvb_vsa_cosine: bad arguments");
  CVB_REQUIRE((d & 3) != 0 || (aligned(a, 16) && aligned(b, 16)), kBadArgument, "cvb_vsa_cosine: rows must be 16-byte aligned");
  cosine_kernel<<<ew_grid(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(a, b, out, rows, a_rows, b_rows, d);
  return check_launch("cosine_kernel");
}

int cvb_vsa_cosine_backward(const float* a, const float* b, const float* grad_out, float* da, float* db, long long rows,
                            long long a_rows, long long b_rows, int d, void* stream) {
  CVB_REQUIRE(a && b && grad_out && (da || db) && rows > 0 && d >= 1, kBadArgument, "cvb_vsa_cosine_backward: bad arguments");
  cosine_bwd_kernel<<<ew_grid(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(a, b, grad_out, da, db, rows, a_rows, b_rows, d);
  return check_launch("cosine_bwd_kernel");
}

int cvb_vsa_normalize(const float* x, float* out, long long rows, int d, void* stream) {
  CVB_REQUIRE(x && out && rows > 0 && d >= 1, kBadArgument, "cvb_vsa_normalize: bad arguments");
  const int vec4 = (d % 4 == 0) && aligned(x, 16) && aligned(out, 16);
  normalize_kernel<<<ew_grid(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(x, out, rows, d, vec4);
  return check_launch("normalize_kernel");
}

int cvb_vsa_normalize_backward(const float* x, const float* grad_out, float* dx, long long rows, int d, void* stream) {
  CVB_REQUIRE(x && grad_out && dx && rows > 0 && d >= 1, kBadArgument, "cvb_vsa_normalize_backward: bad arguments");
  normalize_bwd_kernel<<<ew_grid(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(x, grad_out, dx, rows, d);
  return check_launch("normalize_bwd_kernel");
}

int cvb_vsa_hrr_init(float* out, long long n, int d, unsigned long long seed, unsigned long long offset, void* stream) {
  CVB_REQUIRE(out && n > 0 && d >= 1, kBadArgument, "cvb_vsa_hrr_init: bad arguments");
  const long long total = n * d;
  normal_fill_kernel<<<ew_grid((total + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(out, total, 1.0f / sqrtf((float)d),
                                                                                       make_key(seed, offset, 3));
  return check_launch("normal_fill_kernel");
}

int cvb_vsa_unitary_init(float* out, long long n, int d, float eps, unsigned long long seed, unsigned long long offset,
                         void* stream) {
  CVB_REQUIRE(out && n > 0 && d >= 2, kBadArgument, "cvb_vsa_unitary_init: bad arguments");
  return cvb_internal_unitary(out, n, d, eps, seed, offset, stream);
}

}  // extern "C"
