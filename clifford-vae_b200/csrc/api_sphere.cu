// C ABI entry points for the D-dimensional PowerSpherical / vMF / uniform-sphere kernels.
#include "launch.cuh"
#include "sphere_kernels.cuh"
#include "../../include/clifford_b200.h"

using namespace cvb;

namespace {
inline int row_warp_grid(long long rows) {
  long long b = (rows * 32 + 255) / 256;
  const long long cap = (long long)sm_count() * 8;
  return (int)(b < cap ? (b < 1 ? 1 : b) : cap);
}
}  // namespace

namespace {
// D <= 1024: the register-resident kernel (K = ceil(D / 128) element groups per lane); larger D: the two-pass kernel
template <int FAMILY>
int launch_sphere_rsample(const SphereParams& p, cudaStream_t st, const char* what) {
  const int grid = row_warp_grid(p.rows);
  const int k = (p.D + 127) / 128;
  if (k <= 8) {
    with_int<1, 8>(k, [&](auto K) { sphere_rsample_reg_kernel<FAMILY, decltype(K)::value><<<grid, 256, 0, st>>>(p); return kOk; });
  } else {
    sphere_rsample_kernel<FAMILY><<<grid, 256, 0, st>>>(p);
  }
  return check_launch(what);
}
template <int FAMILY>
int launch_sphere_rsample_bwd(const SphereParams& p, cudaStream_t st, const char* what) {
  const int grid = row_warp_grid(p.rows);
  const int k = (p.D + 127) / 128;
  if (k <= 8) {
    with_int<1, 8>(k, [&](auto K) { sphere_rsample_bwd_reg_kernel<FAMILY, decltype(K)::value><<<grid, 256, 0, st>>>(p); return kOk; });
  } else {
    sphere_rsample_bwd_kernel<FAMILY><<<grid, 256, 0, st>>>(p);
  }
  return check_launch(what);
}
}  // namespace

extern "C" {

int cvb_powerspherical_rsample(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                               const float* gnoise, unsigned long long seed, unsigned long long offset, float* z,
                               float* save, long long rows, int D, void* stream) {
  CVB_REQUIRE(loc && kappa && z && rows > 0 && loc_rows > 0 && D >= 2, kBadArgument, "cvb_powerspherical_rsample: bad arguments");
  CVB_REQUIRE((tprime == nullptr) == (gnoise == nullptr), kBadArgument, "cvb_powerspherical_rsample: give both tprime and gnoise or neither");
  SphereParams p{};
  p.loc = loc; p.kappa = kappa; p.loc_rows = loc_rows; p.tprime = tprime; p.gnoise = gnoise; p.g_pitch = D - 1;
  p.g_off = 0; p.z = z; p.save = save; p.rows = rows; p.D = D; p.norm_eps = 1e-7f; p.clamp_eps = 1e-7f;
  p.house_eps = 1e-7f; p.key = make_key(seed, offset, 0);
  return launch_sphere_rsample<kFamilyPS>(p, (cudaStream_t)stream, "sphere_rsample_kernel<PS>");
}

// rsample fused with entropy() / KL to the uniform prior (dists/clifford.py:204-212, :335-337): one launch for the
// training step's latent terms.  entropy / kl / dentropy: (loc_rows), each optional.
static int powerspherical_rsample_kl_impl(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                  const float* gnoise, unsigned long long seed, unsigned long long offset, float* z,
                                  float* save, float* entropy, float* kl, float* dentropy, long long rows, int D,
                                  KappaHead head, void* stream) {
  CVB_REQUIRE(loc && kappa && z && rows > 0 && loc_rows > 0 && D >= 2, kBadArgument, "cvb_powerspherical_rsample_kl: bad arguments");
  CVB_REQUIRE((tprime == nullptr) == (gnoise == nullptr), kBadArgument, "cvb_powerspherical_rsample_kl: give both tprime and gnoise or neither");
  SphereParams p{};
  p.loc = loc; p.kappa = kappa; p.loc_rows = loc_rows; p.tprime = tprime; p.gnoise = gnoise; p.g_pitch = D - 1;
  p.g_off = 0; p.z = z; p.save = save; p.rows = rows; p.D = D; p.norm_eps = 1e-7f; p.clamp_eps = 1e-7f;
  p.house_eps = 1e-7f; p.key = make_key(seed, offset, 0);
  p.entropy = entropy; p.kl = kl; p.dentropy = dentropy; p.head = head;
  // HypersphericalUniform.entropy (dists/clifford.py:109-121): ln 2 + (D/2) ln pi - lgamma(D/2)
  p.prior_entropy = 0.69314718055994530942 + 0.5 * (double)D * 1.14472988584940017414 - lgamma(0.5 * (double)D);
  return launch_sphere_rsample<kFamilyPS>(p, (cudaStream_t)stream, "sphere_rsample_kernel<PS,kl>");
}

static int powerspherical_rsample_backward_impl(const float* grad_z, const float* loc, const float* kappa, long long loc_rows,
                                        const float* tprime, const float* gnoise, const float* save,
                                        unsigned long long seed, unsigned long long offset, float* dloc, float* dkappa,
                                        long long rows, int D, KappaHead head, void* stream) {
  CVB_REQUIRE(grad_z && loc && kappa && dloc && dkappa && rows > 0 && loc_rows > 0 && D >= 2, kBadArgument,
              "cvb_powerspherical_rsample_backward: bad arguments");
  CVB_REQUIRE((tprime && gnoise) || (save && !tprime && !gnoise), kBadArgument,
              "cvb_powerspherical_rsample_backward: need (tprime, gnoise) or save");
  SphereParams p{};
  p.loc = loc; p.kappa = kappa; p.loc_rows = loc_rows; p.tprime = tprime; p.gnoise = gnoise; p.g_pitch = D - 1;
  p.g_off = 0; p.save = const_cast<float*>(save); p.grad_z = grad_z; p.dloc = dloc; p.dkappa = dkappa; p.rows = rows;
  p.D = D; p.norm_eps = 1e-7f; p.clamp_eps = 1e-7f; p.house_eps = 1e-7f; p.key = make_key(seed, offset, 0); p.head = head;
  return launch_sphere_rsample_bwd<kFamilyPS>(p, (cudaStream_t)stream, "sphere_rsample_bwd_kernel<PS>");
}

int cvb_powerspherical_log_prob(const float* value, const float* loc, const float* kappa, long long loc_rows,
                                float* log_prob, float* coef, float* dlp_dkappa, long long rows, int D, void* stream) {
  CVB_REQUIRE(value && loc && kappa && log_prob && rows > 0 && loc_rows > 0 && D >= 2, kBadArgument,
              "cvb_powerspherical_log_prob: bad arguments");
  CVB_REQUIRE((coef == nullptr) == (dlp_dkappa == nullptr), kBadArgument, "cvb_powerspherical_log_prob: give both coef and dlp_dkappa or neither");
  SphereLogProbParams p{value, loc, kappa, loc_rows, log_prob, coef, dlp_dkappa, rows, D};
  powerspherical_log_prob_kernel<<<row_warp_grid(rows), 256, 0, (cudaStream_t)stream>>>(p);
  return check_launch("powerspherical_log_prob_kernel");
}

int cvb_ps_log_normalizer(const float* kappa, long long rows, double half_dm1, float* log_norm, float* dlog_norm,
                          void* stream) {
  CVB_REQUIRE(kappa && log_norm && rows > 0, kBadArgument, "cvb_ps_log_normalizer: bad arguments");
  int blocks = (int)((rows + 127) / 128);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  ps_log_normalizer_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(kappa, rows, half_dm1, log_norm, dlog_norm);
  return check_launch("ps_log_normalizer_kernel");
}

int cvb_sphere_uniform_rsample(const float* gnoise, unsigned long long seed, unsigned long long offset, float* z,
                               long long rows, int D, float norm_eps, void* stream) {
  CVB_REQUIRE(z && rows > 0 && D >= 1, kBadArgument, "cvb_sphere_uniform_rsample: bad arguments");
  SphereParams p{};
  p.gnoise = gnoise; p.g_pitch = D; p.g_off = 0; p.z = z; p.rows = rows; p.D = D; p.norm_eps = norm_eps;
  p.loc_rows = 1; p.key = make_key(seed, offset, 0);
  sphere_rsample_kernel<kFamilyUniform><<<row_warp_grid(rows), 256, 0, (cudaStream_t)stream>>>(p);
  return check_launch("sphere_rsample_kernel<Uniform>");
}

int cvb_vmf_rsample(const float* loc, const float* kappa, long long loc_rows, const double* e_rounds,
                    const double* u_rounds, int n_rounds, const float* gnoise, unsigned long long seed,
                    unsigned long long offset, float* z, float* save, long long rows, int D, void* stream) {
  CVB_REQUIRE(loc && kappa && z && rows > 0 && loc_rows > 0 && D >= 2, kBadArgument, "cvb_vmf_rsample: bad arguments");
  const bool injected = gnoise != nullptr;
  if (injected) {
    CVB_REQUIRE(u_rounds && n_rounds >= 1 && (D == 3 || e_rounds), kBadArgument, "cvb_vmf_rsample: injected mode needs e_rounds/u_rounds");
  } else {
    CVB_REQUIRE(!e_rounds && !u_rounds, kBadArgument, "cvb_vmf_rsample: give all injected draws or none");
  }
  SphereParams p{};
  p.loc = loc; p.kappa = kappa; p.loc_rows = loc_rows; p.e_rounds = e_rounds; p.u_rounds = u_rounds;
  p.n_rounds = n_rounds; p.gnoise = gnoise; p.g_pitch = D; p.g_off = 1; p.z = z; p.save = save; p.rows = rows; p.D = D;
  p.norm_eps = 0.0f; p.clamp_eps = 1e-10f; p.house_eps = 1e-5f; p.key = make_key(seed, offset, 0);
  return launch_sphere_rsample<kFamilyVMF>(p, (cudaStream_t)stream, "sphere_rsample_kernel<VMF>");
}

// rsample fused with entropy / KL to the uniform prior / log-normaliser (von_mises_fisher.py:183-217): one launch.
static int vmf_rsample_kl_impl(const float* loc, const float* kappa, long long loc_rows, const double* e_rounds,
                       const double* u_rounds, int n_rounds, const float* gnoise, unsigned long long seed,
                       unsigned long long offset, float* z, float* save, float* entropy, float* kl, float* dentropy,
                       float* log_norm, float* dlog_norm, long long rows, int D, KappaHead head, void* stream) {
  CVB_REQUIRE(loc && kappa && z && rows > 0 && loc_rows > 0 && D >= 2, kBadArgument, "cvb_vmf_rsample_kl: bad arguments");
  const bool injected = gnoise != nullptr;
  if (injected) {
    CVB_REQUIRE(u_rounds && n_rounds >= 1 && (D == 3 || e_rounds), kBadArgument, "cvb_vmf_rsample_kl: injected mode needs e_rounds/u_rounds");
  } else {
    CVB_REQUIRE(!e_rounds && !u_rounds, kBadArgument, "cvb_vmf_rsample_kl: give all injected draws or none");
  }
  SphereParams p{};
  p.loc = loc; p.kappa = kappa; p.loc_rows = loc_rows; p.e_rounds = e_rounds; p.u_rounds = u_rounds;
  p.n_rounds = n_rounds; p.gnoise = gnoise; p.g_pitch = D; p.g_off = 1; p.z = z; p.save = save; p.rows = rows; p.D = D;
  p.norm_eps = 0.0f; p.clamp_eps = 1e-10f; p.house_eps = 1e-5f; p.key = make_key(seed, offset, 0);
  p.entropy = entropy; p.kl = kl; p.dentropy = dentropy; p.log_norm = log_norm; p.dlog_norm = dlog_norm; p.head = head;
  // vMF HypersphericalUniform.entropy (hyperspherical_uniform.py:48-54) in fp32 like the reference's tensor
  p.prior_entropy = (double)(float)(0.69314718055994530942 + 0.5 * (double)D * 1.14472988584940017414 - lgamma(0.5 * (double)D));
  return launch_sphere_rsample<kFamilyVMF>(p, (cudaStream_t)stream, "sphere_rsample_kernel<VMF,kl>");
}

static int vmf_rsample_backward_impl(const float* grad_z, const float* loc, const float* kappa, long long loc_rows,
                             const float* gnoise, const float* save, unsigned long long seed, unsigned long long offset,
                             float* dloc, float* dkappa, long long rows, int D, KappaHead head, void* stream) {
  CVB_REQUIRE(grad_z && loc && kappa && save && dloc && dkappa && rows > 0 && loc_rows > 0 && D >= 2, kBadArgument,
              "cvb_vmf_rsample_backward: bad arguments");
  SphereParams p{};
  p.loc = loc; p.kappa = kappa; p.loc_rows = loc_rows; p.gnoise = gnoise; p.g_pitch = D; p.g_off = 1;
  p.save = const_cast<float*>(save); p.grad_z = grad_z; p.dloc = dloc; p.dkappa = dkappa; p.rows = rows; p.D = D;
  p.norm_eps = 0.0f; p.clamp_eps = 1e-10f; p.house_eps = 1e-5f; p.key = make_key(seed, offset, 0); p.head = head;
  return launch_sphere_rsample_bwd<kFamilyVMF>(p, (cudaStream_t)stream, "sphere_rsample_bwd_kernel<VMF>");
}

int cvb_vmf_entropy_lognorm(const float* kappa, long long rows, int D, float* entropy, float* log_norm, float* dentropy,
                            float* dlog_norm, void* stream) {
  CVB_REQUIRE(kappa && rows > 0 && D >= 2, kBadArgument, "cvb_vmf_entropy_lognorm: bad arguments");
  int blocks = (int)((rows + 127) / 128);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  vmf_entropy_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(kappa, rows, D, entropy, log_norm, dentropy, dlog_norm);
  return check_launch("vmf_entropy_kernel");
}

// VonMisesFisher.log_prob (von_mises_fisher.py:193-212): kappa <loc, x> - log_norm; dot (rows) optional
int cvb_vmf_log_prob(const float* value, const float* loc, const float* kappa, const float* log_norm, long long loc_rows,
                     float* log_prob, float* dot, long long rows, int D, void* stream) {
  CVB_REQUIRE(value && loc && kappa && log_norm && log_prob && rows > 0 && loc_rows > 0 && D >= 1, kBadArgument,
              "cvb_vmf_log_prob: bad arguments");
  VmfLogProbParams p{value, loc, kappa, log_norm, loc_rows, log_prob, dot, rows, D};
  vmf_log_prob_kernel<<<row_warp_grid(rows), 256, 0, (cudaStream_t)stream>>>(p);
  return check_launch("vmf_log_prob_kernel");
}

// backward helper of the row log-densities: dvalue = w (x) loc, dloc = sum over samples of w (x) value
int cvb_sphere_logprob_backward(const float* w, const float* value, const float* loc, long long loc_rows, float* dvalue,
                                float* dloc, long long rows, int D, void* stream) {
  CVB_REQUIRE(w && value && loc && rows > 0 && loc_rows > 0 && D >= 1 && rows % loc_rows == 0 && (dvalue || dloc), kBadArgument,
              "cvb_sphere_logprob_backward: bad arguments");
  RowScaleParams p{w, value, loc, loc_rows, rows, D, dvalue, dloc};
  long long blocks = (loc_rows * (long long)D + 255) / 256;
  const long long cap = (long long)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  row_scale_pair_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  return check_launch("row_scale_pair_kernel");
}

// ---- public entry points over the implementations above: plain concentration, or the concentration head folded in
// (kappa = min(softplus(raw_scale) + floor, kmax), mnist/mlp_vae.py:69-71; every kappa-derivative is then d / d raw_scale)
int cvb_powerspherical_rsample_kl(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                  const float* gnoise, unsigned long long seed, unsigned long long offset, float* z,
                                  float* save, float* entropy, float* kl, float* dentropy, long long rows, int D,
                                  void* stream) {
  return powerspherical_rsample_kl_impl(loc, kappa, loc_rows, tprime, gnoise, seed, offset, z, save, entropy, kl, dentropy, rows, D,
                                        KappaHead{0, 0.f, 0.f}, stream);
}
int cvb_powerspherical_rsample_kl_head(const float* loc, const float* raw_scale, long long loc_rows, float floor, float kmax,
                                       const float* tprime, const float* gnoise, unsigned long long seed,
                                       unsigned long long offset, float* z, float* save, float* entropy, float* kl,
                                       float* dentropy_draw, long long rows, int D, void* stream) {
  CVB_REQUIRE(kmax > floor && floor >= 0.f, kBadArgument, "cvb_powerspherical_rsample_kl_head: need 0 <= floor < kmax");
  return powerspherical_rsample_kl_impl(loc, raw_scale, loc_rows, tprime, gnoise, seed, offset, z, save, entropy, kl, dentropy_draw,
                                        rows, D, KappaHead{1, floor, kmax}, stream);
}
int cvb_powerspherical_rsample_backward(const float* grad_z, const float* loc, const float* kappa, long long loc_rows,
                                        const float* tprime, const float* gnoise, const float* save,
                                        unsigned long long seed, unsigned long long offset, float* dloc, float* dkappa,
                                        long long rows, int D, void* stream) {
  return powerspherical_rsample_backward_impl(grad_z, loc, kappa, loc_rows, tprime, gnoise, save, seed, offset, dloc, dkappa, rows, D,
                                              KappaHead{0, 0.f, 0.f}, stream);
}
int cvb_powerspherical_rsample_backward_head(const float* grad_z, const float* loc, const float* raw_scale, long long loc_rows,
                                             float floor, float kmax, const float* tprime, const float* gnoise,
                                             const float* save, unsigned long long seed, unsigned long long offset,
                                             float* dloc, float* draw_scale, long long rows, int D, void* stream) {
  return powerspherical_rsample_backward_impl(grad_z, loc, raw_scale, loc_rows, tprime, gnoise, save, seed, offset, dloc, draw_scale,
                                              rows, D, KappaHead{1, floor, kmax}, stream);
}
int cvb_vmf_rsample_kl(const float* loc, const float* kappa, long long loc_rows, const double* e_rounds,
                       const double* u_rounds, int n_rounds, const float* gnoise, unsigned long long seed,
                       unsigned long long offset, float* z, float* save, float* entropy, float* kl, float* dentropy,
                       float* log_norm, float* dlog_norm, long long rows, int D, void* stream) {
  return vmf_rsample_kl_impl(loc, kappa, loc_rows, e_rounds, u_rounds, n_rounds, gnoise, seed, offset, z, save, entropy, kl, dentropy,
                             log_norm, dlog_norm, rows, D, KappaHead{0, 0.f, 0.f}, stream);
}
int cvb_vmf_rsample_kl_head(const float* loc, const float* raw_scale, long long loc_rows, float floor, float kmax,
                            const double* e_rounds, const double* u_rounds, int n_rounds, const float* gnoise,
                            unsigned long long seed, unsigned long long offset, float* z, float* save, float* entropy,
                            float* kl, float* dentropy_draw, float* log_norm, float* dlog_norm_draw, long long rows, int D,
                            void* stream) {
  CVB_REQUIRE(kmax > floor && floor >= 0.f, kBadArgument, "cvb_vmf_rsample_kl_head: need 0 <= floor < kmax");
  return vmf_rsample_kl_impl(loc, raw_scale, loc_rows, e_rounds, u_rounds, n_rounds, gnoise, seed, offset, z, save, entropy, kl,
                             dentropy_draw, log_norm, dlog_norm_draw, rows, D, KappaHead{1, floor, kmax}, stream);
}
int cvb_vmf_rsample_backward(const float* grad_z, const float* loc, const float* kappa, long long loc_rows,
                             const float* gnoise, const float* save, unsigned long long seed, unsigned long long offset,
                             float* dloc, float* dkappa, long long rows, int D, void* stream) {
  return vmf_rsample_backward_impl(grad_z, loc, kappa, loc_rows, gnoise, save, seed, offset, dloc, dkappa, rows, D,
                                   KappaHead{0, 0.f, 0.f}, stream);
}
int cvb_vmf_rsample_backward_head(const float* grad_z, const float* loc, const float* raw_scale, long long loc_rows,
                                  float floor, float kmax, const float* gnoise, const float* save, unsigned long long seed,
                                  unsigned long long offset, float* dloc, float* draw_scale, long long rows, int D,
                                  void* stream) {
  return vmf_rsample_backward_impl(grad_z, loc, raw_scale, loc_rows, gnoise, save, seed, offset, dloc, draw_scale, rows, D,
                                   KappaHead{1, floor, kmax}, stream);
}

}  // extern "C"
