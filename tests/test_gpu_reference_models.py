"""GPU, model level: the reference's OWN model code -- `mnist.mlp_vae.MLPVAE` + `vae_loss` (mnist/mlp_vae.py:19-143) and
`cnn.models.VAE` + `compute_loss` (cnn/models.py:134-315) -- imported UNMODIFIED (checkout when present, else the copy
staged under oracle/_ref by oracle/stage_reference.py) and run on the drop-in distributions, against fixtures the real
reference produced on CPU with the same seeded weights, inputs and recorded latent draws
(tests/golden/vae_step.npz, conv_vae_step.npz; oracle/gen_golden.py:gen_vae_step / gen_conv_vae_step)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _ref():
    from oracle import reference_loader as RL
    ref = RL.load()
    if ref is None:
        pytest.skip("no copy of the reference (neither /root/reference nor oracle/_ref)")
    return RL, ref


def _case(fname, dist_name):
    z = np.load(os.path.join(GOLDEN, fname))
    return {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(dist_name + "/")}


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture(autouse=True)
def _exact_fp32_gemms():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("dist_name,z_dim", [("clifford", 16), ("powerspherical", 9), ("vmf", 9)])
def test_reference_mlp_vae_loss_unchanged_on_drop_ins(dist_name, z_dim):
    """Without a copy of the reference, the same fixture is checked on the restated layer layout of test_gpu_vae_step."""
    from clifford_b200 import _lib, distributions as D
    from clifford_b200.testing import injected_draws
    from oracle import reference_loader as RL
    ref = RL.load()
    if ref is None:
        import test_gpu_vae_step
        test_gpu_vae_step.test_mlp_vae_loss_and_gradients_match_reference(dist_name, z_dim)
        return
    mv = RL.models(ref, "mnist")
    assert mv.CliffordPowerSphericalDistribution is D.CliffordPowerSphericalDistribution
    c = _case("vae_step.npz", dist_name)
    torch.manual_seed(20240 + z_dim)
    model = mv.MLPVAE(h_dim=128, z_dim=z_dim, distribution=dist_name)
    assert abs(sum(p.double().sum().item() for p in model.parameters()) - float(c["param_checksum"])) < 1e-9
    model = model.to(DEV)
    x = T(c["x"])
    if dist_name == "vmf":
        R = c["e_rounds"].shape[0]
        draws = (T(c["e_rounds"]).reshape(R, -1), T(c["u_rounds"]).reshape(R, -1), T(c["g"]))
    else:
        draws = (T(c["tprime"]), T(c["g"]))
    n0 = _lib.launch_count()
    with injected_draws(draws):
        res = mv.vae_loss(model, x, beta=1.0, return_dict=True)
    res["total"].backward()
    assert _lib.launch_count() - n0 >= 2          # sampler (+ fused entropy / KL) and backward ran in libclifford_b200.so
    assert abs(float(res["recon"]) - float(c["recon"])) < 2e-5 * abs(float(c["recon"]))
    assert abs(float(res["kl"]) - float(c["kl"])) < 2e-5 * max(1.0, abs(float(c["kl"])), abs(float(c["entropy"])))
    assert abs(float(res["entropy"]) - float(c["entropy"])) < 2e-5 * max(1.0, abs(float(c["entropy"])))
    assert abs(float(res["total"]) - float(c["total"])) < 2e-5 * abs(float(c["total"]))
    for name, prm in model.named_parameters():
        want = float(c["grad_norm/" + name])
        assert abs(float(prm.grad.norm()) - want) < 2e-4 * max(want, 1e-3), (name, float(prm.grad.norm()), want)
    assert rel_err(model.fc_scale.weight.grad.cpu(), c["grad/fc_scale.weight"]) < 5e-4
    assert rel_err(model.fc_mean.bias.grad.cpu(), c["grad/fc_mean.bias"]) < 1e-4
    assert rel_err(model.decoder[0].bias.grad.cpu(), c["grad/decoder.0.bias"]) < 1e-4


@pytest.mark.parametrize("dist_name,latent_dim", [("clifford", 64), ("powerspherical", 33)])
def test_reference_conv_vae_step_unchanged_on_drop_ins(dist_name, latent_dim):
    """The C3 model class (cnn/models.py VAE: ResBlock encoder, fc_mu / fc_concentration heads with the dimension-
    dependent concentration floor, ResUpBlock decoder) at a small latent; convolutions run on cuDNN in strict fp32."""
    from clifford_b200 import _lib
    from clifford_b200.testing import injected_draws
    RL, ref = _ref()
    cm = RL.models(ref, "cnn")
    c = _case("conv_vae_step.npz", dist_name)
    torch.manual_seed(777 + latent_dim)
    model = cm.VAE(latent_dim=latent_dim, in_channels=3, distribution=dist_name, device="cpu", recon_loss_type="l1")
    assert abs(sum(p.double().sum().item() for p in model.parameters()) - float(c["param_checksum"])) < 1e-9
    model = model.to(DEV)
    model.device = DEV
    x = T(c["x"])
    n0 = _lib.launch_count()
    with injected_draws((T(c["tprime"]), T(c["g"]))):
        x_recon, q_z, p_z, mu = model(x)
        losses = model.compute_loss(x, x_recon, q_z, p_z, 1.0)
    losses["total_loss"].backward()
    assert _lib.launch_count() - n0 >= 2
    assert rel_err(mu.detach().cpu(), c["mu"]) < 2e-5
    assert rel_err(x_recon.detach().cpu(), c["x_recon"]) < 5e-5
    assert abs(float(losses["recon_loss"]) - float(c["recon"])) < 2e-5 * abs(float(c["recon"]))
    assert abs(float(losses["kld_loss"]) - float(c["kl"])) < 2e-5 * max(1.0, abs(float(c["kl"])), abs(float(c["entropy"])))
    assert abs(float(losses["entropy"]) - float(c["entropy"])) < 2e-5 * max(1.0, abs(float(c["entropy"])))
    assert abs(float(losses["total_loss"]) - float(c["total"])) < 2e-5 * abs(float(c["total"]))
    for name, prm in model.named_parameters():
        want = float(c["grad_norm/" + name])
        assert abs(float(prm.grad.norm()) - want) < 5e-4 * max(want, 1e-3), (name, float(prm.grad.norm()), want)
    assert rel_err(model.encoder.fc_concentration.weight.grad.cpu(), c["grad/encoder.fc_concentration.weight"]) < 1e-3
    assert rel_err(model.encoder.fc_mu.bias.grad.cpu(), c["grad/encoder.fc_mu.bias"]) < 2e-4
    assert rel_err(model.decoder.fc.bias.grad.cpu(), c["grad/decoder.fc.bias"]) < 2e-4


class _C3LayoutVAE(torch.nn.Module):
    """The C3 model's layer layout at latent_dim=2048, 'clifford' (the parameter names of conv_vae_step.npz; the shapes
    follow from its 18,447,300 parameters): four ResBlocks 3-64-128-256-512 (4x4 stride-2 conv + 1x1 stride-2 skip),
    fc_mu / fc_concentration, fc -> 512x2x2, three transposed ResUpBlocks, a 4x4 transposed output conv.  Its activations
    and initialisation are not the reference's, so it stands in only where nothing is compared with stored values."""

    def __init__(self, d=2048, floor=0.13):
        super().__init__()
        nn, ch = torch.nn, [3, 64, 128, 256, 512]

        def block(conv, skip):
            b = nn.Module()
            b.conv, b.skip = conv, skip
            return b
        self.d, self.floor = d, floor
        self.encoder = nn.Module()
        self.encoder.blocks = nn.ModuleList(block(nn.Conv2d(ch[i], ch[i + 1], 4, 2, 1), nn.Conv2d(ch[i], ch[i + 1], 1, 2))
                                            for i in range(4))
        self.encoder.fc_mu = nn.Linear(2048, d)
        self.encoder.fc_concentration = nn.Linear(2048, 1)
        self.decoder = nn.Module()
        self.decoder.fc = nn.Linear(2 * d, 2048)
        self.decoder.blocks = nn.ModuleList(
            block(nn.ConvTranspose2d(ch[4 - i], ch[3 - i], 4, 2, 1), nn.ConvTranspose2d(ch[4 - i], ch[3 - i], 1, 2, output_padding=1))
            for i in range(3))
        self.decoder.final = nn.Sequential(nn.ConvTranspose2d(64, 3, 4, 2, 1), nn.Tanh())

    def forward(self, x):
        from dists.clifford import CliffordPowerSphericalDistribution, CliffordTorusUniform
        F = torch.nn.functional
        h = x
        for b in self.encoder.blocks:
            h = F.leaky_relu(b.conv(h), 0.2) + b.skip(h)
        h = h.flatten(1)
        mu = self.encoder.fc_mu(h)
        kap = torch.clamp(F.softplus(self.encoder.fc_concentration(h)) + self.floor, max=10.0)
        q = CliffordPowerSphericalDistribution(mu, kap.expand_as(mu))
        h = self.decoder.fc(q.rsample()).view(-1, 512, 2, 2)
        for b in self.decoder.blocks:
            h = F.leaky_relu(b.conv(h), 0.2) + b.skip(h)
        return self.decoder.final(h), q, CliffordTorusUniform(self.d, device=x.device), mu

    def compute_loss(self, x, x_recon, q, p, beta):
        recon = (x_recon - x).abs().sum() / x.shape[0]
        kld = torch.distributions.kl.kl_divergence(q, p).mean()
        return {"recon_loss": recon, "kld_loss": kld, "total_loss": recon + beta * kld}


def test_c3_model_trains_with_device_rng():
    """cnn.models.VAE(latent_dim=2048, 'clifford') -- the BASELINE config-3 model, 18.4 M parameters -- a few optimiser
    steps on the drop-in kernels with the device generator: finite losses, loss goes down, KL >= 0.  Without a copy of
    the reference, the same steps run on a model of the same layer layout (_C3LayoutVAE)."""
    from oracle import reference_loader as RL
    ref = RL.load()
    torch.manual_seed(0)
    if ref is None:
        model = _C3LayoutVAE().to(DEV)
    else:
        model = RL.models(ref, "cnn").VAE(latent_dim=2048, in_channels=3, distribution="clifford", device=DEV,
                                          recon_loss_type="l1")
    assert sum(p.numel() for p in model.parameters()) == 18_447_300
    opt = torch.optim.AdamW(model.parameters(), lr=3e-4)
    x = torch.rand(64, 3, 32, 32, device=DEV) * 2 - 1
    hist = []
    for _ in range(6):
        opt.zero_grad()
        x_recon, q_z, p_z, _ = model(x)
        losses = model.compute_loss(x, x_recon, q_z, p_z, 1.0)
        losses["total_loss"].backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        hist.append(float(losses["total_loss"]))
        assert float(losses["kld_loss"]) >= 0 and np.isfinite(hist[-1])
    assert hist[-1] < hist[0]
