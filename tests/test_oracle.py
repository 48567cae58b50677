"""The oracle against the golden vectors recorded from the reference's own classes (oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_l2
from oracle.gan import GANOracle, lightning_step, sample_patch_origins, synthetic_batch, gather_patches
from oracle.monai_unet import UNet
from oracle.nets import CasNetGenerator, Discriminator, PatchDiscriminator

# intra-op threads the golden vectors were recorded with.  torch's CPU convolutions split their reductions by thread, and
# two comparisons here amplify the resulting rounding differences past their bounds: the gradient norms of the
# perceptual step's near-zero tensors, and everything after Adam's first update (~lr * sign(g)) in the 2-D twin step
GOLDEN_THREADS = 8


@pytest.fixture(autouse=True)
def _golden_thread_count():
    saved = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(saved)


def _load(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def _grad_summary(named_params):
    return {n: torch.stack([p.grad.double().norm(), p.grad.double().sum()]).float() for n, p in named_params}


def _close(a, b, tol=2e-5):
    assert rel_l2(a, b) <= tol, (rel_l2(a, b), a.flatten()[:4], b.flatten()[:4])


def test_unet_structure_invariants():
    # SURVEY.md section 8a/8c: 75 parameter tensors / 402 442 parameters per 2-D UNet(16,32,64,128); shape-preserving
    u = UNet(2, 1, 1, (16, 32, 64, 128), (2, 2, 2), num_res_units=2)
    assert len(list(u.parameters())) == 75
    assert sum(p.numel() for p in u.parameters()) == 402442
    x = torch.zeros(1, 1, 32, 32)
    assert u(x).shape == x.shape
    keys = list(u.state_dict().keys())
    assert keys[0] == "model.0.conv.unit0.conv.weight" and "model.0.residual.weight" in keys
    assert any(k.startswith("model.1.submodule.1.submodule.1.submodule.conv.unit0") for k in keys)  # bottom layer
    assert u.state_dict()["model.2.0.conv.weight"].shape == (32, 1, 3, 3)  # ConvT weight (Cin, Cout, k, k)
    assert "model.2.1.conv.unit0.conv.weight" in keys and "model.2.1.conv.unit0.norm.weight" not in keys


def test_generator_matches_reference_3d():
    fix = _load("ref_generator_3d.pt")
    torch.manual_seed(fix["seed_weights"])
    g = CasNetGenerator((1, 16, 16, 16), 6, dims=3)
    assert len(list(g.parameters())) == fix["n_param_tensors"] == 450
    assert sum(p.numel() for p in g.parameters()) == fix["n_params"] == 7121832
    assert list(g.state_dict().keys()) == fix["state_keys"]
    x = torch.rand(fix["input_shape"], generator=torch.Generator().manual_seed(fix["seed_input"])) * 2 - 1
    _close(g(x), fix["out"])


def test_patch_discriminator_matches_reference_3d():
    fix = _load("ref_patch_discriminator_3d.pt")
    torch.manual_seed(fix["seed_weights"])
    d = PatchDiscriminator((1, 16, 16, 16), dims=3, spatial=16)
    x = torch.rand(fix["input_shape"], generator=torch.Generator().manual_seed(fix["seed_input"])) * 2 - 1
    v, acts = d(x)
    _close(v, fix["validity"])
    assert len(acts) == 16 and [list(acts[k].shape) for k in range(16)] == fix["act_shapes"]
    _close(torch.stack([acts[k].double().sum() for k in range(16)]).float(), fix["act_sums"], 1e-4)
    v.sum().backward()
    got = _grad_summary(d.named_parameters())
    for k, ref in fix["grad_summary"].items():
        assert abs(float(got[k][0]) - float(ref[0])) <= 1e-4 * max(1e-6, float(ref[0])) + 1e-9, k
    _close(d.model_conv[1].running_mean, fix["bn_running_mean_0"])


def test_perceptual_step_matches_reference_3d():
    fix = _load("ref_perceptual_step_3d.pt")
    B, S, NS = fix["B"], fix["S"], fix["num_samples"]
    torch.manual_seed(fix["seed_weights"])
    batch = synthetic_batch(B, 3, S, seed=fix["seed_input"])
    # the reference GAN draws the generator first, then the discriminator: same order here
    m = GANOracle("perceptual", dims=3, spatial=S, num_samples=NS)
    origins = sample_patch_origins(np.random.RandomState(fix["seed_origins"]), B, NS, (S, S, S), 16)
    assert np.array_equal(origins, fix["origins"].numpy())
    for opt_idx in (0, 1):
        for net, on in ((m.generator, opt_idx == 0), (m.discriminator, opt_idx == 1)):
            for p in net.parameters():
                p.requires_grad_(on)
        loss = m.training_step(batch, 0, opt_idx, patch_origins=origins)
        _close(loss.detach().reshape(-1), fix[f"loss{opt_idx}"])
        loss.backward()
        net = m.generator if opt_idx == 0 else m.discriminator
        got = _grad_summary(net.named_parameters())
        ref = fix[f"grad_summary{opt_idx}"]
        worst = max(abs(float(got[k][0]) - float(ref[k][0])) / max(float(ref[k][0]), 1e-8) for k in ref
                    if float(ref[k][0]) > 1e-6)
        assert worst <= 1e-3, worst
        for p in m.parameters():
            p.grad = None
    for k, v in fix["logged"].items():
        if k in m.logged:
            _close(m.logged[k].reshape(-1), v)


def test_patch_gather_is_exact_copy():
    rng = np.random.RandomState(3)
    vol = torch.rand(2, 1, 20, 24)
    o = sample_patch_origins(rng, 2, 5, (20, 24), 16)
    p = gather_patches(vol, o, 16)
    assert p.shape == (10, 1, 16, 16)
    for b in range(2):
        for s in range(5):
            oh, ow = o[b, s]
            assert torch.equal(p[b * 5 + s, 0], vol[b, 0, oh:oh + 16, ow:ow + 16])
    assert o.min() >= 0 and o[..., 0].max() <= 4 and o[..., 1].max() <= 8


def test_2d_twin_golden_step():
    fix = _load("oracle_final_step_2d_64.pt")
    torch.manual_seed(fix["seed_weights"])
    m = GANOracle("final", dims=2, spatial=fix["S"])
    batch = synthetic_batch(fix["B"], 2, fix["S"], seed=fix["seed_input"])
    opts, _ = m.configure_optimizers()
    grads = {}
    losses = lightning_step(m, opts, batch, 0, keep_grads=grads)
    _close(losses[0].reshape(-1), fix["g_loss"])
    _close(losses[1].reshape(-1), fix["d_loss"])
    big = [k for k, v in fix["grad_norms"].items() if float(v) > 1e-5]
    worst = max(abs(float(grads[k].double().norm()) - float(fix["grad_norms"][k])) / float(fix["grad_norms"][k]) for k in big)
    assert worst <= 2e-3, worst
    with torch.no_grad():
        m.eval()
        _close(m(batch["t1w"]), fix["eval_out_after_step"], 1e-4)


def test_saturation_after_one_step():
    """SURVEY.md section 0: the reference's adversarial path saturates; BCE clamps at 100 and D's gradient vanishes."""
    torch.manual_seed(0)
    m = GANOracle("final", dims=2, spatial=64)
    batch = synthetic_batch(2, 2, 64, seed=1)
    opts, _ = m.configure_optimizers()
    lightning_step(m, opts, batch, 0)
    lightning_step(m, opts, batch, 1)
    assert float(m.logged["g_adv_loss"]) > 10.0  # saturating towards the -100 log clamp


def test_final_discriminator_matches_reference_128():
    fix = _load("ref_final_discriminator_128.pt")
    torch.manual_seed(fix["seed_weights"])
    d = Discriminator((1, 128, 128, 128), dims=3, spatial=128)
    assert sum(p.numel() for p in d.parameters()) == fix["n_params"] == 12760065
    assert list(d.state_dict().keys()) == fix["state_keys"]
    assert d.model_linear[1].in_features == 256 * 29 ** 3  # GAN_final.py:201
    if os.environ.get("MPGAN_SLOW") != "1":
        pytest.skip("128^3 forward takes ~20 s of CPU; set MPGAN_SLOW=1")
    x = torch.rand(fix["input_shape"], generator=torch.Generator().manual_seed(fix["seed_input"])) * 2 - 1
    with torch.no_grad():
        _close(d(x), fix["validity"], 1e-4)
