"""Host-side logic that needs no GPU: convolution geometry of the plan builder, percentile rank selection, checkpoint
hyper-parameter resolution."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from mpgan import ops
from mpgan import transforms as T
from oracle import transforms as ot


@pytest.mark.parametrize("k,s,p,size", [(3, 1, 0, 256), (3, 1, 1, 128), (3, 2, 1, 256), (4, 2, 0, 252), (4, 2, 0, 125), (1, 1, 0, 32)])
def test_conv_spec_matches_torch_output_sizes(k, s, p, size):
    conv = nn.Conv2d(2, 3, k, stride=s, padding=p)
    spec = ops.ConvSpec.from_module(conv)
    y = conv(torch.zeros(1, 2, size, size))
    assert spec.y_of_x((size, size)) == tuple(y.shape[2:]) and not spec.transposed and (spec.cx, spec.cy) == (2, 3)
    g = spec.geom(5, (size, size), tuple(y.shape[2:]))
    assert (g.rank, g.n, g.cx, g.cy) == (2, 5, 2, 3) and list(g.xs) == [1, size, size] and list(g.k) == [1, k, k]
    if s == 2 and k == 3:   # MONAI's up path: ConvTranspose(k3, s2, p1, output_padding 1) doubles the size
        ct = nn.ConvTranspose2d(3, 2, k, stride=s, padding=p, output_padding=s - 1)
        st = ops.ConvSpec.from_module(ct)
        out = ct(torch.zeros(1, 3, size // 2, size // 2))
        assert st.transposed and (st.cx, st.cy) == (2, 3) and st.x_of_y((size // 2, size // 2)) == tuple(out.shape[2:])


def test_conv_spec_rank3():
    conv = nn.Conv3d(1, 64, 3)
    spec = ops.ConvSpec.from_module(conv)
    assert spec.rank == 3 and spec.taps == 27 and spec.y_of_x((128, 128, 128)) == (126, 126, 126)   # GAN_final.py:167-169


@pytest.mark.parametrize("n", [1, 2, 5, 2097152])
@pytest.mark.parametrize("q", [0, 1.0, 37.5, 99.0, 100])
def test_percentile_rank_selection_matches_numpy_positions(n, q):
    lo, hi, frac = T.percentile_ranks(n, q)
    assert (lo, hi, frac) == ot.percentile_ranks(n, q)
    pos = q / 100.0 * (n - 1)
    assert lo == int(np.floor(pos)) and 0 <= lo <= hi <= n - 1 and hi - lo in (0, 1) and abs(lo + frac - pos) < 1e-9
    if q in (0, 100) or n == 1:
        assert hi == lo and frac == 0          # exact percentiles need one order statistic (min / max fast path)


def test_load_from_checkpoint_resolves_hparams_like_the_reference(tmp_path):
    """inferrence.py:97-106 passes channels/width/height/depth, an hparams.yaml and img_shape next to the checkpoint."""
    import mpgan
    torch.manual_seed(0)
    m = mpgan.GAN(1, 32, 32, g_lr=1e-3)
    ckpt = str(tmp_path / "m.ckpt")
    m.save_checkpoint(ckpt)
    yml = tmp_path / "hparams.yaml"
    yml.write_text("d_lr: 0.002\nb1: 0.4\nlatent_dim: 100\n")
    back = mpgan.GAN.load_from_checkpoint(channels=1, width=32, height=32, checkpoint_path=ckpt, hparams_file=str(yml),
                                          img_shape=(32, 32), strict=False)
    assert back.hparams.g_lr == 1e-3 and back.hparams.d_lr == 0.002 and back.hparams.b1 == 0.4
    opts, scheds = back.configure_optimizers()
    assert len(opts) == 2 and scheds == []
    with pytest.raises(RuntimeError, match="channels"):
        torch.save({"state_dict": m.state_dict()}, str(tmp_path / "bare.ckpt"))
        mpgan.GAN.load_from_checkpoint(str(tmp_path / "bare.ckpt"))


def test_flat_adam_is_a_torch_optimizer_with_adams_state_layout():
    """GAN_final.py:298-308 returns two torch.optim.Adam; pytorch-lightning's toggle_optimizer walks
    ``optimizer.param_groups`` and its checkpoints store ``optimizer.state_dict()``."""
    import mpgan
    torch.manual_seed(0)
    m = mpgan.GAN(1, 32, 32, g_lr=1e-3, d_lr=2e-3, b1=0.4)
    (og, od), _ = m.configure_optimizers()
    for opt, net, lr in ((og, m.generator, 1e-3), (od, m.discriminator, 2e-3)):
        assert isinstance(opt, torch.optim.Optimizer) and len(opt.param_groups) == 1
        g = opt.param_groups[0]
        assert g["lr"] == lr and g["betas"] == (0.4, 0.999) and g["eps"] == 1e-8
        assert [id(p) for p in g["params"]] == [id(p) for p in net.parameters()]
        sd = opt.state_dict()
        assert sd["state"] == {} and sd["param_groups"][0]["params"] == list(range(len(g["params"])))
        ref = torch.optim.Adam(net.parameters(), lr=lr, betas=(0.4, 0.999)).state_dict()
        assert set(sd["param_groups"][0].keys()) >= {"lr", "betas", "eps", "weight_decay", "amsgrad", "params"}
        assert sd["param_groups"][0]["params"] == ref["param_groups"][0]["params"]
    for p in og.param_groups[0]["params"]:     # toggle_optimizer semantics reach the network's own parameters
        p.requires_grad = False
    assert not any(p.requires_grad for p in m.generator.parameters()) and all(p.requires_grad for p in m.discriminator.parameters())
    with pytest.raises(RuntimeError, match="CUDA"):
        og.step()                               # no CPU fallback: the fused Adam kernel needs the device buffers


def test_monai_key_remap_both_ways():
    from mpgan.nets import remap_monai_keys
    legacy = {"generator.model.0.model.0.conv.unit0.norm.weight": 1, "generator.model.0.model.0.conv.unit1.act.weight": 2,
              "generator.model.0.model.2.0.norm.running_var": 3, "discriminator.model_conv.1.weight": 4,
              "generator.model.0.model.0.residual.weight": 5}
    adn = remap_monai_keys(legacy, "adn")
    assert set(adn) == {"generator.model.0.model.0.conv.unit0.adn.N.weight", "generator.model.0.model.0.conv.unit1.adn.A.weight",
                        "generator.model.0.model.2.0.adn.N.running_var", "discriminator.model_conv.1.weight",
                        "generator.model.0.model.0.residual.weight"}
    assert remap_monai_keys(adn, "legacy") == legacy and remap_monai_keys(legacy, "legacy") == legacy


def test_label_constants_are_never_evicted():
    """ADVICE r1: a captured graph holds raw pointers to the label tensors of its batch size."""
    import mpgan
    m = mpgan.GAN(1, 32, 32)
    a = m._consts(4, "cpu")
    b = m._consts(3, "cpu")
    assert m._consts(4, "cpu")[0] is a[0] and m._consts(3, "cpu")[1] is b[1]
    assert float(a[1][0]) == pytest.approx(0.9) and a[0].shape == (4, 1) and b[2].shape == (3, 1)


def test_entry_point_names_and_data_module_message():
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("ref_entry", os.path.join(root, "code", "GAN", "GAN.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for name in ("GAN", "CasNetGenerator", "Discriminator", "PatchDiscriminator", "HumanBrainDataModule", "transforms"):
        assert hasattr(mod, name), name
    with pytest.raises(NotImplementedError, match="private dataset"):
        mod.HumanBrainDataModule()


def test_gan_is_a_lightning_module_when_lightning_is_importable(tmp_path):
    """pytorch-lightning is absent from this image, so a minimal stand-in package is put on the path of a SUBPROCESS:
    mpgan.GAN must then derive from its LightningModule, call save_hyperparameters like GAN_final.py:231 and keep the
    reference's surface."""
    import os
    import subprocess
    import sys
    pkg = tmp_path / "pytorch_lightning"
    pkg.mkdir()
    (pkg / "__init__.py").write_text(
        "import inspect\nimport torch.nn as nn\n"
        "class _HP(dict):\n    __getattr__ = dict.__getitem__\n"
        "class LightningModule(nn.Module):\n"
        "    def __init__(self):\n        super().__init__()\n        self._hparams = _HP()\n        self.trainer = None\n"
        "    @property\n    def hparams(self):\n        return self._hparams\n"
        "    def save_hyperparameters(self, *names):\n"
        "        loc = inspect.currentframe().f_back.f_locals\n"
        "        for n in names:\n            self._hparams[n] = loc[n]\n"
        "    def log(self, *a, **k):\n        pass\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys; sys.path[:0] = [%r, %r, %r]\n"
            "import pytorch_lightning as pl, mpgan, torch\n"
            "m = mpgan.GAN(1, 32, 32, g_lr=1e-3)\n"
            "assert isinstance(m, pl.LightningModule) and mpgan.gan.HAVE_LIGHTNING\n"
            "assert m.hparams.g_lr == 1e-3 and m.hparams.one_sided_label_value == 0.9 and m.hparams.latent_dim == 100\n"
            "opts, sch = m.configure_optimizers()\n"
            "assert all(isinstance(o, torch.optim.Optimizer) for o in opts)\n"
            "p = mpgan.GAN(1, 32, 32, variant='perceptual'); assert p.hparams.g_lr == 2e-4\n"
            "print('ok')\n") % (str(tmp_path), os.path.join(root, "cross-modality-minipig-gan_b200"), root)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]


def test_rounding_matched_oracle_rounds_where_the_bf16_mode_does():
    """oracle/rounding.py: weights land on the bf16 grid, forward differs from fp32 by the cascade's rounding floor,
    and the instrumented copy leaves the original untouched."""
    from oracle.nets import CasNetGenerator as OGen, Discriminator as ODis
    from oracle.rounding import bf16_matched, rnd
    from oracle.gan import synthetic_batch
    torch.manual_seed(0)
    g = OGen((1, 32, 32), 2, 2)
    w0 = g.model[0].model[0].conv.unit0.conv.weight.detach().clone()
    m = bf16_matched(g)
    assert torch.equal(g.model[0].model[0].conv.unit0.conv.weight, w0)
    wm = m.model[0].model[0].conv.unit0.conv.weight
    assert torch.equal(wm, rnd(wm)) and not torch.equal(wm, w0)
    x = synthetic_batch(2, 2, 32, seed=1)["t1w"]
    with torch.no_grad():
        e = float((m(x) - g(x)).norm() / g(x).norm())
    assert 1e-3 < e < 2e-1, e
    d = ODis((1, 32, 32), dims=2, spatial=32)
    with torch.no_grad():
        ed = float((bf16_matched(d)(x) - d(x)).norm() / d(x).norm())
    assert 0 < ed < 1e-2, ed
    t = torch.tensor([1.0, 1.0 + 2 ** -12, 1.0 + 2 ** -10])
    assert torch.equal(rnd(t, "tf32"), torch.tensor([1.0, 1.0, 1.0 + 2 ** -10]))


def test_oracle_ref_recipe_copies_only_into_oracle_ref(tmp_path, monkeypatch):
    """build_ref copies exactly the reference's two files of the path, verbatim, into the git-ignored oracle/_ref.
    A stand-in reference tree (the two files plus one that must not be copied) replaces the reference checkout,
    which is not part of this repository."""
    from oracle import build_ref, ref_shim
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src, dst = tmp_path / "reference", tmp_path / "_ref"
    for rel in build_ref.FILES + ("code/inferrence.py",):
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_text(f"# {rel}\n")
    monkeypatch.setattr(build_ref, "REFERENCE_ROOT", str(src))
    monkeypatch.setattr(build_ref, "REF_COPY_ROOT", str(dst))
    assert build_ref.build(verbose=False)
    assert sorted(str(p.relative_to(dst)) for p in dst.rglob("*") if p.is_file()) == sorted(build_ref.FILES)
    for rel in build_ref.FILES:
        assert (dst / rel).read_text() == (src / rel).read_text()
    monkeypatch.setattr(build_ref, "REFERENCE_ROOT", str(tmp_path / "absent"))
    assert not build_ref.build(verbose=False)
    assert os.path.relpath(ref_shim.REF_COPY_ROOT, root) == os.path.join("oracle", "_ref")
    gi = open(os.path.join(root, ".gitignore")).read()
    assert "oracle/_ref/" in gi
