"""Host-side logic of the drop-in layer that needs no GPU: override detection for the README's
extension mechanism, the bit-packed resident dataset, and the C header / ctypes agreement."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_builtin_losses_are_marked_and_overrides_detected():
    import ns_gan, mm_gan, w_gan, w_gp_gan, ls_gan, dra_gan, be_gan, ra_gan, f_gan, fisher_gan, info_gan
    for m, t in ((ns_gan, "NSGANTrainer"), (mm_gan, "MMGANTrainer"), (w_gan, "WGANTrainer"), (w_gp_gan, "WGPGANTrainer"),
                 (ls_gan, "LSGANTrainer"), (dra_gan, "DRAGANTrainer"), (be_gan, "BEGANTrainer"), (ra_gan, "RaNSGANTrainer"),
                 (f_gan, "fGANTrainer"), (fisher_gan, "FisherGANTrainer"), (info_gan, "InfoGANTrainer")):
        T = getattr(m, t)
        assert getattr(T.train_D, "_gm_builtin", False) and getattr(T.train_G, "_gm_builtin", False), t

    class Mine(ns_gan.NSGANTrainer):                      # README.md:31: "edit train_D and train_G"
        def train_D(self, images):
            return torch.zeros(())

    model = ns_gan.NSGAN(784, 400, 20)
    assert not ns_gan.NSGANTrainer(model, [], [], [])._has_custom_step()
    assert Mine(model, [], [], [])._has_custom_step()


def test_forward_without_engine_fails_loudly():
    """No eager / CPU path: the modules refuse to run until a CUDA engine exists."""
    import ns_gan
    from gm_b200 import GmError
    model = ns_gan.NSGAN(784, 400, 20)
    with pytest.raises(GmError, match="CUDA engine"):
        model.G(torch.randn(4, 20))


def test_device_dataset_bit_packing_matches_numpy():
    from gm_b200.gan_api import DeviceDataset
    g = torch.Generator().manual_seed(1)
    imgs = (torch.rand(37, 1, 28, 28, generator=g) < 0.13).float()
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(imgs, torch.zeros(37)), batch_size=10, shuffle=True)
    dd = DeviceDataset.from_loader(loader)
    assert dd is not None and len(dd) == 4 and dd.bits.shape == (37, 98) and dd.bits.dtype == torch.uint8
    back = np.unpackbits(dd.bits.cpu().numpy(), axis=1)[:, :784]        # MSB first, row-aligned: the kernel's layout
    assert np.array_equal(back, imgs.view(37, -1).numpy().astype(np.uint8))
    dd.seed(5)
    a = dd.sample()
    dd.seed(5)
    b = dd.sample()
    assert torch.equal(a, b) and a.unique().numel() == 10 and int(a.max()) < 37
    # grey-level data cannot be packed: the Trainer then keeps the reference's process_batch path
    loader2 = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(torch.rand(8, 1, 28, 28), torch.zeros(8)), batch_size=4)
    assert DeviceDataset.from_loader(loader2) is None
    assert DeviceDataset.from_loader([(imgs, None)]) is None               # plain list iterators: nothing to cache


def test_every_header_function_has_ctypes_argtypes():
    """include/gm_b200.h and gm_b200/_lib.py stay in step: each declared entry point gets its argument
    types declared (a missing declaration would pass Python ints as 32-bit C ints)."""
    hdr = open(os.path.join(ROOT, "include", "gm_b200.h")).read()
    names = sorted(set(re.findall(r"\b(gm_[a-z0-9_]+)\s*\(", hdr)))
    src = open(os.path.join(ROOT, "generative-models_b200", "gm_b200", "_lib.py")).read()
    no_args = {"gm_version"}
    missing = [n for n in names if n not in no_args and ("L.%s.argtypes" % n) not in src]
    assert not missing, missing


def test_reference_made_checkpoints_load_into_the_dropin_modules():
    """tests/golden/ref_*.ckpt were written by the REFERENCE's own save_model (tests/golden/make_golden.py
    make_checkpoints): same state_dict keys, shapes and values load into the drop-in modules (src/ns_gan.py:283-290)."""
    import numpy as np
    import ns_gan
    import vae as V
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    sd = torch.load(os.path.join(here, "ref_nsgan_h32_z8.ckpt"))
    model = ns_gan.NSGAN(784, 32, 8)
    assert list(sd.keys()) == list(model.state_dict().keys())
    model.load_state_dict(sd)
    for k, v in model.state_dict().items():
        assert torch.equal(v, sd[k]), k
    assert list(np.load(os.path.join(here, "ref_nsgan_h32_z8_outputs.npz"))["keys"]) == list(sd.keys())
    vsd = torch.load(os.path.join(here, "ref_vae_h32_z8.ckpt"))
    vmodel = V.VAE(784, 32, 8)
    assert list(vsd.keys()) == list(vmodel.state_dict().keys())
    vmodel.load_state_dict(vsd)
    for k, v in vmodel.state_dict().items():
        assert torch.equal(v, vsd[k]), k


def test_dcgan_dropin_surface_without_a_gpu(monkeypatch):
    """dc_gan.py mirrors the NSGAN class surface for the conv model the README recommends (README.md:68,96): usual DCGAN
    state_dict keys / shapes, the reference's attributes, and a loud failure instead of a CPU fallback."""
    import dc_gan
    from gm_b200 import GmError
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)     # the same refusal on a machine that has a GPU
    model = dc_gan.DCGAN(image_size=64 * 64 * 3, hidden_dim=16, z_dim=100)
    sd = model.state_dict()
    assert sd["G.l1.weight"].shape == (100, 128, 4, 4) and sd["G.l5.weight"].shape == (16, 3, 4, 4)
    assert sd["D.l1.weight"].shape == (16, 3, 4, 4) and sd["D.l5.weight"].shape == (1, 128, 4, 4)
    assert "G.bn1.running_mean" in sd and "D.bn4.weight" in sd and "D.bn1.weight" not in sd
    assert (model.z_dim, model.image_size, model.hidden_dim, model.shape) == (100, 12288, 16, 64)
    it = [(torch.zeros(2, 3, 64, 64), torch.zeros(2))]
    tr = dc_gan.DCGANTrainer(model, it, it, it)
    assert tr.Glosses == [] and tr.num_epochs == 0 and tr.name == "DCGAN"
    with pytest.raises(GmError):
        model.G(torch.randn(2, 100))
    with pytest.raises(GmError):
        dc_gan.DCGAN(image_size=784)


def test_space_to_depth_conv_identity():
    """DESIGN 6b `Next`: the k4 s2 p1 convolution, its two gradients and the transposed convolution as four ROW-SHIFTED GEMMs
    on the space-to-depth matrix (tools/s2d_conv_prototype.py) agree with torch to rounding, also for odd grid extents."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("s2d", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "s2d_conv_prototype.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    for kw in (dict(), dict(seed=1, B=3, H=4, W=4, C=8, Co=16), dict(seed=2, B=1, H=10, W=6, C=2, Co=3)):
        err = m.check(**kw)
        assert max(err.values()) < 1e-12, (kw, err)
