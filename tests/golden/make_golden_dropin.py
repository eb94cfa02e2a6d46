#!/usr/bin/env python
"""tests/golden/dropin.npz: what the reference's own wrappers do with the drop-in installed (tests/test_dropin_cpu.py).

    python tests/golden/make_golden_dropin.py <reference checkout>

Imports the UNMODIFIED reference tree (nothing of it is copied); the four I/O-only modules its ``model`` package
imports (SimpleITK, torchsummary, skimage, matplotlib) are replaced by inert stubs in ``sys.modules``.  Network, loss
and metric kernels are the drop-in's, run on CPU through the test-only emulated backend (tests/emu_backend.py).
Records:
  bind/<module>       the names of ``install()``'s table that each reference module binds, and ``install_count``
  spec/<net>, init/<net>
                      the state_dict layout ("name:shape") of the reference's own network as its wrapper builds it,
                      and per-tensor (sum, sum of squares) after ``torch.manual_seed(INIT_SEED)`` and the reference's
                      ``initialize_weights``
  train/*             BinaryUNet2dModel(32, 32, 1, 1, batch_size=2).trainprocess for one epoch over two synthetic
                      8-bit images (the PNG files the reference reads are written from the same arrays): per-tensor
                      fingerprints of the weights when the optimizer is created and of the saved checkpoint, the
                      train / validation losses and Dice, and the wrapper's ``predict`` of a zero image
"""
import importlib
import os
import sys
import tempfile
import types

import numpy as np
import torch

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

INIT_SEED = 5
# wrapper -> (reference network module, class, constructor arguments the wrapper passes)
NETS = {"VNet3d": ("networks.VNet3d", "VNet3d", (1, 2)), "UNet2d": ("networks.Unet2d", "UNet2d", (1, 1)),
        "VNet2d": ("networks.VNet2d", "VNet2d", (1, 1))}


def train_images():
    """the two 32x32 uint8 images and masks both the reference run and the test use"""
    rng = np.random.RandomState(0)
    imgs, masks = [], []
    for _ in range(2):
        imgs.append((rng.rand(32, 32) * 255).astype(np.uint8))
        masks.append(((rng.rand(32, 32) > 0.7) * 255).astype(np.uint8))
    return imgs, masks


def fingerprints(sd):
    return np.array([[v.double().sum().item(), (v.double() ** 2).sum().item()] for v in sd.values()])


def spec(module):
    return np.array([f"{k}:{','.join(map(str, v.shape))}" for k, v in module.state_dict().items()])


def _stub(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def import_reference(ref):
    sys.path.insert(0, ref)
    noop = lambda *a, **k: None
    _stub("SimpleITK", sitkLinear=1, sitkNearestNeighbor=0, GetImageFromArray=noop, WriteImage=noop,
          GetArrayFromImage=noop)
    _stub("torchsummary", summary=noop)
    sk = _stub("skimage")
    sk.metrics = _stub("skimage.metrics", structural_similarity=noop)
    mp = _stub("matplotlib", use=noop)

    class _Style:
        use = staticmethod(noop)
    mp.pyplot = _stub("matplotlib.pyplot", style=_Style, figure=noop, plot=noop, title=noop, xlabel=noop,
                      ylabel=noop, legend=noop, savefig=noop, close=noop, show=noop, imshow=noop, subplot=noop)
    pkg = types.ModuleType("model")
    pkg.__path__ = [os.path.join(ref, "model")]          # skip model/__init__.py (drags ResNet/GAN wrappers)
    sys.modules["model"] = pkg
    names = ["networks", "networks.VNet3d", "networks.VNet2d", "networks.Unet3d", "networks.Unet2d", "model.losses",
             "model.metric", "model.modelVNet", "model.modelUnet"]
    return {n: importlib.import_module(n) for n in names}


def main(ref):
    import cv2
    import pytorchdeeplearing_b200 as b200
    from pytorchdeeplearing_b200 import runtime
    inst = importlib.import_module("pytorchdeeplearing_b200.install")
    from emu_backend import EmuBackend

    torch.set_num_threads(1)
    mods = import_reference(ref)
    runtime._set_backend_for_testing(EmuBackend())
    runtime.set_precision("fp32")
    out = {}

    # ---- which names install() rebinds, module by module
    table = inst._NET_NAMES + inst._LOSS_NAMES + inst._METRIC_NAMES
    for modname in inst._MODULES:
        mod = sys.modules.get(modname)
        if mod is not None:
            out["bind/" + modname] = np.array([n for n in table if hasattr(mod, n)])
    out["install_count"] = np.array(b200.install())
    b200.uninstall()

    # ---- the reference's own networks: layout and initialiser
    class VNet3dFixed(mods["networks.VNet3d"].VNet3d):      # networks/VNet3d.py:127 reads self.feature
        feature = property(lambda self: self.features)
    for key, (modname, cls, args) in NETS.items():
        net = (VNet3dFixed if key == "VNet3d" else getattr(mods[modname], cls))(*args)
        out["spec/" + key] = spec(net)
        torch.manual_seed(INIT_SEED)
        net.apply(mods["networks"].initialize_weights)
        out["init/" + key] = fingerprints(net.state_dict())

    # ---- one epoch of the reference's trainprocess on the drop-in
    mu = mods["model.modelUnet"]
    b200.install()
    imgs, masks = train_images()
    with tempfile.TemporaryDirectory() as tmp:
        ip, mp = [], []
        for i, (im, mk) in enumerate(zip(imgs, masks)):
            ip.append(os.path.join(tmp, f"img{i}.png"))
            mp.append(os.path.join(tmp, f"mask{i}.png"))
            cv2.imwrite(ip[-1], im)
            cv2.imwrite(mp[-1], mk)
        torch.manual_seed(0)
        w = mu.BinaryUNet2dModel(32, 32, 1, 1, batch_size=2, loss_name="BinaryDiceLoss", use_cuda=False)
        seen = {"loss": [], "dice": []}
        adamw = mu.optim.AdamW

        class SnapshotAdamW(adamw):
            def __init__(self, params, **kw):
                params = list(params)
                seen["init"] = fingerprints({i: p.detach() for i, p in enumerate(params)})
                super().__init__(params, **kw)
        lossname = w._loss_function
        accuracy = w._accuracy_function

        def loss_function(name):
            fn = lossname(name)

            def record(z, y):
                v = fn(z, y)
                seen["loss"].append(v.item())
                return v
            return record

        def accuracy_function(name, pred, y):
            a = accuracy(name, pred, y)
            seen["dice"].append(float(a))
            return a
        w._loss_function, w._accuracy_function = loss_function, accuracy_function
        mu.optim.AdamW = SnapshotAdamW
        try:
            w.trainprocess(ip, mp, ip, mp, os.path.join(tmp, "out"), epochs=1, lr=1e-3)
        finally:
            mu.optim.AdamW = adamw
        sd = torch.load(os.path.join(tmp, "out", "BinaryUNet2d.pth"))
        ds = mu.datasetModelSegwithopencv(ip, mp, targetsize=(1, 32, 32))
        staged = [ds[i] for i in range(2)]
    from oracle import staging
    assert torch.equal(torch.stack([s["image"] for s in staged]), staging.zscore_u8(np.stack(imgs)))
    assert torch.equal(torch.stack([s["label"] for s in staged]), staging.labels_from_u8(np.stack(masks), False))
    out["train/names"] = np.array(list(sd))
    out["train/init"] = seen["init"]
    out["train/final"] = fingerprints(sd)
    out["train/loss"] = np.array(seen["loss"])            # [train step, validation pass]
    out["train/dice"] = np.array(seen["dice"])
    out["train/predict"] = w.predict(np.zeros((1, 32, 32), np.float32))
    b200.uninstall()
    np.savez_compressed(os.path.join(HERE, "dropin.npz"), **out)
    print({k: v.shape for k, v in out.items()})
    print("install_count", int(out["install_count"]), "loss", seen["loss"], "dice", seen["dice"])


if __name__ == "__main__":
    main(os.path.abspath(sys.argv[1]))
