"""The drop-in against what the reference's own wrappers did with it installed (SURVEY.md 8b / a19), on CPU through the
test-only emulated backend.  tests/golden/dropin.npz (tests/golden/make_golden_dropin.py) holds what the reference
did: the names ``install()`` rebinds in each of its modules, the state_dict layout and ``initialize_weights`` draws of
the networks its wrappers build, and one epoch of its UNMODIFIED ``trainprocess`` loop (model/modelUnet.py:90-205:
``model(x) -> loss -> dice_coeff -> zero_grad/backward/AdamW.step``, checkpoint written) on two synthetic 8-bit
images.  Here that loop is restated step for step over the drop-in and must reproduce the reference's run."""
import os
import sys
import types

import numpy as np
import pytest
import torch
from torch.utils.data import DataLoader

import pytorchdeeplearing_b200 as b200
from pytorchdeeplearing_b200 import runtime
from emu_backend import EmuBackend
from conftest import GOLDEN

INIT_SEED = 5          # the seed make_golden_dropin.py draws the reference's initialize_weights with


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(GOLDEN, "dropin.npz")))


@pytest.fixture()
def emu():
    runtime._set_backend_for_testing(EmuBackend())
    prev = runtime.get_precision()
    runtime.set_precision("fp32")
    yield
    b200.uninstall()
    runtime._set_backend_for_testing(None)
    runtime.set_precision(prev)


def fingerprints(tensors):
    return np.array([[v.double().sum().item(), (v.double() ** 2).sum().item()] for v in tensors])


def layout(module):
    return [f"{k}:{','.join(map(str, v.shape))}" for k, v in module.state_dict().items()]


def train_images():
    """the two 32x32 uint8 images and masks of the reference run (written there as PNG files and read back by its
    dataset class)"""
    rng = np.random.RandomState(0)
    imgs, masks = [], []
    for _ in range(2):
        imgs.append((rng.rand(32, 32) * 255).astype(np.uint8))
        masks.append(((rng.rand(32, 32) > 0.7) * 255).astype(np.uint8))
    return imgs, masks


def test_install_rebinds_and_uninstall_restores(gold, emu, monkeypatch):
    """Stand-ins for the reference's modules, each binding the names the reference module binds (to placeholders)."""
    mods = {}
    for key, names in gold.items():
        if key.startswith("bind/"):
            m = types.ModuleType(key[len("bind/"):])
            for n in names:
                setattr(m, n, type(n, (), {}))
            monkeypatch.setitem(sys.modules, m.__name__, m)
            mods[m.__name__] = m
    mv, mu, ml, mm = (mods[n] for n in ("model.modelVNet", "model.modelUnet", "model.losses", "model.metric"))
    before = {(name, n): getattr(m, n) for name, m in mods.items() for n in gold["bind/" + name]}
    n = b200.install()
    assert n == int(gold["install_count"]) and n >= 20
    assert mv.VNet3d is b200.VNet3d and mv.VNet2d is b200.VNet2d
    assert mu.UNet2d is b200.UNet2d and mu.UNet3d is b200.UNet3d
    assert mv.MutilDiceLoss is b200.MutilDiceLoss and mu.BinaryFocalLoss is b200.BinaryFocalLoss
    assert ml.MutilCrossEntropyDiceLoss is b200.MutilCrossEntropyDiceLoss
    assert mv.dice_coeff is b200.dice_coeff and mm.multiclass_dice_coeff is b200.multiclass_dice_coeff
    for name, attr in before:
        assert getattr(mods[name], attr) is getattr(b200, attr), (name, attr)
    assert b200.install() == 0                                   # idempotent
    b200.uninstall()
    assert all(getattr(mods[name], attr) is obj for (name, attr), obj in before.items())


def test_wrappers_construct_with_dropin(gold, emu):
    """The reference's wrappers build ``VNet3d(1, 2)`` (MutilVNet3dModel, model/modelVNet.py:710-733), ``UNet2d(1, 1)``
    (BinaryUNet2dModel) and ``VNet2d(1, 1)`` (BinaryVNet2dModel); with the drop-in installed they get the drop-in
    classes, which must have the reference networks' state_dict (names, order, shapes) and take the same draws from
    ``initialize_weights`` (isinstance dispatch, module order)."""
    for key, args in (("VNet3d", (1, 2)), ("UNet2d", (1, 1)), ("VNet2d", (1, 1))):
        m = getattr(b200, key)(*args)
        assert layout(m) == list(gold["spec/" + key]), key
        torch.manual_seed(INIT_SEED)
        m.apply(b200.initialize_weights)
        assert np.allclose(fingerprints(m.state_dict().values()), gold["init/" + key], rtol=1e-12, atol=1e-12), key
        if key == "VNet3d":
            sd = m.state_dict()
            assert len(sd) == 128 and sum(v.numel() for v in sd.values()) == 9492658      # SURVEY.md App. A
            assert list(sd)[:4] == ["in_tr.conv1.weight", "in_tr.conv1.bias", "in_tr.conv2.weight", "in_tr.conv2.bias"]
            assert torch.all(m.in_tr.bn1.weight == 1) and torch.all(m.out_tr.conv.bias == 0)
    assert type(b200.VNet2d(1, 1)) is b200.VNet2d and len(b200.UNet2d(1, 1).state_dict()) == 64


def test_reference_trainprocess_runs_unchanged_on_the_dropin(gold, emu, tmp_path):
    """BASELINE.json config 1 shape of path: BinaryUNet2dModel(32, 32, 1, 1, batch_size=2).trainprocess for one epoch
    (model/modelUnet.py:90-205), in its order of generator draws: the wrapper builds UNet2d(1, 1) after
    ``torch.manual_seed(0)``; the trainer applies initialize_weights, creates AdamW(lr=1e-3) and two shuffling loaders
    of the z-scored images (datasetModelSegwithopencv), runs each batch as model(x) -> BinaryDiceLoss -> dice_coeff ->
    zero_grad/backward/step, then a validation pass, and saves the state_dict when the validation Dice beats 0.
    Weights at the optimizer's creation, losses, Dice, checkpoint and ``predict`` equal the reference's own run."""
    from oracle import staging
    imgs, masks = train_images()
    x = staging.zscore_u8(np.stack(imgs))
    y = staging.labels_from_u8(np.stack(masks), binarize=False)
    data = [{"image": x[i], "label": y[i]} for i in range(2)]
    torch.manual_seed(0)
    model = b200.UNet2d(1, 1)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    model.apply(b200.initialize_weights)
    lossfn = b200.BinaryDiceLoss()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    assert np.allclose(fingerprints(model.parameters()), gold["train/init"], rtol=1e-12, atol=1e-12)
    train_loader = DataLoader(data, shuffle=True, batch_size=2, num_workers=0)
    val_loader = DataLoader(data, shuffle=True, batch_size=2, num_workers=0)
    losses, dice = [], []
    model.train()
    for batch in train_loader:
        xb, yb = batch["image"], batch["label"]
        yb[yb != 0] = 1
        logit, pred = model(xb)
        loss = lossfn(logit, yb)
        losses.append(loss.item())
        dice.append(float(b200.dice_coeff(pred, yb)))
        opt.zero_grad()
        loss.backward()
        opt.step()
    model.eval()
    with torch.no_grad():
        for batch in val_loader:
            xb, yb = batch["image"], batch["label"]
            yb[yb != 0] = 1
            logit, pred = model(xb)
            losses.append(lossfn(logit, yb).item())
            dice.append(float(b200.dice_coeff(pred, yb)))
    assert np.allclose(losses, gold["train/loss"], rtol=1e-6, atol=1e-7), (losses, gold["train/loss"])
    assert np.allclose(dice, gold["train/dice"], rtol=1e-6, atol=1e-7), (dice, gold["train/dice"])
    assert dice[-1] > 0                       # the trainer writes the checkpoint only when the validation Dice beats 0
    ckpt = tmp_path / "BinaryUNet2d.pth"
    torch.save(model.state_dict(), str(ckpt))
    sd = torch.load(str(ckpt))
    assert list(sd.keys()) == list(before.keys()) == list(gold["train/names"]) and len(sd) == 64
    assert all(torch.isfinite(v).all() for v in sd.values())
    changed = sum(int(not torch.equal(sd[k], before[k])) for k in sd)
    assert changed > 32                                          # initialize_weights + one AdamW step moved them
    assert np.allclose(fingerprints(sd.values()), gold["train/final"], rtol=1e-6, atol=1e-9)
    with torch.no_grad():                                        # the wrapper's own predict (modelUnet.py:207-228)
        _, out = model(torch.zeros(1, 1, 32, 32))
    pred = ((out[0].squeeze().numpy() > 0.5) * 255).astype(np.uint8)
    assert pred.shape == (32, 32) and pred.dtype == np.uint8
    assert np.array_equal(pred, gold["train/predict"])
