"""Evaluation path and checkpoint loading (harness/eval_synth.py, SURVEY.md 8(f) N4) against fixtures produced by the
reference's own evaluate.py functions (tests/golden/make_eval_golden.py) and against the semantics of
utils/pyt_utils.py:47-85 `load_model`."""
import os
import sys
from collections import OrderedDict

import numpy as np
import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from harness import eval_synth as ev  # noqa: E402

G = np.load(os.path.join(ROOT, "tests", "golden", "eval_sliding.npz"))


def golden_net():
    classes = int(G["classes"])
    net = nn.Sequential(nn.Conv2d(3, 8, 3, stride=2, padding=1), nn.ReLU(), nn.Conv2d(8, classes, 3, stride=2, padding=1)).double().eval()
    net.load_state_dict({k[len("net."):]: torch.from_numpy(G[k]) for k in G.files if k.startswith("net.")})

    class ListNet(nn.Module):
        def __init__(self, m):
            super().__init__()
            self.m = m

        def forward(self, x):
            y = self.m(x)
            return [y, y * 0]
    return ListNet(net), classes


def test_tile_grid_covers_the_image_and_stays_inside():
    for (H, W, th, tw) in ((50, 70, 32, 32), (1024, 2048, 769, 769), (20, 45, 32, 32), (769, 769, 769, 769)):
        wins = ev.tile_grid((H, W), (th, tw))
        cover = np.zeros((H, W), dtype=int)
        for (y1, y2, x1, x2) in wins:
            assert 0 <= y1 < y2 <= H and 0 <= x1 < x2 <= W and y2 - y1 <= th and x2 - x1 <= tw
            cover[y1:y2, x1:x2] += 1
        assert cover.min() >= 1
    assert len(ev.tile_grid((1024, 2048), (769, 769))) == 8          # 2 x 4 windows per Cityscapes image (evaluate.py:106-110)


@pytest.mark.parametrize("tile_batch", [1, 3])
def test_predict_sliding_matches_reference_function(tile_batch):
    net, classes = golden_net()
    tile = tuple(int(t) for t in G["tile"])
    got = ev.predict_sliding(net, torch.from_numpy(G["image"]), tile, classes, tile_batch=tile_batch)
    assert got.shape == G["sliding"].shape
    np.testing.assert_allclose(got.numpy(), G["sliding"], rtol=0, atol=1e-5)
    small = ev.predict_sliding(net, torch.from_numpy(G["image_small"]), tile, classes, tile_batch=tile_batch)
    np.testing.assert_allclose(small.numpy(), G["sliding_small"], rtol=0, atol=1e-5)     # window smaller than the tile: zero padding


def test_predict_whole_and_mirrored_average_match_reference_functions():
    net, classes = golden_net()
    tile = tuple(int(t) for t in G["tile"])
    img = torch.from_numpy(G["image"])
    np.testing.assert_allclose(ev.predict_whole(net, img).numpy(), G["whole"], rtol=0, atol=1e-5)
    # evaluate.py:171 mirrors the flipped prediction back along axis 1; unflip_axis=1 reproduces that line, the default is axis 2 (W)
    ref_like = ev.predict_multiscale(net, img, tile, [1.0], classes, True, unflip_axis=1)
    np.testing.assert_allclose(ref_like.numpy(), G["multi_flip"], rtol=0, atol=1e-5)
    plain = ev.predict_multiscale(net, img, tile, [1.0], classes, False)
    np.testing.assert_allclose(plain.numpy(), G["sliding"], rtol=0, atol=1e-5)
    sym = ev.predict_multiscale(net, img, tile, [1.0], classes, True)
    mirrored = ev.predict_multiscale(net, img.flip(3), tile, [1.0], classes, True)
    np.testing.assert_allclose(sym.numpy(), mirrored.flip(2).numpy(), rtol=0, atol=1e-6)   # mirror-equivariant with the W un-flip


def test_zoom_is_scipy_order1_zoom():
    got = ev.zoom_bilinear(torch.from_numpy(G["image"]), 0.75)
    np.testing.assert_allclose(got.numpy(), G["zoom075"], rtol=0, atol=1e-6)
    assert ev.zoom_bilinear(torch.from_numpy(G["image"]), 1.0).shape == G["image"].shape


def test_confusion_matrix_and_mean_iou():
    cm = ev.get_confusion_matrix(torch.from_numpy(G["cm_gt"]), torch.from_numpy(G["cm_pred"]), int(G["classes"]))
    np.testing.assert_array_equal(cm.numpy(), G["cm"])
    c = G["cm"]
    tp, pos, res = np.diag(c), c.sum(1), c.sum(0)
    want = (tp / np.maximum(1.0, pos + res - tp)).mean()              # evaluate.py:268-274
    got, per_class = ev.mean_iou(cm)
    assert abs(got - want) < 1e-12 and per_class.shape == (int(G["classes"]),)
    # labels beyond the last (gt, pred) pair seen leave trailing zero rows, as the reference's bounds check does (evaluate.py:190)
    cm2 = ev.get_confusion_matrix(torch.tensor([0, 1]), torch.tensor([0, 0]), 4)
    assert cm2.shape == (4, 4) and cm2.sum() == 2 and cm2[1, 0] == 1


def test_evaluate_batch_drops_ignored_pixels():
    net, classes = golden_net()
    img = torch.from_numpy(G["image"])
    label = torch.randint(0, classes, (1, 50, 70), generator=torch.Generator().manual_seed(1))
    label[:, :7] = 255
    cm = ev.evaluate_batch(net, img, label, (32, 32), classes)
    assert cm.sum().item() == 43 * 70


class _Tiny(nn.Module):
    def __init__(self):
        super().__init__()
        self.a = nn.Linear(3, 2)
        self.b = nn.BatchNorm1d(2)


def test_load_model_semantics(tmp_path):
    src = _Tiny()
    with torch.no_grad():
        src.a.weight.fill_(0.25)
    sd = src.state_dict()
    # 1. plain state dict; 2. wrapped in {'model': ...} on disk (pyt_utils.py:52-53)
    m, missing, unexpected = ev.load_model(_Tiny(), sd)
    assert not missing and not unexpected and torch.equal(m.a.weight, src.a.weight)
    f = tmp_path / "snap.pth"
    torch.save({"model": sd, "iter": 3}, f)
    m, missing, unexpected = ev.load_model(_Tiny(), str(f))
    assert not missing and not unexpected and torch.equal(m.a.weight, src.a.weight)
    # 3. is_restore: keys get the 'module.' prefix of a DataParallel wrapper (pyt_utils.py:58-63)
    wrapped = nn.DataParallel(_Tiny())               # with one visible GPU this moves the module to cuda:0
    m, missing, unexpected = ev.load_model(wrapped, sd, is_restore=True)
    assert not missing and not unexpected and torch.equal(m.module.a.weight.cpu(), src.a.weight)
    # 4. non-strict: missing and unexpected keys are reported, the rest is loaded (pyt_utils.py:65-77)
    part = OrderedDict((k, v) for k, v in sd.items() if not k.startswith("b."))
    part["head.extra"] = torch.zeros(1)
    m, missing, unexpected = ev.load_model(_Tiny(), part)
    assert unexpected == ["head.extra"] and set(missing) == {k for k in sd if k.startswith("b.")}
    assert torch.equal(m.a.weight, src.a.weight)
    # 5. a checkpoint saved from a wrapper loads into the bare network
    m, missing, unexpected = ev.load_model(_Tiny(), OrderedDict(("module." + k, v) for k, v in sd.items()))
    assert not missing and not unexpected and torch.equal(m.a.weight, src.a.weight)


def test_reference_style_checkpoint_fills_the_attention_module(tmp_path):
    """The released R=2 weights carry head.cca.{gamma, query_conv.*, key_conv.*, value_conv.*} (networks/ccnet.py:105,
    cc_attention/functions.py:19-24): a checkpoint with the reference's key set loads into the harness network with nothing
    missing and nothing unexpected, and the 7 operator tensors arrive in ccnet_b200.CrissCrossAttention."""
    from harness.ccnet_model import CCNet
    import ccnet_b200
    with torch.device("meta"):
        shapes = {k: tuple(v.shape) for k, v in CCNet(num_classes=19, recurrence=2).state_dict().items()}
    net = CCNet(num_classes=19, layers=(1, 1, 1, 1), recurrence=2)
    own = net.state_dict()
    ckpt = OrderedDict(("module." + k, torch.full_like(v, 0.5) if v.is_floating_point() else v.clone()) for k, v in own.items())
    torch.save({"model": ckpt}, tmp_path / "CS_scenes_synth.pth")
    net, missing, unexpected = ev.load_model(net, str(tmp_path / "CS_scenes_synth.pth"))
    assert not missing and not unexpected
    cca_keys = sorted(k for k in own if k.startswith("head.cca."))
    assert cca_keys == sorted("head.cca." + s for s in ("gamma", "query_conv.weight", "query_conv.bias", "key_conv.weight",
                                                         "key_conv.bias", "value_conv.weight", "value_conv.bias"))
    assert type(net.head.cca) is ccnet_b200.CrissCrossAttention
    assert net.head.cca.gamma.item() == 0.5 and net.head.cca.value_conv.weight.flatten()[0].item() == 0.5
    assert all(k in shapes for k in cca_keys)
