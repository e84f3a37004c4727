"""The harness network (harness/ccnet_model.py, used for BASELINE configs[2] / [3]) names and shapes every tensor exactly like
the reference's Seg_Model (its layout is stored in tests/golden/ccnet_state_dict.npz by tests/golden/make_network_golden.py)."""
import os

import numpy as np
import torch

from conftest import GOLDEN_DIR


def test_harness_network_matches_reference_state_dict():
    d = np.load(os.path.join(GOLDEN_DIR, "ccnet_state_dict.npz"))
    a = {str(k): tuple(int(n) for n in s[:nd]) for k, s, nd in zip(d["keys"], d["shapes"], d["ndim"])}
    from harness.ccnet_model import CCNet
    with torch.device("meta"):
        ours = CCNet(num_classes=19, recurrence=2)
    b = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    assert list(a) == list(b), (sorted(set(a) ^ set(b))[:20])
    assert a == b, [k for k in a if k in b and a[k] != b[k]][:10]
    assert sum(p.numel() for p in ours.parameters()) == int(d["n_params"])
    assert ours.recurrence == int(d["recurrence"])


def test_harness_network_forward_shapes_on_cpu_fallback_free():
    """Tiny structural check without the operator: the head's attention needs CUDA, so only the backbone + dsn run here."""
    from harness.ccnet_model import CCNet
    net = CCNet(num_classes=5, layers=(1, 1, 1, 1), recurrence=1).eval()
    x = torch.randn(1, 3, 65, 65)
    with torch.no_grad():
        y = torch.relu(net.bn1(net.conv1(x)))
        y = torch.relu(net.bn2(net.conv2(y)))
        y = net.maxpool(torch.relu(net.bn3(net.conv3(y))))
        y = net.layer3(net.layer2(net.layer1(y)))
        assert y.shape == (1, 1024, 9, 9)                # 65 -> 33 -> 17 -> 9: output stride 8
        assert net.dsn(y).shape == (1, 5, 9, 9)
        assert net.layer4(y).shape == (1, 2048, 9, 9)
