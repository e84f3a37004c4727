"""Row (b) of the scope table: the reference's networks/ccnet.py imports `CrissCrossAttention` from the `cc_attention` package
(networks/ccnet.py:13) and builds its RCCA head around it (networks/ccnet.py:105).  With this repository on the path that name
is the B200 operator, and the head it builds has the reference's parameter layout (tests/golden/ccnet_state_dict.npz, taken
from the reference's own Seg_Model by tests/golden/make_network_golden.py)."""
import os
from collections import OrderedDict

import numpy as np
import torch

from conftest import GOLDEN_DIR, load_golden

CCA_PARAMS = ("gamma", "query_conv.weight", "query_conv.bias", "key_conv.weight", "key_conv.bias", "value_conv.weight",
              "value_conv.bias")


def reference_head_shapes():
    d = np.load(os.path.join(GOLDEN_DIR, "ccnet_state_dict.npz"))
    return {str(k): tuple(int(n) for n in s[:nd]) for k, s, nd in zip(d["keys"], d["shapes"], d["ndim"])
            if k.startswith("head.cca.")}


def test_reference_network_builds_on_the_b200_operator():
    import cc_attention
    import ccnet_b200
    from harness.ccnet_model import CCNet
    assert cc_attention.CrissCrossAttention is ccnet_b200.CrissCrossAttention      # what networks/ccnet.py:13 imports
    want = reference_head_shapes()
    assert set(want) == {"head.cca." + n for n in CCA_PARAMS}
    with torch.device("meta"):
        model = CCNet(num_classes=19, recurrence=2)                                 # networks/ccnet.py:199-205
    assert type(model.head.cca) is ccnet_b200.CrissCrossAttention                   # networks/ccnet.py:105
    got = {k: tuple(v.shape) for k, v in model.state_dict().items() if k.startswith("head.cca.")}
    assert got == want
    assert want["head.cca.query_conv.weight"] == (64, 512, 1, 1) and want["head.cca.value_conv.weight"] == (512, 512, 1, 1)
    assert model.recurrence == 2


def test_released_checkpoint_keys_load_into_the_module():
    """utils/pyt_utils.py:47-85 load_model(strict=False) path: a state dict with the reference's head.cca.* entries restores
    the B200 module's parameters (SURVEY 8f N4: on-disk format adjacent to the path).  The values are the reference module's
    own parameters (tests/golden/cca_smoke_*.npz, C=64); the C=512 key set and shapes are those of the reference's network."""
    import ccnet_b200
    from harness import eval_synth as ev

    def wrap(head):
        wrapper = torch.nn.Module()
        wrapper.head = torch.nn.Module()
        wrapper.head.cca = head
        return wrapper

    g = load_golden("smoke_2x64x5x6")
    ref = {n: torch.from_numpy(g["p_" + n]) for n in CCA_PARAMS}
    head = ccnet_b200.CrissCrossAttention(64)
    out, missing, unexpected = ev.load_model(wrap(head), OrderedDict(("head.cca." + n, v) for n, v in ref.items()))
    assert out.head.cca is head and not missing and not unexpected
    for n, v in ref.items():
        assert torch.equal(head.state_dict()[n], v), n

    torch.manual_seed(0)
    ckpt = OrderedDict((k, torch.randn(s)) for k, s in reference_head_shapes().items())
    head = ccnet_b200.CrissCrossAttention(512)
    out, missing, unexpected = ev.load_model(wrap(head), ckpt)
    assert out.head.cca is head and not missing and not unexpected
    for k, v in ckpt.items():
        assert torch.equal(head.state_dict()[k[len("head.cca."):]], v), k
