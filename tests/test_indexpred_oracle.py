"""CPU: the index-prediction restatement (oracle/indexpred_ref) against the fixture made from the real
reference UNet / MultiHeadFCNHead classes (oracle/make_golden_indexpred.py), the mirror's checkpoint ABI,
and the BatchNorm folding the CUDA path relies on (host logic)."""
import os

import numpy as np
import torch

import golden_recipes as R
from oracle import indexpred_ref as IR

GOLD = os.path.join(os.path.dirname(__file__), "golden", "index_pred.npz")


def _tiny_state():
    from text2human_b200.index_pred_arch import MultiHeadFCNHead, UNet
    u, f = UNet(**R.TINY_UNET), MultiHeadFCNHead(**R.TINY_FCN)
    return u, f, R.fill_state_dict(R.spec_of(u), 91), R.fill_state_dict(R.spec_of(f), 92)


def test_restatement_matches_reference_fixture():
    gold = R.load_golden(GOLD)
    u, f, sdu, sdf = _tiny_state()
    x = R.latent(93, (2, R.TINY_UNET["in_channels"], 32, 16), 1.0, "feature_top")
    with torch.no_grad():
        dec = IR.unet(sdu, x)
        logits = torch.stack(IR.fcn_heads(sdf, dec))
    for i, d in enumerate(dec):
        want = torch.from_numpy(gold[f"dec{i}"])
        assert d.shape == want.shape and (d - want).abs().max() <= 1e-5 * want.abs().max(), i
    want = torch.from_numpy(gold["logits"])
    assert (logits - want).abs().max() <= 1e-5 * want.abs().max()


def test_mirror_keeps_the_checkpoint_abi_of_the_real_size_nets():
    from text2human_b200.index_pred_arch import MultiHeadFCNHead, UNet
    gold = R.load_golden(GOLD)
    u, f = UNet(**R.REAL_UNET), MultiHeadFCNHead(**R.REAL_FCN)
    assert [f"{k}:{tuple(v.shape)}" for k, v in u.state_dict().items()] == list(gold["unet_keys"])
    assert [f"{k}:{tuple(v.shape)}" for k, v in f.state_dict().items()] == list(gold["fcn_keys"])


def test_batchnorm_folding_equals_eval_conv_bn():
    from text2human_b200.index_pred_arch import ConvModule
    cm = ConvModule(8, 16, 3, padding=1)
    cm.load_state_dict(R.fill_state_dict(R.spec_of(cm), 5), strict=True)
    cm.eval()
    x = R.latent(6, (2, 8, 5, 7))
    with torch.no_grad():
        want = torch.relu(cm.bn(cm.conv(x)))
        w, b = cm.folded()
        got = torch.relu(torch.nn.functional.conv2d(x, w, b, padding=1))
    assert (got - want).abs().max() <= 1e-5


def test_bot_index_prediction_restatement_returns_reference_structure():
    u, f, sdu, sdf = _tiny_state()
    x = R.latent(93, (2, R.TINY_UNET["in_channels"], 32, 16), 1.0, "feature_top")
    mask = R.blocky_mask(94, 2, 512, 256, 64, extra_ids=(20,))
    out = IR.bot_index_prediction(sdu, sdf, x, mask)
    tex = torch.nn.functional.interpolate(mask, (32, 16), mode="nearest")[:, 0].long()
    assert len(out) == 18 and all(o.shape == (2, 32, 16) and o.dtype == torch.int64 for o in out)
    stacked = torch.stack(out)
    for k in range(18):
        assert bool(((stacked[k] >= 0) == (tex == k)).all())        # exactly its own texture's positions
    assert bool((stacked[:, tex == 20] == -1).all())                 # ids outside 0..17 select no head
