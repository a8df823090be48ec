"""Generate tests/golden/index_pred.npz by running the REAL reference UNet / MultiHeadFCNHead classes
(/root/reference/models/archs/unet_arch.py, fcn_arch.py) on the deterministic recipes.

Those files import mmcv / mmseg (mmcv-full==1.2.1, mmsegmentation==0.9.0: absent here, no network), so the
handful of names they import are provided by stand-ins registered in sys.modules before loading them by
file path: `ConvModule` restates mmcv's published conv(bias=False) -> BatchNorm2d -> ReLU module with its
attribute names (`conv`, `bn`, `activate`), `build_upsample_layer` is the registry lookup that instantiates
the reference's own `InterpConv`, the rest are initialisers / loggers that the forward path never calls.
Everything structural (stage layout, pooling, upsampling, concatenation, heads) is the reference's code.

Run in the build container only:  python oracle/make_golden_indexpred.py
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import golden_recipes as R  # noqa: E402

REF = "/root/reference/models/archs"
OUT = os.path.join(ROOT, "tests", "golden")


class ConvModule(nn.Module):
    """mmcv.cnn.ConvModule 1.2.1 for (conv_cfg=None, norm_cfg=BN, act_cfg=ReLU, order conv-norm-act)"""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 bias="auto", conv_cfg=None, norm_cfg=None, act_cfg=dict(type="ReLU"), **kw):
        super().__init__()
        assert conv_cfg is None
        with_norm = norm_cfg is not None
        if bias == "auto":
            bias = not with_norm
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias)
        self.with_norm, self.with_act = with_norm, act_cfg is not None
        if with_norm:
            assert norm_cfg["type"] == "BN"
            self.bn = nn.BatchNorm2d(out_channels)
        if self.with_act:
            assert act_cfg["type"] == "ReLU"
            self.activate = nn.ReLU(inplace=True)

    def forward(self, x):
        x = self.conv(x)
        if self.with_norm:
            x = self.bn(x)
        if self.with_act:
            x = self.activate(x)
        return x


class _Registry:
    def __init__(self):
        self.d = {}

    def register_module(self):
        def deco(cls):
            self.d[cls.__name__] = cls
            return cls
        return deco


def _stub_modules():
    reg = _Registry()

    def build_upsample_layer(cfg, *a, **kw):
        cfg = dict(cfg)
        return reg.d[cfg.pop("type")](*a, **kw, **cfg)

    def build_norm_layer(cfg, n):
        return "bn", nn.BatchNorm2d(n)

    def build_activation_layer(cfg):
        return nn.ReLU(inplace=True)

    noop = lambda *a, **k: None  # noqa: E731
    mods = {
        "mmcv": types.ModuleType("mmcv"),
        "mmcv.cnn": types.ModuleType("mmcv.cnn"),
        "mmcv.runner": types.ModuleType("mmcv.runner"),
        "mmcv.utils": types.ModuleType("mmcv.utils"),
        "mmcv.utils.parrots_wrapper": types.ModuleType("mmcv.utils.parrots_wrapper"),
        "mmseg": types.ModuleType("mmseg"),
        "mmseg.utils": types.ModuleType("mmseg.utils"),
        "mmseg.ops": types.ModuleType("mmseg.ops"),
    }
    c = mods["mmcv.cnn"]
    c.UPSAMPLE_LAYERS, c.ConvModule = reg, ConvModule
    c.build_activation_layer, c.build_norm_layer, c.build_upsample_layer = (build_activation_layer,
                                                                            build_norm_layer, build_upsample_layer)
    c.constant_init = c.kaiming_init = c.normal_init = noop
    mods["mmcv.runner"].load_checkpoint = noop
    mods["mmcv.utils.parrots_wrapper"]._BatchNorm = nn.modules.batchnorm._BatchNorm
    mods["mmseg.utils"].get_root_logger = noop
    mods["mmseg.ops"].resize = torch.nn.functional.interpolate
    sys.modules.update(mods)


def _load(name):
    spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(REF, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def build(unet_cfg, fcn_cfg):
    _stub_modules()
    un, fc = _load("unet_arch"), _load("fcn_arch")
    unet = un.UNet(**unet_cfg)
    fcn = fc.MultiHeadFCNHead(**fcn_cfg)
    unet.load_state_dict(R.fill_state_dict(R.spec_of(unet), 91), strict=True)
    fcn.load_state_dict(R.fill_state_dict(R.spec_of(fcn), 92), strict=True)
    return unet.eval(), fcn.eval()


def main():
    torch.set_num_threads(8)
    unet, fcn = build(R.TINY_UNET, R.TINY_FCN)
    x = R.latent(93, (2, R.TINY_UNET["in_channels"], 32, 16), 1.0, "feature_top")
    with torch.no_grad():
        dec = unet(x)
        logits = fcn(dec)
    out = {"logits": torch.stack(logits).numpy()}
    for i, d in enumerate(dec):
        out[f"dec{i}"] = d.numpy()
    # key/shape listings of the real-size nets (the checkpoint ABI the mirror must keep)
    unet_r, fcn_r = build(R.REAL_UNET, R.REAL_FCN)
    out["unet_keys"] = np.array([f"{k}:{tuple(v.shape)}" for k, v in unet_r.state_dict().items()])
    out["fcn_keys"] = np.array([f"{k}:{tuple(v.shape)}" for k, v in fcn_r.state_dict().items()])
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, "index_pred.npz")
    R.save_golden(path, out)
    print(path, os.path.getsize(path), [tuple(d.shape) for d in dec], len(out["unet_keys"]), len(out["fcn_keys"]))


if __name__ == "__main__":
    main()
