"""Generate tests/golden/sampler_train.npz by running the REAL reference training loss
(/root/reference/models/transformer_model.py TransformerTextureAwareModel._train_loss / q_sample /
sample_time, unbound, on a stand-in ``self`` that carries only the attributes they read) around the REAL
reference TransformerMultiHead, then ``loss.backward()`` and one real ``torch.optim.Adam`` step.

The random draws the reference makes (t, the q_sample mask) are recorded in the fixture so that the
restatement (oracle/transformer_ref.train_loss) and the CUDA trainer can be fed the same ones.
Run in the build container only:  python oracle/make_golden_train.py
"""
import importlib.util
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import golden_recipes as R  # noqa: E402

REF = "/root/reference/models"
OUT = os.path.join(ROOT, "tests", "golden")


def _load(modname, path):
    spec = importlib.util.spec_from_file_location(modname, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[modname] = mod
    spec.loader.exec_module(mod)
    return mod


def main():
    torch.set_num_threads(8)
    # `import models` pulls mmcv/lpips; register bare packages and load the three files by path
    for name in ("models", "models.archs"):
        sys.modules.setdefault(name, types.ModuleType(name))
    _load("models.archs.vqgan_arch", os.path.join(REF, "archs", "vqgan_arch.py"))
    tr = _load("models.archs.transformer_arch", os.path.join(REF, "archs", "transformer_arch.py"))
    tm = _load("models.transformer_model", os.path.join(REF, "transformer_model.py"))
    Model = tm.TransformerTextureAwareModel

    cfg = R.TINY_TRANSFORMER
    net = tr.TransformerMultiHead(**cfg)
    net.load_state_dict(R.fill_state_dict(R.spec_of(net), 71), strict=True)
    x_0, gt_list, segm, tex = R.sampler_train_batch(72)

    rec = {}
    fake = types.SimpleNamespace(num_timesteps=1000, mask_id=cfg["codebook_size"], mask_schedule="random",
                                 loss_type="reweighted_elbo", _denoise_fn=net, segm_tokens=segm,
                                 texture_tokens=tex)

    def sample_time(b, device, method="uniform"):
        t, pt = Model.sample_time(fake, b, device, method)
        rec["t"] = t.clone()
        return t, pt

    def q_sample(x_0, x_0_gt_list, t):
        x_t, ign, mask = Model.q_sample(fake, x_0=x_0, x_0_gt_list=x_0_gt_list, t=t)
        rec["mask"] = mask.clone()
        return x_t, ign, mask

    fake.sample_time, fake.q_sample = sample_time, q_sample
    torch.manual_seed(73)
    net.train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, weight_decay=0)
    loss, vb = Model._train_loss(fake, x_0, gt_list)
    opt.zero_grad()
    loss.backward()
    out = {"t": rec["t"].numpy(), "mask": rec["mask"].numpy(), "loss": loss.detach().numpy(),
           "vb_loss": vb.detach().numpy()}
    for k, p in net.named_parameters():
        out["grad/" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy().copy()
    opt.step()
    for k, p in net.named_parameters():
        out["param1/" + k] = p.detach().numpy().copy()
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, "sampler_train.npz")
    R.save_golden(path, out)
    print(path, os.path.getsize(path), "loss", float(loss), "vb", float(vb), "t", rec["t"].tolist(),
          "masked", int(rec["mask"].sum()))


if __name__ == "__main__":
    main()
