"""Generate tests/golden/boundary.npz by running the REAL reference wrapper methods of VQImageSegmTextureModel
(models/vqgan_model.py encode / decode / forward_step / training_step / optimize_parameters, unbound, on the stand-in
``self`` of oracle/ref_loader.vq_top_wrapper) around the REAL reference Encoder / Decoder / VectorQuantizerTexture /
Discriminator and models/losses/vqgan_loss.py, on the CPU, with LPIPS stubbed to zero.

Recorded, for the reduced nets and inputs of tests/test_gpu_boundary.py:
  * forward_step in eval mode under no_grad: the decoded pixels, the codebook loss, the continual indices;
  * optimize_parameters at step R.TINY_VQGAN_TRAIN["step"] with the global CPU RNG seeded R.VQGAN_TRAIN_AUG_SEED
    (DiffAugment's draws): the logged losses, the adaptive weight, the smallest distance of a discriminator
    pre-activation to its LeakyReLU kink, and per gradient tensor its norm, its largest magnitude and a fixed
    sample of R.GRAD_SAMPLE entries (full gradients would be tens of MB); decoder.conv_out.weight after Adam.

Run where the reference sources are available:  python oracle/make_golden_boundary.py
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import golden_recipes as R  # noqa: E402
from oracle import ref_loader as RL  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _grad_record(out, prefix, name, g):
    g = g.detach().reshape(-1)
    out[f"{prefix}norm/{name}"] = g.norm().numpy()
    out[f"{prefix}max/{name}"] = g.abs().max().numpy()
    out[f"{prefix}sample/{name}"] = g[R.grad_sample_index(g.numel(), name)].numpy().copy()


def main():
    torch.set_num_threads(8)
    cfg = R.TINY_VQGAN_TRAIN
    opt = R.boundary_opt()
    ns = RL.install("reference", wrappers=("vqgan_model",))
    with contextlib.redirect_stdout(io.StringIO()):
        w = RL.vq_top_wrapper(ns, opt, "cpu", with_disc=True, ndf=cfg["ndf"], disc_layers=cfg["disc_layers"])
    w.configure_optimizers()
    for name, seed in R.BOUNDARY_SEEDS:
        mod = getattr(w, name)
        mod.load_state_dict(R.fill_state_dict(R.spec_of(mod), seed), strict=True)
    cb = R.codebooks(106, 18, cfg["n_embed"], cfg["embed_dim"], "trained")
    with torch.no_grad():
        for k, emb in enumerate(w.quantize.embedding_list):
            emb.weight.copy_(cb[k])
    data = R.boundary_data()
    out = {}

    for n in ("encoder", "decoder", "quantize", "quant_conv", "post_quant_conv"):
        getattr(w, n).eval()
    x, mask = w.feed_data(data)
    with torch.no_grad():
        dec, diff = w.forward_step(x, mask)
        _, _, (_, cont, _) = w.encode(x, mask)
    out.update(fwd_dec=dec.numpy(), fwd_diff=diff.numpy(), fwd_cont=cont.numpy())

    margins = []
    hooks = [mod.register_forward_pre_hook(lambda m_, inp: margins.append(float(inp[0].detach().abs().min())))
             for mod in w.disc.main if isinstance(mod, torch.nn.LeakyReLU)]
    torch.manual_seed(R.VQGAN_TRAIN_AUG_SEED)
    w.optimize_parameters(data, cfg["step"])
    for h in hooks:
        h.remove()
    out["kink_margin"] = np.float32(min(margins))
    for k in ("nll_loss", "g_loss", "codebook_loss"):
        out[k] = np.float32(w.log_dict[k])
    out["d_weight"] = np.float32(w.log_dict["d_weight"].item())
    out["d_loss"] = np.float32(w.log_dict["d_loss"].item())
    n_g = 0
    for name in ("encoder", "decoder", "quantize", "quant_conv", "post_quant_conv"):
        for k, p in getattr(w, name).named_parameters():
            if p.grad is not None and float(p.grad.abs().max()) > 0.0:
                _grad_record(out, "g", f"{name}.{k}", p.grad)
                n_g += 1
    for k, p in w.disc.named_parameters():
        _grad_record(out, "d", k, p.grad)
    out["conv_out_after_adam"] = w.decoder.conv_out.weight.detach().numpy().copy()
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, "boundary.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "generator tensors", n_g, "kink margin", float(out["kink_margin"]),
          {k: float(out[k]) for k in ("nll_loss", "g_loss", "codebook_loss", "d_weight", "d_loss")})


if __name__ == "__main__":
    main()
