"""The drop-in boundary SURVEY.md §8b states, exercised end to end: the B200 mirrors of the reference's modules
(`text2human_b200.vqgan_arch`, `.transformer_arch`) driven through the calls the reference's wrapper files make on
them, as ordinary autograd modules under stock PyTorch, against what the reference's own wrapper code computed on
its own modules (tests/golden/boundary.npz from oracle/make_golden_boundary.py, tests/golden/sample_fn.npz from
oracle/make_golden_sample.py):

  * VQImageSegmTextureModel.forward_step (vqgan_model.py:548)            pixels / codebook loss / indices
  * VQImageSegmTextureModel.optimize_parameters (:329-344, :444-488: loss.backward(), two torch.optim.Adam,
    calculate_adaptive_weight's autograd.grad, DiffAugment, hinge_d_loss)   losses, gradients, the Adam step
  * BaseSampleModel.sample_fn (sample_model.py:256)                         reveal schedule and tokens
"""
import contextlib
import io
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import golden_recipes as R

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _rel(got, ref):
    got, ref = got.double(), ref.double()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


class _MirrorWrapper:
    """The calls models/vqgan_model.py VQImageSegmTextureModel makes on its modules (encode, decode, forward_step,
    training_step with models/losses/vqgan_loss.py, optimize_parameters with the optimisers of
    configure_optimizers), issued on the mirrors.  LPIPS is stubbed to zero, as in the fixture.  DiffAugment runs on
    the host (oracle/vqgan_train_ref.diff_augment, pinned to the reference's) so that its draws come from the CPU
    generator in the order the fixture consumed them; autograd carries the gradient across the copies."""

    def __init__(self, opt, dev):
        from text2human_b200 import vqgan_arch as va
        self.opt, self.dev, self.log_dict = opt, dev, {}
        with contextlib.redirect_stdout(io.StringIO()):
            self.encoder = va.Encoder(ch=opt["ch"], num_res_blocks=opt["num_res_blocks"],
                                      attn_resolutions=opt["attn_resolutions"], ch_mult=opt["ch_mult"],
                                      in_channels=opt["in_channels"], resolution=opt["resolution"],
                                      z_channels=opt["z_channels"], double_z=opt["double_z"], dropout=opt["dropout"])
            self.decoder = va.Decoder(in_channels=opt["in_channels"], resolution=opt["resolution"],
                                      z_channels=opt["z_channels"], ch=opt["ch"], out_ch=opt["out_ch"],
                                      num_res_blocks=opt["num_res_blocks"], attn_resolutions=opt["attn_resolutions"],
                                      ch_mult=opt["ch_mult"], dropout=opt["dropout"], resamp_with_conv=True,
                                      give_pre_end=False)
        self.quantize = va.VectorQuantizerTexture(opt["n_embed"], opt["embed_dim"], beta=0.25)
        self.quant_conv = torch.nn.Conv2d(opt["z_channels"], opt["embed_dim"], 1)
        self.post_quant_conv = torch.nn.Conv2d(opt["embed_dim"], opt["z_channels"], 1)
        self.disc = va.Discriminator(opt["n_channels"], opt["ndf"], n_layers=opt["disc_layers"])
        for n in ("encoder", "decoder", "quantize", "quant_conv", "post_quant_conv", "disc"):
            setattr(self, n, getattr(self, n).to(dev))
        self.optimizer = torch.optim.Adam(
            list(self.encoder.parameters()) + list(self.decoder.parameters()) + list(self.quantize.parameters()) +
            list(self.quant_conv.parameters()) + list(self.post_quant_conv.parameters()), lr=opt["lr"])
        self.disc_optimizer = torch.optim.Adam(self.disc.parameters(), lr=opt["lr"])

    def feed_data(self, data):
        return data["image"].float().to(self.dev), data["texture_mask"].float().to(self.dev)

    def encode(self, x, mask):
        return self.quantize(self.quant_conv(self.encoder(x)), mask)

    def forward_step(self, x, mask):
        quant, diff, _ = self.encode(x, mask)
        return self.decoder(self.post_quant_conv(quant)), diff

    def _diff_augment(self, x):
        from oracle.vqgan_train_ref import diff_augment
        return diff_augment(x.cpu()).to(self.dev)

    def training_step(self, data, step):
        x, mask = self.feed_data(data)
        xrec, codebook_loss = self.forward_step(x, mask)
        nll_loss = torch.mean(torch.abs(x - xrec))
        xrec = self._diff_augment(xrec)
        g_loss = -torch.mean(self.disc(xrec))
        last = self.decoder.conv_out.weight
        rg = torch.autograd.grad(nll_loss, last, retain_graph=True)[0]
        gg = torch.autograd.grad(g_loss, last, retain_graph=True)[0]
        d_weight = torch.clamp(torch.norm(rg) / (torch.norm(gg) + 1e-4), 0.0, self.opt["disc_weight_max"]).detach()
        d_weight = d_weight * (1 if step >= self.opt["disc_start_step"] else 0.0)
        loss = nll_loss + d_weight * g_loss + codebook_loss
        self.log_dict.update(nll_loss=nll_loss.item(), g_loss=g_loss.item(), codebook_loss=codebook_loss.item(),
                             d_weight=float(d_weight))
        d_loss = None
        if step > self.opt["disc_start_step"]:
            logits_real = self.disc(self._diff_augment(x.detach()))
            logits_fake = self.disc(xrec.detach())
            d_loss = 0.5 * (torch.mean(F.relu(1.0 - logits_real)) + torch.mean(F.relu(1.0 + logits_fake)))
            self.log_dict["d_loss"] = d_loss.item()
        return loss, d_loss

    def optimize_parameters(self, data, step):
        for n in ("encoder", "decoder", "quantize", "quant_conv", "post_quant_conv"):
            getattr(self, n).train()
        loss, d_loss = self.training_step(data, step)
        self.optimizer.zero_grad()
        loss.backward()
        self.optimizer.step()
        if step > self.opt["disc_start_step"]:
            self.disc_optimizer.zero_grad()
            d_loss.backward()
            self.disc_optimizer.step()


def _fill(w):
    """the fixture's seeded weights, loaded through the wrapper's attributes"""
    for name, seed in R.BOUNDARY_SEEDS:
        mod = getattr(w, name)
        mod.load_state_dict({k: v.cuda() for k, v in R.fill_state_dict(R.spec_of(mod), seed).items()}, strict=True)
    cb = R.codebooks(106, 18, R.TINY_VQGAN_TRAIN["n_embed"], R.TINY_VQGAN_TRAIN["embed_dim"], "trained")
    with torch.no_grad():
        for k, emb in enumerate(w.quantize.embedding_list):
            emb.weight.copy_(cb[k])


def _check_grads(gold, prefix, named):
    """every gradient tensor the fixture lists: its norm, its largest magnitude and its sampled entries; gradients
    that vanish in exact arithmetic (a conv bias in front of a per-channel GroupNorm) are rounding noise in the
    reference as well: held to an absolute floor.  -> (worst relative error, tensors checked)"""
    keys = [k[len(prefix) + 5:] for k in gold.files if k.startswith(prefix + "norm/")]
    gmax = max(float(gold[f"{prefix}max/{k}"]) for k in keys)
    worst = 0.0
    for key in keys:
        g = named[key].grad
        assert g is not None, key
        g = g.detach().reshape(-1).double().cpu()
        want_max, want_norm = float(gold[f"{prefix}max/{key}"]), float(gold[f"{prefix}norm/{key}"])
        sample = torch.from_numpy(gold[f"{prefix}sample/{key}"]).double()
        got = g[R.grad_sample_index(g.numel(), key)]
        err = max(float((got - sample).abs().max()), abs(float(g.abs().max()) - want_max))
        if want_max < 1e-6 * gmax:
            assert err < 1e-5 * gmax, key
            continue
        e = max(err / want_max, abs(float(g.norm()) - want_norm) / want_norm)
        assert e < 1e-3, (key, e)
        worst = max(worst, e)
    return worst, len(keys)


def test_reference_vqgan_wrapper_calls_on_the_mirrors(cuda):
    from text2human_b200 import ops
    ops.set_precision("fp32")
    gold = np.load(os.path.join(GOLDEN, "boundary.npz"))
    data = R.boundary_data()
    wm = _MirrorWrapper(R.boundary_opt(), cuda)
    _fill(wm)

    # inference: forward_step under no_grad, eval mode (vqgan_model.py:493-506)
    for n in ("encoder", "decoder", "quantize", "quant_conv", "post_quant_conv"):
        getattr(wm, n).eval()
    x, mask = wm.feed_data(data)
    with torch.no_grad():
        dec_m, diff_m = wm.forward_step(x, mask)
        _, _, (_, cont_m, _) = wm.encode(x, mask)
    assert torch.equal(cont_m.cpu(), torch.from_numpy(gold["fwd_cont"]))
    assert _rel(dec_m.cpu(), torch.from_numpy(gold["fwd_dec"])) < 1e-3
    assert abs(float(diff_m) - float(gold["fwd_diff"])) <= 1e-3 * abs(float(gold["fwd_diff"]))

    # training: optimize_parameters with DiffAugment's draws from the fixture's seed.  The step's gradient is
    # discontinuous at the discriminator's LeakyReLU / hinge kinks; under this seed the reference run has no
    # pre-activation within the recorded margin of a kink.
    step = R.TINY_VQGAN_TRAIN["step"]
    margin = float(gold["kink_margin"])
    print(f"[boundary] DiffAugment seed {R.VQGAN_TRAIN_AUG_SEED}: min distance of a discriminator pre-activation to "
          f"its kink {margin:.2e}")
    assert margin > 3e-5
    before = {k: v.detach().clone() for k, v in wm.decoder.state_dict().items()}
    torch.manual_seed(R.VQGAN_TRAIN_AUG_SEED)
    wm.optimize_parameters(data, step)
    for k in ("nll_loss", "g_loss", "codebook_loss"):
        assert abs(wm.log_dict[k] - float(gold[k])) <= 2e-4 * max(1.0, abs(float(gold[k]))), k
    assert abs(wm.log_dict["d_weight"] - float(gold["d_weight"])) <= 2e-3 * float(gold["d_weight"])
    assert abs(wm.log_dict["d_loss"] - float(gold["d_loss"])) <= 2e-4
    named = {f"{n}.{k}": p for n in ("encoder", "decoder", "quantize", "quant_conv", "post_quant_conv")
             for k, p in getattr(wm, n).named_parameters()}
    worst, n_g = _check_grads(gold, "g", named)
    print(f"[boundary] training step on the mirrors: {n_g} generator tensors, worst gradient rel err {worst:.2e}")
    dworst, n_d = _check_grads(gold, "d", dict(wm.disc.named_parameters()))
    print(f"[boundary] {n_d} discriminator tensors, worst gradient rel err {dworst:.2e}")
    assert n_g > 200 and n_d >= 10
    # both Adam steps happened on the mirrors' own parameters
    after = wm.decoder.state_dict()
    assert any(not torch.equal(before[k], after[k]) for k in before)
    assert _rel(wm.decoder.conv_out.weight.detach().cpu(), torch.from_numpy(gold["conv_out_after_adam"])) < 1e-3


def test_reference_sample_fn_on_the_mirror_transformer(cuda):
    """BaseSampleModel.sample_fn (sample_model.py:256-328, restated by oracle/transformer_ref.sample_fn, which
    reproduces the fixture token for token on the reference transformer) with the mirror transformer on the GPU as
    its sampler_fn; the loop's draws stay on the CPU generator the fixture was recorded with: the same reveal
    schedule exactly, and the same tokens except where two candidates tie within float rounding of the logits."""
    from oracle import transformer_ref as TR
    from text2human_b200 import ops
    from text2human_b200.transformer_arch import TransformerMultiHead
    ops.set_precision("fp32")
    cfg = R.SAMPLE_TRANSFORMER
    net = TransformerMultiHead(**cfg)
    net.load_state_dict(R.fill_state_dict(R.spec_of(net), 81), strict=True)
    net = net.to(cuda).eval()
    segm, mask = R.sample_inputs(82, R.SAMPLE_BATCH)

    def sampler_fn(x, s, t):
        return [lg.cpu() for lg in net(x.to(cuda), s.to(cuda), t.to(cuda))]
    torch.manual_seed(83)
    with torch.no_grad():
        out, _ = TR.sample_fn(sampler_fn, segm, mask, cfg["latent_shape"], cfg["codebook_size"], R.SAMPLE_STEPS)
    got = torch.stack(out)
    want = torch.from_numpy(np.load(os.path.join(GOLDEN, "sample_fn.npz"))["lists"].astype(np.int64))
    assert got.shape == want.shape
    assert torch.equal(got >= 0, want >= 0)
    agree = float((got == want).float().mean())
    print(f"[boundary] reference sample_fn on the mirror transformer: {100 * agree:.3f} % of tokens identical")
    assert agree > 0.995
