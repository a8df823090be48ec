"""GPU parity of the index-prediction path (UNet guidance encoder + 18-head FCN + per-texture argmax, and the
whole sample_and_refine decode around it) through libt2h, against the fixture from the real reference classes
and against the torch fp32 restatement.  Tolerance 1e-3 relative on logits/features; indices must be equal
wherever the reference's top-2 logit margin exceeds the logit tolerance (a sub-tolerance difference can
legitimately flip an argmax)."""
import contextlib
import io
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import golden_recipes as R

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "index_pred.npz")
TOL = 1e-3


def _ops():
    from text2human_b200 import ops
    ops.set_precision("fp32")
    return ops


def _rel(got, ref):
    got = torch.as_tensor(got).double().cpu()
    ref = torch.as_tensor(ref).double().cpu()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def _join(planes):
    return planes.float().sum(0)


@pytest.mark.parametrize("shape", [(2, 32, 16, 64), (1, 4, 2, 512), (3, 2, 2, 1024), (2, 6, 10, 8)])
def test_maxpool_and_bilinear_conversions(cuda, shape):
    ops = _ops()
    x = torch.randn(shape, device=cuda)
    xn = x.permute(0, 3, 1, 2)
    got = _join(ops.f32_to_planes(x, ops.CVT_MAXPOOL2)).permute(0, 3, 1, 2)
    assert _rel(got, F.max_pool2d(xn, 2)) < 1e-6
    got = _join(ops.f32_to_planes(x, ops.CVT_BILINEAR2X)).permute(0, 3, 1, 2)
    want = F.interpolate(xn, scale_factor=2, mode="bilinear", align_corners=False)
    assert got.shape == want.shape and _rel(got, want) < 1e-5


@pytest.mark.parametrize("N,H,W,Cin,Cout,k", [(2, 32, 16, 256, 64, 3), (2, 2, 1, 512, 1024, 3), (1, 4, 2, 512, 512, 3),
                                               (3, 8, 4, 128, 256, 3), (2, 4, 2, 1024, 512, 1), (2, 32, 16, 128, 64, 1),
                                               (2, 32, 16, 64, 1152, 3), (2, 16, 8, 16, 8, 3)])
def test_conv_bn_relu_module(cuda, N, H, W, Cin, Cout, k):
    """ConvModule = conv (no bias) -> eval BatchNorm -> ReLU as one tap-GEMM, incl. the 2x1 / 4x2 maps of the
    deepest UNet stages and the 1x1 convs after the bilinear upsample"""
    ops = _ops()
    from text2human_b200.index_pred_arch import ConvModule
    cm = ConvModule(Cin, Cout, k, padding=k // 2)
    cm.load_state_dict(R.fill_state_dict(R.spec_of(cm), 3), strict=True)
    cm = cm.to(cuda).eval()
    x = R.latent(4, (N, Cin, H, W)).to(cuda)
    with torch.no_grad():
        want = torch.relu(cm.bn(cm.conv(x)))
    a = ops.nchw_to_planes(x)
    got = cm.forward_planes(a, planes_out=False).permute(0, 3, 1, 2)
    assert _rel(got, want) < TOL
    got_p = _join(cm.forward_planes(a, planes_out=True)).permute(0, 3, 1, 2)
    assert _rel(got_p, want) < TOL
    assert float(got.min()) >= 0.0


def test_grouped_gemm_with_per_group_bias_and_argmax(cuda):
    ops = _ops()
    G, M, ch, ncls, T = 18, 700, 64, 512, 2
    y = torch.randn(M, G * ch, device=cuda)
    w = torch.randn(G, ncls, ch, device=cuda) / 8
    b = torch.randn(G, ncls, device=cuda)
    yp = ops.split_planes(y, T)
    a = yp.view(T, M, G, ch).permute(0, 2, 1, 3)
    got = ops.bmm_nt(a, ops.split_planes(w, T), bias_col=b)
    want = torch.einsum("mgc,gnc->gmn", y.view(M, G, ch).double(), w.double()) + b.double()[:, None, :]
    assert got.shape == (G, M, ncls) and _rel(got, want) < 1e-4
    head = torch.randint(0, G, (M,), device=cuda)
    head[::7] = 20
    head[1::7] = -1
    lg = got.clone()
    lg[3, 5, 100] = lg[3, 5, 400] = 1e4                              # a tie: the lowest index wins
    head[5] = 3
    idx = ops.argmax_heads(lg, head)
    ok = (head >= 0) & (head < G)
    want_idx = lg[head.clamp(0, G - 1), torch.arange(M, device=cuda)].argmax(-1)
    assert torch.equal(idx[ok], want_idx[ok]) and bool((idx[~ok] == -1).all()) and int(idx[5]) == 100


def _mirror(unet_cfg, fcn_cfg, cuda):
    from text2human_b200.index_pred_arch import MultiHeadFCNHead, UNet
    u, f = UNet(**unet_cfg), MultiHeadFCNHead(**fcn_cfg)
    sdu, sdf = R.fill_state_dict(R.spec_of(u), 91), R.fill_state_dict(R.spec_of(f), 92)
    u.load_state_dict(sdu, strict=True)
    f.load_state_dict(sdf, strict=True)
    return u.to(cuda).eval(), f.to(cuda).eval(), sdu, sdf


def test_unet_and_fcn_heads_match_reference_fixture(cuda):
    _ops()
    gold = R.load_golden(GOLD)
    u, f, _, _ = _mirror(R.TINY_UNET, R.TINY_FCN, cuda)
    x = R.latent(93, (2, R.TINY_UNET["in_channels"], 32, 16), 1.0, "feature_top").to(cuda)
    dec = u(x)
    for i, d in enumerate(dec):
        assert _rel(d, gold[f"dec{i}"]) < TOL, i
    logits = torch.stack(f(dec))
    assert logits.shape == gold["logits"].shape and _rel(logits, gold["logits"]) < TOL


def test_real_size_index_prediction_matches_restatement(cuda):
    """UNet(256 -> 64..1024) + MultiHeadFCNHead(64, 64, 512 classes) on [B,256,32,16]: logits and the
    per-texture argmax (bot_index_prediction, sample_model.py:183-213)"""
    _ops()
    from oracle import indexpred_ref as IR
    from text2human_b200.index_pred_arch import bot_index_prediction
    u, f, sdu, sdf = _mirror(R.REAL_UNET, R.REAL_FCN, cuda)
    B = 2
    x = R.latent(95, (B, 256, 32, 16), 1.0, "feature_top")
    mask = R.blocky_mask(96, B, 512, 256, 64, extra_ids=(20,))
    with torch.no_grad():
        want_logits = torch.stack(IR.fcn_heads(sdf, IR.unet(sdu, x)))           # [18,B,512,32,16]
        want_list = IR.bot_index_prediction(sdu, sdf, x, mask)
    logits = torch.stack(f(u(x.to(cuda))))
    assert _rel(logits, want_logits) < TOL
    got_list = bot_index_prediction(u, f, x.to(cuda), mask.to(cuda))
    assert len(got_list) == 18
    top2 = want_logits.topk(2, dim=2).values
    margin_ok = (top2[:, :, 0] - top2[:, :, 1]) > 2 * TOL * want_logits.abs().max()   # [18,B,32,16]
    n_checked = 0
    for k in range(18):
        g, w = got_list[k].cpu(), want_list[k]
        assert g.shape == (B, 32, 16) and g.dtype == torch.int64
        assert bool(((g >= 0) == (w >= 0)).all())
        sel = (w >= 0) & margin_ok[k]
        assert torch.equal(g[sel], w[sel])
        n_checked += int(sel.sum())
    assert n_checked > 0.9 * int((torch.stack(want_list) >= 0).sum())


def test_image_packing_and_write_out(cuda, tmp_path):
    """save_image's quantisation (torchvision: mul(255).add_(0.5).clamp_(0,255).to(uint8)) on the GPU, bit-exact,
    incl. the fused (x+1)/2 map and clamp; files round-trip through PIL"""
    ops = _ops()
    from PIL import Image
    from text2human_b200.pipeline import save_images
    x = torch.rand(2, 3, 37, 21, device=cuda) * 1.2 - 0.1            # some values outside [0,1]
    want = x.clamp(0, 1).mul(255).add_(0.5).clamp_(0, 255).permute(0, 2, 3, 1).to(torch.uint8)
    assert torch.equal(ops.pack_u8(x), want)
    y = x * 2 - 1
    want2 = ((y + 1) / 2).clamp(0, 1).mul(255).add_(0.5).clamp_(0, 255).permute(0, 2, 3, 1).to(torch.uint8)
    got2 = ops.pack_u8(y, scale=0.5, shift=0.5)
    assert int((got2.int() - want2.int()).abs().max()) <= 1          # the fused affine map rounds once, torch twice
    save_images(x, str(tmp_path), ["a.png", "b.png"])
    back = np.asarray(Image.open(tmp_path / "b.png"))
    assert np.array_equal(back, want[1].cpu().numpy())


def _sample_opt():
    from bench import HIER_OPT, SAMPLER_OPT
    opt = dict(HIER_OPT)
    opt.update(SAMPLER_OPT)
    opt.update(bot_codebook_spatial_size=2, index_pred_encoder_in_channels=256, index_pred_fc_in_channels=64,
               index_pred_fc_in_index=4, index_pred_fc_channels=64, index_pred_fc_num_convs=1,
               index_pred_fc_concat_input=False, index_pred_fc_dropout_ratio=0.1, index_pred_fc_num_classes=512,
               index_pred_fc_align_corners=False, segm_double_z=False, segm_z_channels=32, segm_resolution=512,
               segm_in_channels=24, segm_out_ch=24, segm_ch=64, segm_ch_mult=[1, 1, 2, 2, 4], segm_num_res_blocks=1,
               segm_attn_resolutions=[16], segm_dropout=0.0, segm_num_segm_classes=24, segm_n_embed=1024,
               segm_embed_dim=32)
    return opt


def test_sample_and_refine_end_to_end_plumbing(cuda):
    """parsing map + texture mask -> images through every stage of SampleFromParsingModel (segm tokenizer,
    4 diffusion steps of the sampler, both codebook gathers, UNet/FCN index prediction, DecoderRes, Decoder);
    the stages' numerics are covered individually, this checks they compose: shapes, ranges, reproducibility
    under a seeded generator (to rounding: the fused GroupNorm statistics are accumulated with atomics, so the
    conv stacks are order-dependent in the last fp32 bits), and that a different seed changes the result"""
    _ops()
    from text2human_b200.pipeline import SampleFromParsingModel
    torch.manual_seed(41)
    with contextlib.redirect_stdout(io.StringIO()):
        m = SampleFromParsingModel(_sample_opt())
    for sub, seed in ((m.index_pred_guidance_encoder, 43), (m.index_pred_decoder, 44)):
        sub.load_state_dict(R.fill_state_dict(R.spec_of(sub), seed), strict=True)
    m = m.to(cuda).eval()
    B = 2
    segm = R.blocky_mask(45, B, 512, 256, 16, n_ids=24).to(cuda)
    mask = R.blocky_mask(46, B, 512, 256, 64).to(cuda)
    imgs = []
    for seed in (7, 7, 8):
        g = torch.Generator(device=cuda).manual_seed(seed)
        imgs.append(m.sample_and_refine(segm, mask, sample_steps=4, generator=g))
    img = imgs[0]
    assert img.shape == (B, 3, 512, 256) and img.dtype == torch.float32
    assert bool(torch.isfinite(img).all()) and float(img.min()) >= 0.0 and float(img.max()) <= 1.0
    assert float((imgs[0] - imgs[1]).abs().max()) < 1e-4
    assert float((imgs[0] - imgs[2]).abs().max()) > 1e-2


def test_sample_and_refine_decode_matches_restatement(cuda):
    """sampled top tokens -> image in [0,1] through the whole refine chain (sample_model.py:215-246), with the
    reference's configs/sample_from_parsing.yml sizes, batched"""
    _ops()
    from oracle import indexpred_ref as IR
    from oracle import vqgan_ref
    from text2human_b200.pipeline import SampleFromParsingModel
    opt = _sample_opt()
    torch.manual_seed(31)
    with contextlib.redirect_stdout(io.StringIO()):
        m = SampleFromParsingModel(opt)
    for name in ("index_pred_guidance_encoder", "index_pred_decoder"):
        sub = getattr(m, name)
        sub.load_state_dict(R.fill_state_dict(R.spec_of(sub), 33), strict=True)
    for q, seed, n_e, d in ((m.top_quantize, 34, 1024, 256), (m.bot_quantize, 35, 512, 1024)):
        cb = R.codebooks(seed, 18, n_e, d, "trained")
        for k, e in enumerate(q.embedding_list):
            e.weight.data.copy_(cb[k])
    m = m.to(cuda).eval()
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    B = 2
    mask = R.blocky_mask(36, B, 512, 256, 64)
    tex = F.interpolate(mask, (32, 16), mode="nearest")[:, 0].long()
    top = torch.randint(0, 1024, (B, 32, 16), generator=torch.Generator().manual_seed(2))
    top_list = [torch.where(tex == k, top, torch.full_like(top, -1)) for k in range(18)]
    img = m.decode_top_tokens([t.to(cuda) for t in top_list], mask.to(cuda))
    assert img.shape == (B, 3, 512, 256) and float(img.min()) >= 0.0 and float(img.max()) <= 1.0
    with torch.no_grad():
        cbt = torch.stack([sd[f"top_quantize.embedding_list.{k}.weight"] for k in range(18)])
        cbb = torch.stack([sd[f"bot_quantize.embedding_list.{k}.weight"] for k in range(18)])
        qt = vqgan_ref.conv(sd, "top_post_quant_conv", vqgan_ref.codebook_entry_texture(cbt, top_list, mask,
                                                                                         (B, 32, 16, 256)), padding=0)
        sdu = {k[len("index_pred_guidance_encoder."):]: v for k, v in sd.items()
               if k.startswith("index_pred_guidance_encoder.")}
        sdf = {k[len("index_pred_decoder."):]: v for k, v in sd.items() if k.startswith("index_pred_decoder.")}
        want_logits = torch.stack(IR.fcn_heads(sdf, IR.unet(sdu, qt)))
        # teacher-forced: the restatement decodes the bottom indices the CUDA path predicted, and those are
        # checked against the restatement's own argmax wherever its margin is clear
        got_bot = m.bot_index_prediction(vqgan_ref.conv(sd, "top_post_quant_conv", vqgan_ref.codebook_entry_texture(
            cbt, top_list, mask, (B, 32, 16, 256)), padding=0).to(cuda), mask.to(cuda))
        got_bot = [g.cpu() for g in got_bot]
        want_bot = IR.bot_index_prediction(sdu, sdf, qt, mask)
        top2 = want_logits.topk(2, dim=2).values
        margin_ok = (top2[:, :, 0] - top2[:, :, 1]) > 2 * TOL * want_logits.abs().max()
        for k in range(18):
            sel = (want_bot[k] >= 0) & margin_ok[k]
            assert torch.equal(got_bot[k][sel], want_bot[k][sel])
        qb = vqgan_ref.codebook_entry_texture(cbb, got_bot, mask, (B, 32, 16, 256), ps=2)
        res = vqgan_ref.decoder_res(sd, vqgan_ref.conv(sd, "bot_post_quant_conv", qb, padding=0), "bot_decoder_res.")
        want = ((vqgan_ref.decoder(sd, qt, "decoder.", bot_h=res) + 1) / 2).clamp(0, 1)
    assert _rel(img, want) < TOL
