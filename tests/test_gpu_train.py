"""GPU parity of the sampler training step (text2human_b200/transformer_train.py + csrc/train.cu) through the
C ABI: kernels against plain torch fp32, loss/gradients/Adam against the fixture made from the real
reference `_train_loss` (tests/golden/sampler_train.npz) and against autograd of the restatement at a
second shape.  Tolerance: 1e-3 relative (north_star) on each gradient tensor's max norm."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import golden_recipes as R

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "sampler_train.npz")
DEV = "cuda"


def _ops():
    from text2human_b200 import ops
    ops.set_precision("fp32")
    return ops


def _join(planes):
    return planes.float().sum(0)


def _rel(got, want):
    return float((got.double() - want.double()).abs().max() / (want.double().abs().max() + 1e-30))


# ----------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("shape", [(1, 64, 64), (3, 50, 72), (2, 512, 40), (2, 33, 47), (1, 130, 65)])
def test_f32_to_planes_t_and_planes_transpose(shape):
    ops = _ops()
    x = torch.randn(shape, device=DEV)
    n4, t4 = ops.f32_to_planes_t(1e-6 * x, scale=2.0 ** 20)     # scaled conversion of small gradients
    assert _rel(_join(n4), 1e-6 * x * 2.0 ** 20) < 1e-6 and torch.equal(t4, n4.transpose(2, 3).contiguous())
    n, t = ops.f32_to_planes_t(x)
    assert _rel(_join(n), x) < 1e-6 and _rel(_join(t), x.transpose(1, 2)) < 1e-6
    assert torch.equal(t, n.transpose(2, 3).contiguous())          # same split, only moved
    back = ops.planes_transpose(t)
    assert torch.equal(back, n)
    # column-sliced source and destination views
    G, Rr, Cc = shape
    if Cc % 16 == 0:
        half = Cc // 2
        wide = torch.zeros((2, G, half, 2 * Rr), dtype=torch.float16, device=DEV)
        ops.planes_transpose(n[..., half:], out=wide[..., Rr:])
        assert torch.equal(wide[..., Rr:], n[..., half:].transpose(2, 3))
        assert float(wide[..., :Rr].abs().max()) == 0.0


@pytest.mark.parametrize("M,N,K", [(64, 64, 256), (512, 512, 8192), (1024, 512, 4104), (96, 200, 1000)])
def test_split_k_weight_gradient_gemm(M, N, K):
    """k-slices reduce-added by TMA into a zeroed output == the unsplit contraction"""
    ops = _ops()
    dy = torch.randn(K, M, device=DEV)
    x = torch.randn(K, N, device=DEV)
    _, dy_t = ops.f32_to_planes_t(dy, want_plain=False)
    _, x_t = ops.f32_to_planes_t(x, want_plain=False)
    ks = ops.wgrad_k_split(M, N, K)
    assert ks >= 2
    out = torch.zeros(M, N, device=DEV)
    ops.linear(dy_t, x_t.unsqueeze(1), out=out, k_split=ks)
    plain = ops.linear(dy_t, x_t.unsqueeze(1))
    want = dy.double().t() @ x.double()
    assert _rel(plain, want) < 1e-4                                # the 3-product split's own accuracy
    assert _rel(out, want) < 1e-4
    assert _rel(out, plain) < 1e-4                                 # only the accumulation order differs
    ops.linear(dy_t, x_t.unsqueeze(1), out=out, k_split=ks)       # accumulates: twice the gradient
    assert _rel(out, 2 * plain) < 1e-4
    # in-place residual accumulate with a column bias (x += lin(a), the small-batch proj / fc2 path)
    base = torch.randn(M, N, device=DEV)
    bias = torch.randn(N, device=DEV)
    acc = base.clone()
    ops.linear(dy_t, x_t.unsqueeze(1), bias, out=acc, k_split=ks)
    assert _rel(acc, base.double() + want + bias.double()) < 1e-4
    with pytest.raises(Exception):
        ops.linear(dy_t, x_t.unsqueeze(1), out=out, k_split=ks, residual=base)


@pytest.mark.parametrize("M,No,Ni", [(64, 64, 64), (1000, 512, 200), (8192, 1536, 512), (520, 96, 2048)])
def test_mn_major_operands_wgrad_and_dgrad(M, No, Ni):
    """tensor-core operands read contraction-major (no transposed copies): dW = dY^T X (both MN-major, plain
    and split-K) and dX = dY W with the forward's [out,in] weight planes (B MN-major)"""
    ops = _ops()
    dy = torch.randn(M, No, device=DEV)
    x = torch.randn(M, Ni, device=DEV)
    w = torch.randn(No, Ni, device=DEV) / 8
    dyp, xp = ops.f32_to_planes_rows(dy), ops.f32_to_planes_rows(x)
    assert _rel(_join(dyp), dy) < 1e-6
    want = dy.double().t() @ x.double()
    out = torch.empty(No, Ni, device=DEV)
    ops.wgrad(dyp, xp, out)
    assert _rel(out, want) < 1e-4
    ks = ops.wgrad_k_split(No, Ni, M)
    if ks >= 2:
        out2 = torch.zeros(No, Ni, device=DEV)
        ops.wgrad(dyp, xp, out2, k_split=ks)
        assert _rel(out2, want) < 1e-4
    wp = ops.f32_to_planes_rows(w).unsqueeze(1)                      # [T,1,No,Ni] as the forward holds it
    dx = ops.linear(dyp, wp, w_kn=True)                              # [M, Ni] = dY W
    assert _rel(dx, dy.double() @ w.double()) < 1e-4
    fwd = ops.linear(xp, wp)                                         # same planes, K-major: X W^T
    assert _rel(fwd, x.double() @ w.double().t()) < 1e-4


@pytest.mark.parametrize("B,T,nh,hs", [(2, 32, 4, 16), (3, 160, 8, 16), (2, 512, 8, 64)])
def test_attention_products_on_the_fused_qkv_layout(B, T, nh, hs):
    """q|k|v side by side in one [M,3C] planes matrix: scores from column-sliced views, att.v with v
    token-major (B MN-major), and the transposed-probability products of the backward pass (A MN-major)"""
    ops = _ops()
    C, M = nh * hs, B * T
    qkv = torch.randn(M, 3 * C, device=DEV)
    qkvp = ops.f32_to_planes_rows(qkv)
    q, k, v = (qkv[:, i * C:(i + 1) * C].view(B, T, nh, hs).permute(0, 2, 1, 3).double() for i in range(3))
    qp, kp, vp = qkvp[:, :, :C], qkvp[:, :, C:2 * C], qkvp[:, :, 2 * C:]
    sc = ops.mha_scores(qp, B, T, nh, k=kp)
    assert _rel(sc, q @ k.transpose(-1, -2)) < 1e-4
    p = torch.softmax(torch.randn(B, nh, T, T, device=DEV), -1)
    pp = ops.f32_to_planes_rows(p)
    y = ops.mha_pv(pp, vp, B, T, nh, planes_out=False, v_tok=True)
    want = (p.double() @ v).permute(0, 2, 1, 3).reshape(M, C)
    assert _rel(y, want) < 1e-4
    wide = torch.zeros(M, 3 * C, device=DEV)
    ops.mha_pv(pp, vp, B, T, nh, planes_out=False, out=wide[:, C:2 * C], p_mn=True, v_tok=True, alpha=0.5)
    want_t = 0.5 * (p.double().transpose(-1, -2) @ v).permute(0, 2, 1, 3).reshape(M, C)
    assert _rel(wide[:, C:2 * C], want_t) < 1e-4 and float(wide[:, :C].abs().max()) == 0.0


def test_colsum_gelu_layernorm_softmax_backward_kernels():
    ops = _ops()
    M, Cc = 200, 96
    x = torch.randn(M, Cc, device=DEV)
    acc = torch.ones(Cc, device=DEV)
    ops.colsum_(acc, x)
    assert _rel(acc, 1 + x.sum(0)) < 1e-5
    # GELU
    a = (3 * torch.randn(M, Cc, device=DEV)).requires_grad_(True)
    dg = torch.randn(M, Cc, device=DEV)
    g_ref = F.gelu(a)
    g_ref.backward(dg)
    assert _rel(_join(ops.gelu_fwd(a.detach())), g_ref.detach()) < 2e-6
    assert _rel(ops.gelu_bwd(a.detach(), dg), a.grad) < 1e-5
    da32, dap = ops.gelu_bwd(a.detach(), dg, want_planes=True)      # fp32 + planes from one pass
    assert _rel(da32, a.grad) < 1e-5 and _rel(_join(dap), da32) < 1e-6
    # LayerNorm backward, overwrite and accumulate, C <= 512 and > 512 paths
    for Cn in (96, 512, 640):
        xx = torch.randn(M, Cn, device=DEV, requires_grad=True)
        gam = (1 + 0.1 * torch.randn(Cn, device=DEV)).requires_grad_(True)
        bet = torch.zeros(Cn, device=DEV, requires_grad=True)
        dy = torch.randn(M, Cn, device=DEV)
        F.layer_norm(xx, (Cn,), gam, bet, 1e-5).backward(dy)
        for acc_mode in (False, True):
            base = torch.randn(M, Cn, device=DEV)
            dx = base.clone()
            dgam = torch.zeros(Cn, device=DEV)
            dbet = torch.zeros(Cn, device=DEV)
            ops.layernorm_bwd_(dx, dy, xx.detach(), gam.detach(), dgam, dbet, 1e-5, accumulate=acc_mode)
            want = xx.grad + base if acc_mode else xx.grad
            assert _rel(dx, want) < 1e-5, (Cn, acc_mode)
            assert _rel(dgam, gam.grad) < 1e-5 and _rel(dbet, bet.grad) < 1e-5, (Cn, acc_mode)
            # fused outputs of the same pass: planes of the updated dx and its column sums (a bias gradient)
            dx2 = base.clone()
            cs = torch.ones(Cn, device=DEV)
            pl = ops.layernorm_bwd_(dx2, dy, xx.detach(), gam.detach(), torch.zeros_like(dgam), torch.zeros_like(dbet),
                                    1e-5, accumulate=acc_mode, want_planes=True, colsum_out=cs)
            assert torch.equal(dx2, dx) and _rel(_join(pl), dx) < 1e-6 and _rel(cs, 1 + dx.sum(0)) < 1e-4
    # softmax backward
    for cols in (32, 512, 600):
        s = torch.randn(6, 5, cols, device=DEV, requires_grad=True)
        dp = torch.randn(6, 5, cols, device=DEV)
        scale = 0.37
        p = F.softmax(s * scale, -1)
        p.backward(dp)
        ds = ops.softmax_bwd(ops.split_planes(p.detach(), 2), dp, scale)
        dsp = ops.softmax_bwd_planes(ops.split_planes(p.detach(), 2), dp, scale, out_scale=256.0)
        assert dsp.shape == (2, 6, 5, cols) and _rel(_join(dsp) / 256.0, ds) < 1e-6
        assert _rel(ds, s.grad) < 1e-5, cols


def test_ce_heads_embed_bwd_adam_kernels():
    ops = _ops()
    M, nh, ncls = 70, 18, 48
    logits = (2 * torch.randn(M, nh, ncls, device=DEV)).requires_grad_(True)
    head = torch.randint(0, nh, (M,), device=DEV)
    tgt = torch.randint(0, ncls, (M,), device=DEV)
    tgt[::3] = -1
    w = torch.rand(M, device=DEV)
    ce, dl = ops.ce_heads(logits.detach(), tgt, head, w)
    own = logits[torch.arange(M, device=DEV), head]                 # [M, ncls]
    ce_ref = F.cross_entropy(own, tgt, ignore_index=-1, reduction="none")
    (w * ce_ref).sum().backward()
    assert _rel(ce, ce_ref.detach()) < 1e-5
    assert _rel(dl.view(M, nh, ncls), logits.grad) < 1e-5
    assert float(dl.view(M, nh, ncls)[tgt < 0].abs().max()) == 0.0
    # embedding scatter-add (token table and positional table)
    Cc, V, T = 64, 11, 10
    dx = torch.randn(40, Cc, device=DEV)
    idx = torch.randint(0, V, (40,), device=DEV)
    dE = torch.zeros(V, Cc, device=DEV)
    ops.embed_bwd_(dE, dx, idx)
    assert _rel(dE, torch.zeros(V, Cc, device=DEV).index_add_(0, idx, dx)) < 1e-5
    dP = torch.zeros(T, Cc, device=DEV)
    ops.embed_bwd_(dP, dx, None, T)
    assert _rel(dP, dx.view(4, T, Cc).sum(0)) < 1e-5
    # Adam against torch.optim.Adam over three steps, with a 1/world gradient scale
    p = torch.randn(1000, device=DEV)
    ref = p.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-3)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    for step in range(1, 4):
        g = torch.randn(1000, device=DEV)
        ref.grad = g.clone()
        opt.step()
        ops.adam_(p, 4 * g, m, v, 1e-3, 0.9, 0.999, 1e-8, step, grad_scale=0.25)
        assert _rel(p, ref.detach()) < 1e-6, step


# ----------------------------------------------------------------------------- the training step
def _make(cfg, seed):
    from text2human_b200.transformer_arch import TransformerMultiHead
    from text2human_b200.transformer_train import SamplerTrainer
    net = TransformerMultiHead(**cfg)
    sd = R.fill_state_dict(R.spec_of(net), seed)
    net.load_state_dict(sd, strict=True)
    net.to(DEV)
    return net, sd, SamplerTrainer(net)


def _grad_report(net, want_grads, loss_scale):
    """max error of every gradient tensor relative to its own max; tensors whose true gradient vanishes
    (key.bias: softmax is invariant to it; start_tok: unused) are measured against the typical scale"""
    rows, worst = [], 0.0
    typical = float(np.median([float(w.abs().max()) for w in want_grads.values()]))
    for k, p in net.named_parameters():
        want = want_grads[k].to(DEV)
        e = float((p.grad / loss_scale - want).abs().max())
        scale = max(float(want.abs().max()), 0.05 * typical)
        rel = e / scale
        rows.append(f"{k:40s} |g|max {scale:.3e} err {e:.3e} rel {rel:.2e}")
        worst = max(worst, rel)
    return worst, "\n".join(rows)


def test_train_step_matches_reference_fixture():
    from text2human_b200.transformer_train import targets_from_gt_list
    _ops()
    cfg = R.TINY_TRANSFORMER
    gold = R.load_golden(GOLD)
    net, sd, tr = _make(cfg, 71)
    x_0, gt_list, segm, tex = [t.to(DEV) if torch.is_tensor(t) else [g.to(DEV) for g in t]
                               for t in R.sampler_train_batch(72)]
    t = torch.from_numpy(gold["t"]).to(DEV)
    mask = torch.from_numpy(gold["mask"]).to(DEV)
    loss, vb = tr.loss_and_grads(x_0, targets_from_gt_list(gt_list), segm, tex, t, mask=mask)
    assert abs(float(loss) - float(gold["loss"])) <= 1e-4 * abs(float(gold["loss"]))
    assert abs(float(vb) - float(gold["vb_loss"])) <= 1e-4 * abs(float(gold["vb_loss"]))
    worst, rep = _grad_report(net, {k: torch.from_numpy(gold["grad/" + k]) for k, _ in net.named_parameters()},
                              tr.loss_scale)
    assert worst <= 1e-3, "\n" + rep
    # one Adam step: compare the parameter moves with the real torch.optim.Adam's
    tr.adam_step()
    typical = float(np.median([float(np.abs(gold["grad/" + k]).max()) for k, _ in net.named_parameters()]))
    for k, p in net.named_parameters():
        d_want = torch.from_numpy(gold["param1/" + k]) - sd[k]
        d_got = p.detach().cpu() - sd[k]
        g = torch.from_numpy(gold["grad/" + k]).abs()
        # Adam's sign-like first step turns rounding noise on (mathematically) zero gradients into +-lr
        # moves in the reference too (key.bias, start_tok): compare only where a gradient exists
        sel = (g > 1e-3 * g.max()) & (g > 1e-4 * typical)
        if sel.any():
            assert float((d_got - d_want)[sel].abs().max()) <= 0.02 * 1e-4, k
    # the inference mirror sees the updated weights (packed-plane caches were dropped)
    lg = torch.stack(net(x_0, segm, tex))
    from oracle import transformer_ref as TR
    sd1 = {k: torch.from_numpy(gold["param1/" + k]) for k in sd}
    want = torch.stack(TR.transformer_logits(sd1, x_0.cpu(), segm.cpu(), tex.cpu(), cfg["bert_n_head"]))
    assert _rel(lg.cpu(), want) < 1e-3


def test_train_step_matches_autograd_of_restatement_mid_shape():
    from oracle import transformer_ref as TR
    from text2human_b200.transformer_train import targets_from_gt_list
    _ops()
    cfg = dict(R.TINY_TRANSFORMER, codebook_size=18 * 64, bert_n_emb=128, bert_n_layers=3, bert_n_head=8,
               block_size=160, latent_shape=[16, 10])
    net, sd, tr = _make(cfg, 81)
    B = 3
    x_0, gt_list, segm, tex = R.sampler_train_batch(82, B=B, cfg=cfg)
    g = R._gen(83, "t")
    t = torch.randint(1, 1001, (B,), generator=g)
    mask = torch.rand(x_0.shape, generator=g) < (t.float().unsqueeze(-1) / 1000)
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss_ref, vb_ref = TR.train_loss(sdr, x_0, gt_list, segm, tex, t, mask, cfg["bert_n_head"], cfg["codebook_size"])
    loss_ref.backward()
    want = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in sdr.items()}
    loss, vb = tr.loss_and_grads(x_0.to(DEV), targets_from_gt_list(gt_list).to(DEV), segm.to(DEV), tex.to(DEV),
                                 t.to(DEV), mask=mask.to(DEV))
    assert abs(float(loss) - float(loss_ref)) <= 1e-4 * abs(float(loss_ref))
    assert abs(float(vb) - float(vb_ref)) <= 1e-4 * abs(float(vb_ref))
    worst, rep = _grad_report(net, want, tr.loss_scale)
    assert worst <= 1e-3, "\n" + rep


def test_training_reduces_loss_at_the_real_sampler_shape():
    """size-independent property at BASELINE's sampler shape (512 tokens, 512 wide, 8 heads; 4 of the 24
    layers to bound the time): repeated steps on one fixed batch / fixed (t, mask) drive the loss down"""
    from text2human_b200.transformer_train import targets_from_gt_list
    _ops()
    cfg = dict(codebook_size=18 * 1024, segm_codebook_size=1024, texture_codebook_size=18, bert_n_emb=512,
               bert_n_layers=4, bert_n_head=8, block_size=512, latent_shape=[32, 16], embd_pdrop=0.0,
               resid_pdrop=0.0, attn_pdrop=0.0, num_head=18)
    net, sd, tr = _make(cfg, 91)
    tr.lr = 1e-3
    B = 4
    x_0, gt_list, segm, tex = [t.to(DEV) if torch.is_tensor(t) else [g.to(DEV) for g in t]
                               for t in R.sampler_train_batch(92, B=B, cfg=cfg)]
    own = targets_from_gt_list(gt_list)
    t = torch.tensor([900, 500, 300, 700], device=DEV)
    g = torch.Generator(device=DEV).manual_seed(5)
    _, mask = tr.q_sample(x_0, t, g)
    losses = []
    for _ in range(12):
        loss, _ = tr.loss_and_grads(x_0, own, segm, tex, t, mask=mask)
        assert math.isfinite(float(loss))
        losses.append(float(loss))
        tr.adam_step()
    assert losses[-1] < 0.7 * losses[0], losses
    # optimize_parameters draws its own t and mask like the reference
    loss, vb = tr.optimize_parameters(x_0, own, segm, tex)
    assert math.isfinite(float(loss)) and math.isfinite(float(vb))


def test_training_wrapper_feed_data_and_step():
    """TransformerTextureAwareModel.feed_data (frozen tokenizers -> tokens, transformer_model.py:273-288) +
    optimize_parameters, real tokenizer sizes (configs/sampler.yml), 2 transformer layers"""
    import contextlib
    import io
    from text2human_b200.pipeline import TransformerTextureAwareModel
    _ops()
    opt = dict(img_ch=128, img_num_res_blocks=2, img_attn_resolutions=[32], img_ch_mult=[1, 1, 2, 2, 4],
               img_in_channels=3, img_resolution=512, img_z_channels=256, img_double_z=False, img_dropout=0.0,
               img_n_embed=1024, img_embed_dim=256, img_out_ch=3,
               segm_double_z=False, segm_z_channels=32, segm_resolution=512, segm_in_channels=24, segm_out_ch=24,
               segm_ch=64, segm_ch_mult=[1, 1, 2, 2, 4], segm_num_res_blocks=1, segm_attn_resolutions=[16],
               segm_dropout=0.0, segm_num_segm_classes=24, segm_n_embed=1024, segm_embed_dim=32,
               codebook_size=18432, segm_codebook_size=1024, texture_codebook_size=18, bert_n_emb=512,
               bert_n_layers=2, bert_n_head=8, block_size=512, latent_shape=[32, 16], embd_pdrop=0.0,
               resid_pdrop=0.0, attn_pdrop=0.0, num_head=18, loss_type="reweighted_elbo", lr=1e-4)
    torch.manual_seed(7)
    with contextlib.redirect_stdout(io.StringIO()):
        m = TransformerTextureAwareModel(opt).to(DEV)
    B = 2
    data = dict(image=R.image(1, B, 3, 512, 256), segm=R.blocky_mask(2, B, 512, 256, 16, n_ids=24),
                texture_mask=R.blocky_mask(3, B, 512, 256, 32))
    m.feed_data(data)
    tex = F.interpolate(data["texture_mask"], (32, 16), mode="nearest").view(B, -1).long().to(DEV)
    assert torch.equal(m.texture_tokens, tex)
    assert m.input_indices.shape == (B, 512) and torch.equal(m.input_indices, m.gt_own + 1024 * tex)
    assert int(m.gt_own.min()) >= 0 and int(m.gt_own.max()) < 1024
    assert m.segm_tokens.shape == (B, 512) and int(m.segm_tokens.max()) < 1024
    g = torch.Generator(device=DEV).manual_seed(3)
    l0, _ = m.optimize_parameters(g)
    l1, vb = m.optimize_parameters(g)
    assert math.isfinite(float(l0)) and math.isfinite(float(l1)) and math.isfinite(float(vb))
    assert m.trainer.step_count == 2
