"""CPU: the training restatement (oracle/transformer_ref.train_loss, adam_update) against the fixture made
from the real reference `_train_loss` + `loss.backward()` + `torch.optim.Adam.step()`
(oracle/make_golden_train.py), and the trainer's flat parameter layout (host logic)."""
import os

import numpy as np
import torch

import golden_recipes as R
from oracle import transformer_ref as TR

GOLD = os.path.join(os.path.dirname(__file__), "golden", "sampler_train.npz")


def _setup():
    from text2human_b200.transformer_arch import TransformerMultiHead
    cfg = R.TINY_TRANSFORMER
    net = TransformerMultiHead(**cfg)
    sd = R.fill_state_dict(R.spec_of(net), 71)
    return cfg, net, sd, R.sampler_train_batch(72), R.load_golden(GOLD)


def test_train_loss_restatement_matches_reference_fixture():
    cfg, net, sd, (x_0, gt_list, segm, tex), gold = _setup()
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    t, mask = torch.from_numpy(gold["t"]), torch.from_numpy(gold["mask"])
    loss, vb = TR.train_loss(sd, x_0, gt_list, segm, tex, t, mask, cfg["bert_n_head"], cfg["codebook_size"])
    loss.backward()
    assert abs(float(loss) - float(gold["loss"])) <= 1e-6 * abs(float(gold["loss"]))
    assert abs(float(vb) - float(gold["vb_loss"])) <= 1e-6 * abs(float(gold["vb_loss"]))
    for k, p in sd.items():
        want = torch.from_numpy(gold["grad/" + k])
        got = p.grad if p.grad is not None else torch.zeros_like(p)
        assert (got - want).abs().max() <= 1e-5 * want.abs().max() + 1e-9, k
        p1, _, _ = TR.adam_update(p.detach(), got, torch.zeros_like(got), torch.zeros_like(got), 1)
        # Adam's first step moves every touched weight by ~lr; compare the moves
        d_want = torch.from_numpy(gold["param1/" + k]) - p.detach()
        assert ((p1 - p.detach()) - d_want).abs().max() <= 2e-3 * 1e-4 + 1e-9, k


def test_trainer_flat_layout_aliases_parameters():
    from text2human_b200.transformer_train import SamplerTrainer, targets_from_gt_list
    cfg, net, sd, (x_0, gt_list, segm, tex), gold = _setup()
    net.load_state_dict(sd, strict=True)
    tr = SamplerTrainer(net)
    # the parameters are views of the flat buffer, values preserved, state_dict keys unchanged
    for k, v in net.state_dict().items():
        assert torch.equal(v, sd[k]), k
    tr.flat_p.add_(1.0)
    for k, v in net.state_dict().items():
        assert torch.equal(v, sd[k] + 1.0), k
    # q|k|v weights and biases are adjacent so that one GEMM produces all three gradients
    a = net.blocks[0].attn
    C = cfg["bert_n_emb"]
    wqkv = tr._flat_view(tr.flat_p, a.query.weight, 3 * C, C)
    assert torch.equal(wqkv, torch.cat((a.query.weight, a.key.weight, a.value.weight), 0))
    bqkv = tr._flat_view(tr.flat_p, a.query.bias, 1, 3 * C)[0]
    assert torch.equal(bqkv, torch.cat((a.query.bias, a.key.bias, a.value.bias), 0))
    wh = tr._flat_view(tr.flat_p, net.head_list[0].weight, cfg["codebook_size"], C)
    assert torch.equal(wh, torch.cat([h.weight for h in net.head_list], 0))
    # gradient views alias the flat gradient buffer; buckets tile it without gaps
    tr.flat_g.fill_(3.0)
    assert all(float(p.grad.min()) == 3.0 for p in net.parameters())
    spans = sorted(tr.group_span.values())
    assert spans[0][0] == 0 and spans[-1][1] == tr.flat_g.numel()
    assert all(spans[i][1] == spans[i + 1][0] for i in range(len(spans) - 1))
    own = targets_from_gt_list(gt_list)
    assert torch.equal(own + 16 * tex, x_0)
