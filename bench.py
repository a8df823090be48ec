"""bench.py — headline benchmark of the Text2Human VQ hot path on B200.

Metric (BASELINE.json): 512x256 images/s, vqvae_top encode -> quantize -> decode.
Workload (configs[1]): vqvae_top.yml nets, batch 16 x 3x512x256 per GPU, codebook 18x1024x256,
synthetic images/masks, random-init weights.  One "step" = one forward_step over one batch.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--precision fp32|fp16] [--impl ours|reference]
                  [--dump-outputs DIR]

N>1 is launched by torchrun (one rank per GPU); the path shards over independent images (replicas,
weak scaling), there is no data-path collective — only the timing reduction (max over ranks).
`--impl reference` times the CPU port of the reference path (oracle/vqgan_ref.py) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

VQVAE_TOP = dict(embed_dim=256, n_embed=1024, double_z=False, z_channels=256, resolution=512, in_channels=3,
                 out_ch=3, ch=128, ch_mult=[1, 1, 2, 2, 4], num_res_blocks=2, attn_resolutions=[32],
                 dropout=0.0)
GFLOP_PER_IMG = 784.4  # reference op graph, 2*MAC (SURVEY.md §8a / BASELINE.md §3)
METRIC = "512x256 images/sec VQ enc-quant-dec (vqvae_top)"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v == "Active":
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def make_inputs(batch, n_variants, seed):
    import golden_recipes as R
    xs, ms = [], []
    for i in range(n_variants):
        xs.append(R.image(seed + i, batch, 3, 512, 256))
        ms.append(R.blocky_mask(seed + i, batch, 512, 256, 32))
    return xs, ms


def host_threads():
    """PyTorch's CPU convolutions stop scaling (and regress) far below the 128+ hardware threads of the
    GPU hosts; 32 is the fastest setting measured there, so that is what the CPU legs use."""
    return max(1, min(32, os.cpu_count() or 1))


def cpu_port_rate(threads, runs, batch=1):
    """images/s of the reference path on the host cores: the reference's own modules when staged (oracle/_ref),
    else the oracle port.  -> (best, mean, times, kind)"""
    import golden_recipes as R
    fn, kind = _reference_forward_fn("cpu", threads)
    x = R.image(2021, batch, 3, 512, 256)
    mask = R.blocky_mask(2021, batch, 512, 256, 32)
    times = []
    fn(x, mask)  # warm-up
    for _ in range(runs):
        t0 = time.perf_counter()
        fn(x, mask)
        times.append(time.perf_counter() - t0)
    return batch / min(times), batch / (sum(times) / len(times)), times, kind


HIER_OPT = dict(embed_dim=256, n_embed=1024, codebook_spatial_size=2, bot_n_embed=512, bot_double_z=False,
                bot_z_channels=256, bot_resolution=512, bot_in_channels=3, bot_out_ch=3, bot_ch=128,
                bot_ch_mult=[1, 1, 2, 4], bot_num_res_blocks=2, bot_attn_resolutions=[64], bot_dropout=0.0,
                top_double_z=False, top_z_channels=256, top_resolution=512, top_in_channels=3, top_out_ch=3,
                top_ch=128, top_ch_mult=[1, 1, 2, 2, 4], top_num_res_blocks=2, top_attn_resolutions=[32],
                top_dropout=0.0)
SAMPLER_OPT = dict(codebook_size=18432, segm_codebook_size=1024, texture_codebook_size=18, bert_n_emb=512,
                   bert_n_layers=24, bert_n_head=8, block_size=512, latent_shape=[32, 16], embd_pdrop=0.0,
                   resid_pdrop=0.0, attn_pdrop=0.0, num_head=18, sample_steps=256)


def side_workloads(dev, precision):
    """BASELINE configs 3 and 4, a few iterations each (reported next to the headline, not instead of it)."""
    import contextlib
    import golden_recipes as R
    from text2human_b200 import ops
    from text2human_b200.pipeline import HierarchyVQSpatialTextureAwareModel, Sampler
    out = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        torch.manual_seed(3)
        with contextlib.redirect_stdout(sys.stderr):
            hm = HierarchyVQSpatialTextureAwareModel(HIER_OPT).to(dev).eval()
        x = R.image(7, 8, 3, 512, 256).to(dev)
        m = R.blocky_mask(7, 8, 512, 256, 32).to(dev)
        for _ in range(2):
            hm.forward_step(x, m)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            hm.forward_step(x, m)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        out["config3_hierarchy_forward_step"] = dict(batch=8, ms_per_step=ms, img_per_s=8 / (ms / 1e3),
                                                     algorithmic_tflops=8 * 1200.9 / ms, precision=precision)
        del hm
        torch.cuda.empty_cache()
        torch.manual_seed(4)
        sm = Sampler(SAMPLER_OPT).to(dev).eval()
        segm = torch.randint(0, 1024, (4, 512), device=dev)
        tm = R.blocky_mask(9, 4, 512, 256, 64).to(dev)
        gen = torch.Generator(device=dev).manual_seed(2021)
        sm.sample_fn(segm, tm, sample_steps=4, generator=gen)
        torch.cuda.synchronize()
        steps = SAMPLER_OPT["sample_steps"]               # the full 256-step sample of BASELINE config 4
        e0.record()
        sm.sample_fn(segm, tm, sample_steps=steps, generator=gen)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out["config4_sampler"] = dict(batch=4, ms_per_diffusion_step=ms, measured_steps=steps,
                                      tokens_per_s_256_steps=2048 / (ms * 256 / 1e3), extrapolated=False,
                                      algorithmic_tflops=4 * 99.86 / ms, precision=precision,
                                      launch="CUDA graph replay of the transformer forward per step; fused attention "
                                             "kernel (t2h_attn_fwd), deterministic split-K + fused reduce/LayerNorm",
                                      launches_per_step=None)
        l0 = ops.COUNTERS["launches"]
        sm.sample_fn(segm, tm, sample_steps=2, generator=gen, use_graph=False)
        out["config4_sampler"]["launches_per_step"] = (ops.COUNTERS["launches"] - l0) // 2
        # informational: the same sampler with single-product fp16 operands (not the parity mode; logits within 2e-3
        # of the reference instead of 6e-6) -- separates the tensor-issue share of a step from its serial latency
        if precision != "fp16":
            old_terms = ops.get_terms()
            try:
                ops.set_precision("fp16")
                sm.sample_fn(segm, tm, sample_steps=4, generator=gen)
                torch.cuda.synchronize()
                e0.record()
                sm.sample_fn(segm, tm, sample_steps=64, generator=gen)
                e1.record()
                torch.cuda.synchronize()
                ms16 = e0.elapsed_time(e1) / 64
                out["config4_sampler"]["single_product_fp16"] = dict(ms_per_diffusion_step=ms16, measured_steps=64,
                                                                     algorithmic_tflops=4 * 99.86 / ms16)
            except Exception as exc:  # noqa: BLE001
                out["config4_sampler"]["single_product_fp16"] = dict(error=repr(exc))
            finally:
                ops._PRECISION["terms"] = old_terms
        # the refine half of sample_and_refine (SURVEY a16): sampled top tokens -> top codebook gather -> UNet/FCN
        # index prediction -> bottom gather -> DecoderRes -> Decoder, batched (the reference decodes one by one)
        del sm
        torch.cuda.empty_cache()
        from text2human_b200.pipeline import SampleFromParsingModel
        opt = dict(HIER_OPT)
        opt.update(SAMPLER_OPT)
        opt.update(bot_codebook_spatial_size=2, index_pred_encoder_in_channels=256, index_pred_fc_in_channels=64,
                   index_pred_fc_in_index=4, index_pred_fc_channels=64, index_pred_fc_num_convs=1,
                   index_pred_fc_concat_input=False, index_pred_fc_dropout_ratio=0.1,
                   index_pred_fc_num_classes=512, index_pred_fc_align_corners=False, segm_double_z=False,
                   segm_z_channels=32, segm_resolution=512, segm_in_channels=24, segm_out_ch=24, segm_ch=64,
                   segm_ch_mult=[1, 1, 2, 2, 4], segm_num_res_blocks=1, segm_attn_resolutions=[16],
                   segm_dropout=0.0, segm_num_segm_classes=24, segm_n_embed=1024, segm_embed_dim=32)
        torch.manual_seed(6)
        with contextlib.redirect_stdout(sys.stderr):
            sp = SampleFromParsingModel(opt).to(dev).eval()
        tex = torch.nn.functional.interpolate(tm, (32, 16), mode="nearest")[:, 0].long()
        top = torch.randint(0, 1024, (4, 32, 16), device=dev)
        top_list = [torch.where(tex == k, top, torch.full_like(top, -1)) for k in range(18)]
        for _ in range(2):
            sp.decode_top_tokens(top_list, tm)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            sp.decode_top_tokens(top_list, tm)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        out["config4_refine_decode"] = dict(batch=4, ms_per_batch=ms, img_per_s=4 / (ms / 1e3), precision=precision,
                                            stages="top gather, 1x1, UNet+FCN index prediction, bottom gather, "
                                                   "DecoderRes, Decoder(bot_h), clamp")
    except Exception as exc:  # side measurements must never break the headline line
        out["error"] = repr(exc)
    return out


def train_workload(dev, precision, world, batch=16, steps=4):
    """SURVEY 8(a17)/(e): one optimiser step of the index-prediction transformer (q_sample masking, forward,
    18 masked cross-entropies, backward, bucketed NCCL gradient all-reduce when world > 1, Adam), per-GPU
    batch fixed (weak scaling).  Every rank must call this when world > 1 (collective inside)."""
    import golden_recipes as R
    from text2human_b200 import dist as D
    from text2human_b200 import ops
    from text2human_b200.transformer_arch import TransformerMultiHead
    from text2human_b200.transformer_train import SamplerTrainer, targets_from_gt_list
    cfg = {k: v for k, v in SAMPLER_OPT.items() if k != "sample_steps"}
    torch.manual_seed(5)
    net = TransformerMultiHead(**cfg).to(dev)
    tr = SamplerTrainer(net)
    x_0, gt_list, segm, tex = R.sampler_train_batch(6 + D.env_rank()[0], B=batch, cfg=cfg)
    x_0, segm, tex = x_0.to(dev), segm.to(dev), tex.to(dev)
    own = targets_from_gt_list([g.to(dev) for g in gt_list])
    gen = torch.Generator(device=dev).manual_seed(1)
    for _ in range(2):
        tr.optimize_parameters(x_0, own, segm, tex, gen)
    D.barrier()
    torch.cuda.synchronize()
    l0 = ops.COUNTERS["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.optimize_parameters(x_0, own, segm, tex, gen)
    e1.record()
    torch.cuda.synchronize()
    ms = D.max_over_ranks(e0.elapsed_time(e1) / steps, device=dev)
    tok = batch * 512 * world
    flops = (6 * (24 * 12 * 512 * 512 + 18432 * 512) + 3 * 24 * 4 * 512 * 512) * tok
    return dict(per_gpu_batch=batch, n_gpus=world, ms_per_step=ms, tokens_per_s=tok / (ms / 1e3),
                algorithmic_tflops=flops / ms / 1e9, launches_per_step=(ops.COUNTERS["launches"] - l0) // steps,
                precision=precision, loss=float(loss), grad_allreduce="nccl, 6 buckets overlapped with backward"
                if world > 1 else "none (1 GPU)", params=tr.flat_p.numel())


def vqgan_train_workload(dev, precision, rank, world, global_batch=64, micro=8, steps=2):
    """BASELINE config 5 (SURVEY 8a18 / 8e): the VQGAN GAN training step (vqgan_model.py:444-488 + :329-344:
    generator forward, L1, DiffAugment, discriminator, adaptive weight, backward, discriminator update, two Adams),
    global batch 64 split over the ranks (strong scaling, as train_vqvae.py under DDP), gradients all-reduced over
    NCCL in buckets that are launched as the backward pass finishes them.  Every rank must call this (collectives
    inside).  Precision: single-product fp16 operands with fp32 accumulation / master weights / Adam -- the
    analogue of config 5's "bf16 autocast" (one tensor-core product per contraction); LPIPS stubbed to zero.
    Also times the same step with the all-reduce disabled: the difference is the EXPOSED (non-overlapped)
    communication time."""
    import contextlib
    import golden_recipes as R
    import torch.distributed as dist
    from text2human_b200 import ops
    from text2human_b200.pipeline import VQImageSegmTextureModel
    from text2human_b200.vqgan_arch import Discriminator
    from text2human_b200.vqgan_train import VQGANTrainer
    old_terms = ops.get_terms()
    ops.set_precision(precision)
    try:
        per_gpu = global_batch // world
        mb = min(micro, per_gpu)
        torch.manual_seed(5)
        with contextlib.redirect_stdout(sys.stderr):
            model = VQImageSegmTextureModel(VQVAE_TOP).to(dev)
        disc = Discriminator(3, 64, n_layers=3).to(dev)
        cb = R.codebooks(7, 18, 1024, 256, "trained")
        with torch.no_grad():
            for k, e in enumerate(model.quantize.embedding_list):
                e.weight.copy_(cb[k])
        tr = VQGANTrainer(model, disc, lr=1e-4, disc_start_step=0, micro_batch=mb)
        data = dict(image=R.image(300 + rank, per_gpu, 3, 512, 256).to(dev),
                    texture_mask=R.blocky_mask(300 + rank, per_gpu, 512, 256, 32).to(dev))
        gen = torch.Generator(device=dev).manual_seed(17 + rank)     # per-rank DiffAugment draws

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def timed(n, reduce_on):
            tr.force_no_reduce = not reduce_on
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = ops.COUNTERS["launches"]
            e0.record()
            for i in range(n):
                tr.optimize_parameters(data, 2 + i, gen)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1) / n
            if world > 1:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = t.item()
            return ms, (ops.COUNTERS["launches"] - l0) // n
        timed(1, True)                                   # warm-up (kernel configuration, allocator)
        ms, launches = timed(steps, True)
        ms_nr = timed(steps, False)[0] if world > 1 else ms
        tr.force_no_reduce = False
        loss = tr.losses()
        # roofline of the step's tensor-core launches (instrumented pass, rank 0): forward / data-gradient tap-GEMMs and
        # the weight-gradient launches, algorithmic FLOPs over their summed CUDA-event time
        kern = None
        if rank == 0:
            ops.profile_tapgemm(True)
            tr.force_no_reduce = True
            tr.training_step(data, 99, gen)
            tr.wait_reduced()
            torch.cuda.synchronize()
            tr.force_no_reduce = False
            agg = {}
            for algo, issued, a, b, shape in ops.profile_records():
                k = "wgrad" if shape[0] == "wgrad" else "fwd_dgrad"
                t = a.elapsed_time(b)
                e = agg.setdefault(k, [0, 0.0, 0.0])
                e[0] += 1; e[1] += t; e[2] += algo
            ops.profile_tapgemm(False)
            pk_ = peaks()
            kern = {k: dict(launches=v[0], ms=v[1], algorithmic_tflops=v[2] / v[1] / 1e9,
                            frac=v[2] / v[1] / 1e9 / pk_["tf_sustained"]) for k, v in agg.items()}
            tpath = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
            if os.path.exists(tpath):
                tj = json.load(open(tpath))
                kern["wgrad_traffic"] = dict(dram_bytes_per_launch=tj["dram_bytes_per_launch"],
                                             algorithmic_bytes_per_launch=tj["algorithmic_bytes_per_launch"],
                                             kernel=tj["kernel"], source=tj["source"])
        if world > 1:
            dist.barrier()
        gflop_img = 3 * GFLOP_PER_IMG                    # generator forward + data + weight gradients (2*MAC)
        return dict(global_batch=global_batch, per_gpu_batch=per_gpu, micro_batch=mb, n_gpus=world, scaling="strong",
                    ms_per_step=ms, img_per_s=global_batch / (ms / 1e3), launches_per_step=launches,
                    ms_per_step_without_allreduce=ms_nr, exposed_allreduce_ms=max(0.0, ms - ms_nr),
                    allreduce_bytes=4 * (tr.gen.total + tr.dsc.total),
                    buckets=dict(generator=[4 * (b - a) for a, b in tr.gen.buckets],
                                 discriminator=[4 * (b - a) for a, b in tr.dsc.buckets],
                                 limiting="the last generator bucket (encoder head): it closes with the final "
                                          "backward kernel, so its reduction cannot overlap anything"),
                    algorithmic_tflops=global_batch * gflop_img / ms, precision=precision,
                    frac_of_peak=global_batch * gflop_img / ms / (peaks()["tf_sustained"] * world),
                    losses={k: float(v) for k, v in loss.items()}, tensor_kernels=kern,
                    note="LPIPS stubbed (config 5); BatchNorm / adaptive weight per micro-batch = per DDP rank")
    finally:
        ops._PRECISION["terms"] = old_terms


def _reference_forward_fn(device, threads=None):
    """-> (fn(x, mask) running the reference's own VQImageSegmTextureModel.forward_step, kind): the UNMODIFIED
    reference sources staged in oracle/_ref (kind "reference"), else the oracle port (kind "port")."""
    import contextlib
    from oracle import ref_loader as RL
    if threads:
        torch.set_num_threads(threads)
    torch.manual_seed(2021)
    if RL.available():
        ns = RL.install("reference", wrappers=("vqgan_model",))
        w = RL.vq_top_wrapper(ns, VQVAE_TOP, device)
        for n in w.modules:
            getattr(w, n).eval()

        def fn(x, mask):
            with torch.no_grad():
                return w.forward_step(x, mask)
        return fn, "reference"
    from oracle import vqgan_ref
    from text2human_b200.pipeline import VQImageSegmTextureModel
    with contextlib.redirect_stdout(sys.stderr):
        m = VQImageSegmTextureModel(VQVAE_TOP).eval()
    sd = {k: v.detach().to(device) for k, v in m.state_dict().items()}
    cb = torch.stack([e.weight.detach() for e in m.quantize.embedding_list]).to(device)

    def fn(x, mask):
        with torch.no_grad():
            r = vqgan_ref.vq_forward_step(sd, cb, x, mask)
        return r["dec"], r["loss"]
    return fn, "port"


def run_reference(args, rank, world):
    """--impl reference: the reference's own implementation of the path (models/vqgan_model.py forward_step around
    models/archs/vqgan_arch.py, loaded unmodified from oracle/_ref) on the host cores, rank 0 only."""
    if rank != 0:
        return None
    threads = host_threads()
    import golden_recipes as R
    fn, kind = _reference_forward_fn("cpu", threads)
    x = R.image(2021, 1, 3, 512, 256)
    mask = R.blocky_mask(2021, 1, 512, 256, 32)
    for _ in range(max(1, min(args.warmup, 2))):
        fn(x, mask)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn(x, mask)
    total = time.perf_counter() - t0
    value = args.steps / total
    line = dict(metric=METRIC, value=value, unit="img/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * total / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", impl="reference",
                config=dict(workload="vqvae_top.yml enc-quant-dec 512x256, the reference's own PyTorch CPU path",
                            step="1 image (bounded sample of the batch-16 workload)"),
                cpu_baseline=dict(value=value, unit="img/s", cores=threads, kind=kind,
                                  sample=f"{args.steps} steps x 1 image 512x256, torch fp32, {threads} threads"),
                e2e=dict(value=value, unit="img/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    return line


def gpu_eager_baseline(dev, batch=16, steps=3):
    """BASELINE.md 5.5 / SURVEY 8d: the reference modules themselves on this B200 in stock PyTorch eager (cuDNN /
    cuBLAS), fp32 with TF32 off and with TF32 allowed, CUDA-event timed -- the bar the hand-written kernels have to
    beat (a baseline leg like cpu_baseline: none of it is on the product path)."""
    import golden_recipes as R
    out = {}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        fn, kind = _reference_forward_fn(dev)
        x = R.image(2021, batch, 3, 512, 256).to(dev)
        mask = R.blocky_mask(2021, batch, 512, 256, 32).to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for name, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(2):
                fn(x, mask)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                fn(x, mask)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[f"config2_{name}"] = dict(img_per_s=batch / (ms / 1e3), ms_per_step=ms, batch=batch, kind=kind)
        del fn, x, mask
        torch.cuda.empty_cache()
        # config 4: one transformer forward (= one diffusion step's model call) at B=4
        from oracle import ref_loader as RL
        cfg = {k: v for k, v in SAMPLER_OPT.items() if k != "sample_steps"}
        torch.manual_seed(4)
        if RL.available():
            ns = RL.install("reference", wrappers=())
            net = ns.transformer_arch.TransformerMultiHead(**cfg).to(dev).eval()
        else:
            net = None
        if net is not None:
            idx = torch.full((4, 512), 18432, dtype=torch.long, device=dev)
            segm = torch.randint(0, 1024, (4, 512), device=dev)
            tex = torch.randint(0, 18, (4, 512), device=dev)
            for name, tf32 in (("fp32", False), ("tf32", True)):
                torch.backends.cuda.matmul.allow_tf32 = tf32
                torch.backends.cudnn.allow_tf32 = tf32
                with torch.no_grad():
                    for _ in range(3):
                        net(idx, segm, tex)
                    torch.cuda.synchronize()
                    e0.record()
                    for _ in range(10):
                        net(idx, segm, tex)
                    e1.record()
                    torch.cuda.synchronize()
                out[f"config4_{name}"] = dict(ms_per_forward=e0.elapsed_time(e1) / 10, batch=4,
                                              note="model forward only; the reference's sample_fn adds 18 Categorical "
                                                   "draws and ~18 host syncs per step on top")
            # the reference's own sampling loop (BaseSampleModel.sample_fn, unmodified, stock PyTorch): per-step cost
            # including its 18 Categorical draws and host synchronisations
            import types
            ns2 = RL.install("reference", wrappers=("sample_model",))
            fake = types.SimpleNamespace(batch_size=4, shape=(32, 16), device=dev, mask_id=18432,
                                         texture_mask=R.blocky_mask(9, 4, 512, 256, 64).to(dev), segm_tokens=segm,
                                         sampler_fn=net)
            for name, tf32 in (("fp32", False), ("tf32", True)):
                torch.backends.cuda.matmul.allow_tf32 = tf32
                torch.backends.cudnn.allow_tf32 = tf32
                with torch.no_grad():
                    ns2.sample_model.BaseSampleModel.sample_fn(fake, temp=1.0, sample_steps=2)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    ns2.sample_model.BaseSampleModel.sample_fn(fake, temp=1.0, sample_steps=8)
                    torch.cuda.synchronize()
                    ms = (time.perf_counter() - t0) * 1e3 / 8
                out[f"config4_sample_fn_{name}"] = dict(ms_per_diffusion_step=ms,
                                                        tokens_per_s_256_steps=2048 / (ms * 256 / 1e3),
                                                        note="the reference's unmodified sample_fn loop, 8 steps, wall clock")
            del net
            torch.cuda.empty_cache()
            # config 5: the reference's own VQImageSegmTextureModel.optimize_parameters (vqgan_model.py:329-344,
            # :444-488; LPIPS stubbed to zero exactly as on our arm), stock PyTorch autograd + torch.optim.Adam,
            # batch 8 (= our micro-batch) at 512x256.  "default" = the reference as shipped: cuDNN convs may use TF32
            # (PyTorch's default), matmuls fp32; bf16_autocast wraps the unmodified step in torch.autocast.
            ns3 = RL.install("reference", wrappers=("vqgan_model",))
            opt = dict(VQVAE_TOP, n_channels=3, ndf=64, disc_layers=3, perceptual_weight=1.0, disc_start_step=0,
                       disc_weight_max=1.0, diff_aug=True, lr=1e-4)
            import contextlib
            with contextlib.redirect_stdout(sys.stderr):
                wr = ns3.vqgan_model.VQImageSegmTextureModel(opt)
            tb = 8
            data = dict(image=R.image(300, tb, 3, 512, 256), texture_mask=R.blocky_mask(300, tb, 512, 256, 32))
            for name, mm_tf32, cudnn_tf32, cast in (("fp32", False, False, False), ("default", False, True, False),
                                                    ("tf32", True, True, False), ("bf16_autocast", True, True, True)):
                try:
                    torch.backends.cuda.matmul.allow_tf32 = mm_tf32
                    torch.backends.cudnn.allow_tf32 = cudnn_tf32
                    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if cast else contextlib.nullcontext()
                    with ctx:
                        wr.optimize_parameters(data, 2)
                        torch.cuda.synchronize()
                        e0.record()
                        for i in range(2):
                            wr.optimize_parameters(data, 3 + i)
                        e1.record()
                        torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1) / 2
                    out[f"config5_train_{name}"] = dict(img_per_s=tb / (ms / 1e3), ms_per_step=ms, batch=tb,
                                                        note="reference optimize_parameters, unmodified, one GPU")
                except Exception as exc:
                    out[f"config5_train_{name}"] = dict(error=repr(exc))
            del wr
            torch.cuda.empty_cache()
    except Exception as exc:
        out["error"] = repr(exc)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return out


class StdoutToStderr:
    """Everything libraries print while the benchmark runs (NCCL's version banner, the Decoder's z-shape
    line, ...) goes to stderr at the file-descriptor level; stdout carries exactly one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


DUMP_BYTES = 64_000_000


def dump_outputs(path, outputs):
    """Write each output as float32 ``path/<name>.npy``.  An output larger than its share of DUMP_BYTES is written as
    ``<name>_sample.npy``: its flattened entries at positions drawn by a fixed seed, the same positions for every run
    of the same shapes, so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(outputs)
    for name, t in outputs.items():
        a = t.detach().float().cpu()
        if a.numel() * 4 > share:
            pick = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:share // 4].sort().values
            a, name = a.reshape(-1)[pick], name + "_sample"
        np.save(os.path.join(path, name + ".npy"), a.numpy())


def emit(line):
    sys.stdout.write(json.dumps(line) + "\n")
    sys.stdout.flush()


def main():
    with StdoutToStderr():
        line = run()
    if line is not None:
        emit(line)


def run():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp16"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extra-train-ddp", action="store_true",
                    help="N>1 only: also time the sampler training step with its NCCL gradient all-reduce")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the short config-3 (hierarchy) and config-4 (sampler) side measurements")
    ap.add_argument("--streams", type=int, default=1,
                    help="run the batch as this many concurrent slices on separate CUDA streams")
    ap.add_argument("--no-train", action="store_true", help="skip the config-5 DDP training-step measurement")
    ap.add_argument("--train-precision", default="fp16", choices=["fp32", "fp16"],
                    help="operand precision of the training step (fp16 = one tensor-core product, config 5's bf16 "
                         "autocast analogue; fp32 = the 3-product parity mode)")
    ap.add_argument("--graph", action="store_true",
                    help="replay one captured CUDA graph per step (measured: no gain for this GPU-bound step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (the decoded images and the "
                         "codebook loss) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    from text2human_b200 import _lib, ops
    from text2human_b200.pipeline import GraphedStep, VQImageSegmTextureModel

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    ops.set_precision(args.precision)

    torch.manual_seed(2021)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):  # the Decoder constructor prints its z-shape like the reference
        model = VQImageSegmTextureModel(VQVAE_TOP).to(dev).eval()
    B = args.batch
    n_var = 3
    xs_h, ms_h = make_inputs(B, n_var, 100 + rank * 10)
    xs_h = [x.pin_memory() for x in xs_h]
    ms_h = [m.pin_memory() for m in ms_h]
    xs_d = [x.to(dev) for x in xs_h]
    ms_d = [m.to(dev) for m in ms_h]
    out_h = torch.empty((B, 3, 512, 256), dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # One step = one forward_step (~340 asynchronous launches; --graph replays them as one CUDA graph).
    def raw_step(x, m):
        dec, loss = model.forward_step(x, m, streams=args.streams)
        return dec, loss
    step = GraphedStep(raw_step, (xs_d[0], ms_d[0])) if args.graph else raw_step

    # ---------------- device-resident throughput (`value`) ----------------
    for i in range(args.warmup):
        step(xs_d[i % n_var], ms_d[i % n_var])
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = ops.COUNTERS["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        dec, loss = step(xs_d[i % n_var], ms_d[i % n_var])
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    launches = ops.COUNTERS["launches"] - l0
    value = world * B * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:   # before the next step can overwrite a graph's static outputs
        dump_outputs(args.dump_outputs, dict(dec=dec, codebook_loss=loss))

    # ---------------- end to end through the public API with host buffers ----------------
    x_in = torch.empty_like(xs_d[0])
    m_in = torch.empty_like(ms_d[0])

    def e2e_step(i):
        x_in.copy_(xs_h[i % n_var], non_blocking=True)   # pinned host -> device, inside the timed region
        m_in.copy_(ms_h[i % n_var], non_blocking=True)
        dec, loss = step(x_in, m_in)
        out_h.copy_(dec, non_blocking=True)              # device -> pinned host
        return loss
    for i in range(2):
        e2e_step(i)
    barrier()
    e0.record()
    for i in range(args.steps):
        e2e_step(i)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    h2d = xs_h[0].numel() * 4 + ms_h[0].numel() * 4
    d2h = out_h.numel() * 4

    # ---------------- roofline of the dominant kernel (t2h tapgemm), instrumented pass ----------------
    pk = peaks()
    roof = None
    if rank == 0:
        ops.profile_tapgemm(True)
        model.forward_step(xs_d[0], ms_d[0])
        torch.cuda.synchronize()
        rec = ops.profile_records()
        algo = sum(r[0] for r in rec)
        issued = sum(r[1] for r in rec)
        t_ms = sum(r[2].elapsed_time(r[3]) for r in rec)
        ops.profile_tapgemm(False)
        achieved = algo / (t_ms * 1e-3) / 1e12
        traffic, traffic_note = None, None
        tpath = os.path.join(ROOT, "profiles", "r01_ncu_traffic.json")
        if os.path.exists(tpath) and args.precision == "fp32":
            tj = json.load(open(tpath))
            traffic = tj["dram_bytes_per_launch"]
            traffic_note = (f"dram read+write bytes of the dominant launch ({tj['kernel']}) from {tj['source']}; "
                            f"algorithmic bytes of that launch {tj['algorithmic_bytes_per_launch']}")
        roof = dict(bound="tensor", kernel="t2h::tapgemm_swap_kernel / tapgemm_kernel (tcgen05 implicit GEMM)",
                    achieved=achieved, peak=pk["tf_sustained"], unit="TFLOP/s", frac=achieved / pk["tf_sustained"],
                    traffic=traffic, traffic_note=traffic_note, peak_source=pk["source"] + ", bf16 sustained",
                    launches_per_step=len(rec), kernel_ms_per_step=t_ms,
                    kernel_share_of_step=t_ms / (ms_total / args.steps),
                    algorithmic_tflop_per_step=algo / 1e12,
                    issued_tensor_tflops=issued / (t_ms * 1e-3) / 1e12,
                    issued_frac=issued / (t_ms * 1e-3) / 1e12 / pk["tf_sustained"],
                    note="achieved = algorithmic FLOPs of the tap-GEMM launches AS EXECUTED (2*MAC; the reference's "
                         "nearest-x2 + 3x3 Upsample convs run folded into four 2x2 convs, so 11.71 TFLOP per batch "
                         "instead of the reference op graph's 12.55 that pipeline_tflops uses) / their summed CUDA-event "
                         "time; in fp32 mode each product is issued as 3 fp16 tensor-core products "
                         "(hi*hi+hi*lo+lo*hi), see issued_*")

    # ---------------- the same workload with the per-layer precision map (reported beside the headline) ----------------
    mixed = None
    if rank == 0 and world == 1 and not args.no_extra and args.precision == "fp32":
        ops.set_precision("mixed")
        try:
            for i in range(3):
                model.forward_step(xs_d[i % n_var], ms_d[i % n_var])
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.steps):
                model.forward_step(xs_d[i % n_var], ms_d[i % n_var])
            e1.record()
            torch.cuda.synchronize()
            ms_mx = e0.elapsed_time(e1) / args.steps
            mixed = dict(img_per_s=B / (ms_mx / 1e3), ms_per_step=ms_mx,
                         pipeline_frac_of_peak=B / (ms_mx / 1e3) * GFLOP_PER_IMG / 1e3 / pk["tf_sustained"],
                         note="ops.set_precision('mixed'): the six 128-ch 3x3 convs of the decoder's 512x256 level "
                              "single-product (profiles/r02_precision_map.txt), everything else 3-product; indices "
                              "bit-identical to the headline mode, pixels within 1e-3 of the reference "
                              "(tests/test_gpu_baseline_configs.py::test_config2_mixed_precision_map)")
        finally:
            ops.set_precision(args.precision)
    # ---------------- side measurements: BASELINE configs 3 and 4 (rank 0, N=1 only) ----------------
    extra = None
    if rank == 0 and world == 1 and not args.no_extra:
        extra = side_workloads(dev, args.precision)
        try:
            extra["sampler_train_step"] = train_workload(dev, args.precision, 1)
        except Exception as exc:
            extra["sampler_train_step"] = dict(error=repr(exc))
    eager = None
    if rank == 0 and world == 1 and not args.no_extra:
        eager = gpu_eager_baseline(dev, batch=B)
        for k in ("config2_fp32", "config2_tf32"):
            if k in eager:
                eager[k]["ours_over_eager"] = value / eager[k]["img_per_s"]
        if extra and "config4_sampler" in extra:
            for k in ("config4_fp32", "config4_tf32"):
                if k in eager:
                    eager[k]["ours_ms_per_step"] = extra["config4_sampler"]["ms_per_diffusion_step"]
    # ---------------- BASELINE config 5: the DDP training step (every rank takes part, every N) ----------------
    ddp_train = None
    if not args.no_train:
        try:
            ddp_train = vqgan_train_workload(dev, args.train_precision, rank, world)
        except Exception as exc:   # a failure here must not take the headline line down (symmetric on all ranks)
            ddp_train = dict(error=repr(exc))
        torch.cuda.empty_cache()
    if world > 1 and args.extra_train_ddp:  # opt-in: a collective runs inside (every rank takes part)
        tw = train_workload(dev, args.precision, world)
        extra = dict(sampler_train_step=tw) if rank == 0 else None

    if world > 1:
        dist.barrier()

    line = None
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            threads = host_threads()
            best, mean, times, kind = cpu_port_rate(threads, runs=3)
            cpu = dict(value=best, unit="img/s", cores=threads, kind=kind,
                       sample=f"best of 3 runs of 1 image 512x256 (mean {mean:.3f} img/s), torch fp32, the "
                              f"reference's own modules (oracle/_ref) when kind == 'reference', {threads} threads")
        line = dict(metric=METRIC, value=value, unit="img/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms_total / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32 (fp16x3 split products, fp32 accumulate)" if args.precision == "fp32"
                    else "f16 operands (TF32-like), fp32 accumulate",
                    data="synthetic",
                    config=dict(workload="vqvae_top.yml batch=16 512x256 encode-quantize-decode, codebook 18x1024x256",
                                batch_per_gpu=B, precision=args.precision, parallelism=f"replicas x{world}",
                                l2="activation working set (>2 GB/step) exceeds the 126 MB L2; inputs rotate "
                                   "over 3 distinct batches",
                                launch="CUDA graph replay of one forward_step" if args.graph else "per-kernel, asynchronous"),
                    clocks=clk,
                    e2e=dict(value=e2e_value, unit="img/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                             ms_per_step=ms_e2e / args.steps),
                    gpu_launches=launches, roofline=roof, cpu_baseline=cpu, gpu_eager_baseline=eager,
                    ddp_train=ddp_train, mixed_precision=mixed, extra=extra,
                    pipeline_tflops=value * GFLOP_PER_IMG / 1e3,
                    pipeline_frac_of_peak=value * GFLOP_PER_IMG / 1e3 / (pk["tf_sustained"] * world))
    if world > 1:
        dist.destroy_process_group()
    return line if rank == 0 else None


if __name__ == "__main__":
    main()
