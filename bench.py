#!/usr/bin/env python
"""bench.py -- masked-token train step (MaskGitTransformer base-256) on N B200s, one JSON line on rank 0.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference algorithm on the host CPU (oracle port, fp32 eager)

Workload = BASELINE.json configs[1]: MaskGitTransformer base (8x512, nh 8, I 2048, seq 257, vocab 2025),
class-conditional, bf16 compute, per-GPU batch 256 of synthetic pre-tokenised ImageNet-shaped samples
(random VQ ids + random class ids; the reference supports pre-encoded tokens and notes that images
"may be pre-encoded for faster training", README.md:137).  A step = the reference loop body
(training/train_maskgit_imagenet.py:403-452): masking recipe -> forward (logits, loss) -> backward ->
AdamW step -> zero_grad.  `value` times it with inputs resident in HBM; `e2e` adds the per-step
host->device copy of the token batch from pinned memory and a device->host read of the loss.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASE_CFG = dict(vocab_size=2025, max_position_embeddings=257, hidden_size=512, num_hidden_layers=8,
                num_attention_heads=8, intermediate_size=2048, codebook_size=1024, num_vq_tokens=256, num_classes=1000,
                hidden_dropout=0.0, attention_dropout=0.0)
PER_GPU_BATCH = 256
FWD_GFLOP_PER_IMG = 18.997  # SURVEY 8d / BASELINE.md section 3 (17.915 linear + 1.082 attention core)
METRIC = "images/sec masked-token train step (base-256)"


def mask_batch(tokens, class_ids, mask_id, codebook, gen=None):
    """prepare_inputs_and_labels without the VQ encode (training/train_maskgit_imagenet.py:375-393)."""
    B, S = tokens.shape
    dev = tokens.device
    timesteps = torch.rand(B, device=dev, generator=gen)
    mask_prob = torch.cos(timesteps * math.pi * 0.5).clip(0.0)
    n_mask = (S * mask_prob).round().clamp(min=1)
    perm = torch.rand(B, S, device=dev, generator=gen).argsort(dim=-1)
    mask = perm < n_mask.unsqueeze(-1)
    input_ids = torch.where(mask, mask_id, tokens)
    labels = torch.where(mask, tokens, -100)
    input_ids = torch.cat([(class_ids + codebook).unsqueeze(-1), input_ids], dim=-1)
    labels = torch.cat([torch.full((B, 1), -100, device=dev, dtype=labels.dtype), labels], dim=-1)
    return input_ids, labels


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def gemm_traffic_from_profile():
    """Average DRAM bytes (read + write) per tcgen05-GEMM launch from the committed `ncu --set full` capture of the step's
    GEMMs (profiles/r02_ncu_kernels.txt: one line per captured launch, sizes in GB / MB), or None."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_kernels.txt")
    if not os.path.exists(path):
        return None
    tot, n = 0.0, 0
    for line in open(path):
        if not line.startswith("gemm_tcgen05_kernel"):
            continue
        try:
            rd = line.split("dram_read=")[1].split()[0]
            wr = line.split("dram_write=")[1].split()[0]
            unit = lambda v: float(v[:-2]) * {"GB": 1e9, "MB": 1e6, "KB": 1e3}[v[-2:]]
            tot += unit(rd) + unit(wr)
            n += 1
        except Exception:
            pass
    return tot / n if n else None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md: ~1.4 PF sustained, 6.65 TB/s)"


def reference_kind():
    """"reference": the UNMODIFIED reference modules (oracle/_ref snapshot made by __graft_entry__.build() from
    /root/reference; git-ignored, travels with the repo) are what gets timed; "port": the oracle restatement."""
    from oracle import ref_snapshot

    return "reference" if ref_snapshot.available() else "port"


def reference_module_step_fn(batch, device="cpu"):
    """fwd + bwd + AdamW of the unmodified reference ``muse.MaskGitTransformer`` (torch eager; fp32 on the CPU, bf16
    autocast on cuda), the loop body of training/train_maskgit_imagenet.py:403-452 on pre-tokenised synthetic batches."""
    from oracle import ref_snapshot

    muse = ref_snapshot.import_reference()
    torch.manual_seed(0)
    model = muse.MaskGitTransformer(**BASE_CFG).to(device).train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, fused=(device != "cpu"))
    g = torch.Generator(device=device).manual_seed(1)

    def step():
        tokens = torch.randint(0, 1024, (batch, 256), generator=g, device=device)
        cls = torch.randint(0, 1000, (batch,), generator=g, device=device)
        inp, lab = mask_batch(tokens, cls, 2024, 1024, gen=g)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(device != "cpu")):
            _, loss = model(inp, labels=lab)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return float(loss.detach())

    return step


def cpu_reference_step_fn(batch, device="cpu"):
    """The reference arm's step: the unmodified reference modules when the oracle/_ref snapshot is present, else the
    oracle port (same torch op sequence, fp32 eager): fwd + bwd + AdamW on `batch` samples.  With device="cuda" the same
    eager ops run under bf16 autocast on the GPU -- what the reference executes on this B200 (the real bar)."""
    if reference_kind() == "reference":
        return reference_module_step_fn(batch, device)
    from oracle import transformer_oracle as T
    from open_muse_b200.modeling_transformer import MaskGitTransformer

    torch.manual_seed(0)
    params = {k: v.clone().to(device).requires_grad_(True) for k, v in MaskGitTransformer(**BASE_CFG).state_dict().items()}
    opt = torch.optim.AdamW(list(params.values()), lr=1e-4, weight_decay=0.01, fused=(device != "cpu"))
    g = torch.Generator(device=device).manual_seed(1)

    def step():
        tokens = torch.randint(0, 1024, (batch, 256), generator=g, device=device)
        cls = torch.randint(0, 1000, (batch,), generator=g, device=device)
        inp, lab = mask_batch(tokens, cls, 2024, 1024, gen=g)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(device != "cpu")):
            _, loss = T.forward(params, BASE_CFG, inp, labels=lab)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return float(loss.detach())

    return step


CPU_SAMPLE_BATCH = int(os.environ.get("MUSE_B200_CPU_SAMPLE_BATCH", "32"))  # the bounded CPU sample (tests shrink it)


def cpu_threads():
    """Threads for the CPU arm: every host core up to 64 (torch-eager fp32 at batch 32 stops scaling, and on a
    128-core box oversubscribing all of them was 10x SLOWER than 8 threads in the first measured run)."""
    return max(1, min(os.cpu_count() or 1, 64))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = cpu_threads()
    torch.set_num_threads(cores)
    on_gpu = args.ref_device == "cuda"
    batch = args.batch if on_gpu else CPU_SAMPLE_BATCH
    step = cpu_reference_step_fn(batch, args.ref_device)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    if on_gpu:
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()  # returns float(loss): synchronises every step
    dt = (time.perf_counter() - t0) / args.steps
    value = batch / dt
    sample = f"{args.steps} steps x batch {batch} of the base-256 train step (fwd+bwd+AdamW), " + (
        "bf16-autocast torch eager on cuda:0 (informational)" if on_gpu else "fp32 torch eager") + (
        "; unmodified reference modules (oracle/_ref)" if reference_kind() == "reference" else "; oracle port of the reference ops")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if on_gpu else "f32", "data": "synthetic",
        "ref_device": args.ref_device,
        "config": {"workload": f"MaskGitTransformer base (8x512, seq 257, vocab 2025) class-cond train step, {args.ref_device} sample batch {batch}",
                   "global_batch": batch, "seq_len": 257},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": reference_kind(), "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def _timeit(fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def kernel_rooflines(dev, peak_tf, peak_hbm):
    """Every named kernel of the hot path timed alone at its BASELINE-config shape (CUDA events on the launching stream,
    inputs >> L2 or freshly produced), with its ALGORITHMIC bytes / FLOPs (DESIGN.md section 4) against the measured
    peaks.  The ncu --set full captures of the same launches are committed under profiles/ (r02_ncu_kernels.txt)."""
    from open_muse_b200 import ops

    B, S, H, I, nh = 256, 257, 512, 2048, 8
    T = B * S
    out = []
    FP32_SIMT_TF = 148 * 128 * 2 * 1.965e9 / 1e12  # 148 SMs x 128 FMA lanes at the max SM clock

    def add(name, ms, nbytes=None, flops=None, bound=None, peak=None):
        if nbytes is not None:
            ach, pk, unit, bound = nbytes / (ms * 1e-3) / 1e9, peak_hbm, "GB/s", bound or "hbm"
            out.append({"kernel": name, "bound": bound, "algorithmic_bytes": nbytes, "us": ms * 1e3, "achieved": ach,
                        "peak": pk, "unit": unit, "frac": ach / pk})
        else:
            pk = peak or peak_tf
            ach = flops / (ms * 1e-3) / 1e12
            out.append({"kernel": name, "bound": bound or "tensor", "algorithmic_flops": flops, "us": ms * 1e3,
                        "achieved": ach, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk})

    bf = lambda *sh: torch.randn(*sh, device=dev).to(torch.bfloat16)
    # ---- norms / GLU / casts (HBM)
    x = torch.randn(T, H, device=dev)
    xb = bf(T, H)
    w = torch.ones(H, device=dev)
    dres = torch.randn(T, H, device=dev)
    _, st = ops.norm_fwd(x, w, 1e-6, torch.bfloat16)
    add("norm_fwd_warp_kernel fp32->bf16 [T,512]", _timeit(lambda: ops.norm_fwd(x, w, 1e-6, torch.bfloat16)), T * H * 6)
    add("norm_fwd_warp_kernel bf16->fp32 +residual", _timeit(lambda: ops.norm_fwd(xb, w, 1e-6, torch.float32, res=x)), T * H * 10)
    add("norm_bwd_warp_kernel bf16 dy, fp32 x, +dres (+ordered dw)",
        _timeit(lambda: ops.norm_bwd(xb, x, w, st, torch.float32, dres=dres, want_dw=True)), T * H * 14)
    add("norm_bwd_warp_kernel fp32 dy, bf16 x -> bf16 (+ordered dw)",
        _timeit(lambda: ops.norm_bwd(x, xb, w, st, torch.bfloat16, want_dw=True)), T * H * 8)
    add("cast_bf16_kernel", _timeit(lambda: ops.cast_bf16(x)), T * H * 6)
    ab, wI, dyI = bf(T, 2 * I), torch.ones(I, device=dev), bf(T, I)
    y, st4 = ops.norm_fwd(ab, wI, 1e-6, torch.bfloat16, act=2)
    add("glu_norm_fwd_kernel [T,2x2048]->[T,2048]", _timeit(lambda: ops.norm_fwd(ab, wI, 1e-6, torch.bfloat16, act=2)), T * I * 6)
    add("glu_norm_bwd_kernel (saved y, +ordered dw)",
        _timeit(lambda: ops.norm_bwd(dyI, ab, wI, st4, torch.bfloat16, act=2, y_fwd=y, want_dw=True)), T * I * 12)
    del ab, dyI, y
    # ---- embedding / loss
    ids = torch.randint(0, 1024, (B, S), device=dev)
    ids[torch.rand(B, S, device=dev) < 0.5] = 2024
    word, pos = torch.randn(2025, H, device=dev), torch.randn(S, H, device=dev)
    add("embed_fwd_kernel", _timeit(lambda: ops.embed_fwd(ids, word, pos)), T * H * 4 + T * 8)
    add("embed_bwd (sorted segments: plan + chunk + final + pos)", _timeit(lambda: ops.embed_bwd_det(ids, x, 2025, S)), 2 * T * H * 4)
    logits = bf(T, 2048)
    lab = torch.randint(0, 1024, (T,), device=dev)
    lab[torch.rand(T, device=dev) < 0.5] = -100
    lo, ws = ops.ce_fwd(logits, lab, 2025, 0.0)
    one = torch.ones(1, device=dev)
    add("ce_fwd_kernel (+ce_reduce) [T,2025]", _timeit(lambda: ops.ce_fwd(logits, lab, 2025, 0.0)), T * 2048 * 2)
    add("ce_bwd_kernel", _timeit(lambda: ops.ce_bwd(logits, lab, ws, one, lo, 2025, 0.0)), T * 2048 * 4)
    del logits
    # ---- attention (tensor)
    qkv = bf(T, 3 * H)
    o, lse = ops.attn_fwd(qkv[:, :H], qkv[:, H:2 * H], qkv[:, 2 * H:], B, nh, S, S, 0.125)
    do, dqkv = bf(T, H), torch.empty(T, 3 * H, dtype=torch.bfloat16, device=dev)
    fl = 4.0 * S * S * 64 * B * nh
    add("attn_fwd_tc_kernel (S=257: 3 balanced tiles)", _timeit(lambda: ops.attn_fwd(qkv[:, :H], qkv[:, H:2 * H], qkv[:, 2 * H:], B, nh, S, S, 0.125)), flops=fl)
    add("attn_bwd_dq_tc_kernel + attn_bwd_dkdv_tc_kernel",
        _timeit(lambda: ops.attn_bwd(qkv[:, :H], qkv[:, H:2 * H], qkv[:, 2 * H:], o, do, lse, dqkv[:, :H], dqkv[:, H:2 * H],
                                     dqkv[:, 2 * H:], B, nh, S, S, 0.125)), flops=2.5 * fl)
    del qkv, dqkv
    # ---- GEMMs by role (tensor)
    for name, N, K in [("qkv", 3 * H, H), ("attn out (+residual)", H, H), ("wi", 2 * I, H), ("wo (+residual)", H, I), ("logits", 2048, H)]:
        wt, xin, dyy = bf(N, K), bf(T, K), bf(T, N)
        res = torch.randn(T, N, device=dev) if "residual" in name else None
        f = 2.0 * T * N * K
        add(f"gemm_tcgen05_kernel fwd {name} [T,{K}]x[{N},{K}]", _timeit(lambda: ops.linear_fwd(xin, wt, res=res)), flops=f)
        add(f"gemm_tcgen05_kernel dgrad {name}", _timeit(lambda: ops.linear_dgrad(dyy, wt)), flops=f)
        add(f"gemm_tcgen05_kernel wgrad {name} (deterministic split-K)", _timeit(lambda: ops.linear_wgrad_det(dyy, xin)), flops=f)
        del wt, xin, dyy, res
    # ---- tokenizer search and the decode-step kernel
    n = 128 * 256
    z, cb = torch.randn(n, 256, device=dev), torch.randn(1024, 256, device=dev)
    add("vq_argmin_kernel (config 3: 32768 rows x 1024 codes x 256)", _timeit(lambda: ops.vq_argmin(z, cb)),
        flops=2.0 * n * 1024 * 256, bound="fp32-simt", peak=FP32_SIMT_TF)
    Bg, L, K = 64, 256, 1024
    lg = bf(Bg, L + 1, K)
    cur = torch.full((Bg, L), 2024, dtype=torch.long, device=dev)
    q = torch.empty(Bg * L, K, device=dev).exponential_(1)
    u = torch.rand(Bg, L, device=dev)
    add("sample_step_kernel (config 5: 64 x 256 x 1024)",
        _timeit(lambda: ops.sample_step(lg, cur, q, u, K, 2024, 100, 0.5, skip_first_token=True)), Bg * L * K * 6)
    # ---- one full-resolution tokenizer convolution + its GroupNorm producer stage
    xc = torch.randn(8, 256, 256, 128, device=dev)
    wc = torch.randn(128, 128, 3, 3, device=dev) * 0.03
    ga, be = torch.ones(128, device=dev), torch.zeros(128, device=dev)
    ms = _timeit(lambda: ops.conv2d(xc, wc, gn=(ga, be, 32, 1e-6)), n=5, warm=2)
    add("groupnorm+SiLU+split -> conv_tc_kernel 3x3 128->128 @256x256 (bf16x3, B=8)", ms, flops=3 * 2.0 * 8 * 256 * 256 * 128 * 128 * 9)
    return out


def t2i_pipeline_latency(dev):
    """benchmark/muse_perf.py:241-293 on this box: PipelineMuse(default-config MaskGiTUViT_v2, ~603 M parameters, taming f16
    VQGANModel) with 12 steps and classifier-free guidance, 256 px (256 tokens) and 512 px (1024 tokens, force_down_up_sample
    as the reference's 512-px model), batch 1 and 8, PIL output.  Random weights, bf16; the CLIP text encoder is third party
    and not in the timed region (precomputed states go in, as `prompt_embeds=`).  BASELINE.md section 2 holds the A100 / RTX 4090
    figures of the reference harness (fp16, text encoder included) -- context, different hardware."""
    from open_muse_b200 import MaskGiTUViT_v2, PipelineMuse
    from open_muse_b200.modeling_taming_vqgan import VQGANModel

    torch.manual_seed(2)
    vae = VQGANModel(num_embeddings=8192).to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(3)
    emb = lambda *s: torch.randn(*s, device=dev, generator=g)
    kw = dict(prompt_embeds=emb(1, 77, 768), pooled_embeds=emb(1, 768), negative_prompt_embeds=emb(1, 77, 768),
              negative_pooled_embeds=emb(1, 768), timesteps=12)
    rows = {}
    for res in (256, 512):
        torch.manual_seed(4)
        tr = MaskGiTUViT_v2(force_down_up_sample=(res == 512))
        with torch.no_grad():  # the zero-initialised output conv would make every logit equal: draw it like the other weights
            torch.nn.init.trunc_normal_(tr.mlm_layer.conv1.weight, std=0.02)
        tr = tr.to(dev).eval()
        pipe = PipelineMuse(vae=vae, transformer=tr, is_class_conditioned=False).to(dev)
        for bs in (1, 8):
            run = lambda: pipe(**kw, num_images_per_prompt=bs, transformer_seq_len=(res // 16) ** 2, generator=g)
            imgs = run()
            assert len(imgs) == bs and imgs[0].size == (res, res), (len(imgs), imgs[0].size)
            ms = _timeit(run, n=3, warm=1)
            rows[f"{res}px_bs{bs}"] = {"latency_ms": ms, "images_per_s": bs / (ms * 1e-3)}
        del tr, pipe
        torch.cuda.empty_cache()
    return {"unit": "ms", "rows": rows,
            "config": "PipelineMuse text-to-image, MaskGiTUViT_v2 class defaults (22 layers x 1024, 3+3 res/attention blocks x 768, "
                      "codebook 8192) + taming VQGANModel decode + PIL, 12 steps, CFG (2x batch inside), bf16, random weights, "
                      "text encoder excluded; 512 px = force_down_up_sample (reference benchmark/muse_perf.py:241-293)",
            "reference_published_ms": {"A100 256px_bs1": 474.0, "A100 512px_bs1": 538.5, "A100 256px_bs8": 601.8,
                                       "A100 512px_bs8": 1004.5, "RTX4090 256px_bs8": 454.1, "RTX4090 512px_bs8": 763.3,
                                       "source": "benchmark/artifacts/all.csv (fp16, xformers + fused norm, text encoder included)"}}


def secondary_metrics(dev, base_model, peak_tf, peak_hbm):
    """The rest of BASELINE.json's metric and configs on the same box: decode steps/sec (config 5), the tokenizer round
    trip (config 3), the reference recipe in torch eager on this same GPU (the real bar), per-kernel rooflines."""
    from open_muse_b200 import MaskGitVQGAN, ops

    out = {}
    # ---- config 5: generate2, base model, B=64, 256 tokens, 12 steps (the whole loop replayed as one CUDA graph)
    base_model.eval()
    gen = torch.Generator(device=dev).manual_seed(7)
    cls0 = torch.randint(0, 1000, (64,), device=dev)

    def dec(graph):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return base_model.generate2(class_ids=cls0.clone(), timesteps=12, generator=gen, use_cuda_graph=graph)

    ms_g = _timeit(lambda: dec(True), n=5, warm=2)
    l0 = ops.launches()
    ms_e = _timeit(lambda: dec(False), n=3, warm=1)
    out["decode_steps_per_s"] = {"value": 12 / (ms_g * 1e-3), "unit": "steps/s", "ms_per_step": ms_g / 12, "ms_per_call": ms_g,
                                 "images_per_s": 64 / (ms_g * 1e-3), "host_launches_per_call": 5,
                                 "config": "generate2, base-256 model, B=64, 256 tokens, 12 steps, temperature 1.0; whole loop "
                                           "replayed as one CUDA graph (+4 input copies)",
                                 "launched_one_by_one": {"steps_per_s": 12 / (ms_e * 1e-3), "ms_per_call": ms_e,
                                                         "kernels_per_call": (ops.launches() - l0) // 4}}
    base_model.train()
    # ---- config 3: MaskGitVQGAN f16-256 encode -> ids -> decode_code, B=128 (chunks of 64)
    torch.manual_seed(1)
    vq = MaskGitVQGAN().to(dev).eval()
    pix = torch.rand(128, 3, 256, 256, device=dev)
    ids = torch.cat([vq.get_code(pix[j:j + 64]) for j in range(0, 128, 64)])
    ms_enc = _timeit(lambda: [vq.get_code(pix[j:j + 64]) for j in range(0, 128, 64)], n=2, warm=1)
    ms_dec = _timeit(lambda: [vq.decode_code(ids[j:j + 64]) for j in range(0, 128, 64)], n=2, warm=1)
    out["vqgan_roundtrip"] = {"value": 128 / ((ms_enc + ms_dec) * 1e-3), "unit": "images/s", "batch": 128, "encode_ms": ms_enc,
                              "decode_ms": ms_dec, "encode_images_per_s": 128 / (ms_enc * 1e-3),
                              "decode_images_per_s": 128 / (ms_dec * 1e-3),
                              "model_tflops": (128.76 + 186.55) * 128 / (ms_enc + ms_dec),
                              "config": "MaskGitVQGAN f16-256 (class defaults) encode -> ids -> decode_code, fp32-faithful bf16x3 "
                                        "tcgen05 convolutions, bit-exact arg-min"}
    del vq, pix
    torch.cuda.empty_cache()
    # ---- the reference recipe in torch eager on this GPU (bf16 autocast): what the unmodified reference runs here
    try:
        rstep = cpu_reference_step_fn(PER_GPU_BATCH, "cuda")
        for _ in range(2):
            rstep()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            rstep()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 3
        out["torch_eager_same_gpu"] = {"value": PER_GPU_BATCH / dt, "unit": "images/s", "ms_per_step": dt * 1e3,
                                       "kind": reference_kind(),
                                       "config": "the reference train step (fwd + bwd + AdamW, bf16 autocast, cuBLAS/ATen kernels) "
                                                 f"at batch {PER_GPU_BATCH} on this B200"}
        del rstep
    except Exception as e:  # informational leg: never sinks the bench line
        out["torch_eager_same_gpu"] = {"error": f"{type(e).__name__}: {e}"}
    torch.cuda.empty_cache()
    try:  # informational leg (the reference's own published benchmark harness), never sinks the bench line
        out["t2i_pipeline_latency"] = t2i_pipeline_latency(dev)
    except Exception as e:
        out["t2i_pipeline_latency"] = {"error": f"{type(e).__name__}: {e}"}
    torch.cuda.empty_cache()
    out["roofline_kernels"] = kernel_rooflines(dev, peak_tf, peak_hbm)
    return out


DUMP_SAMPLE = 1 << 16  # elements kept per parameter tensor in --dump-outputs
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, model, losses):
    """Writes what the timed train step leaves its caller after the last timed step, as float32 .npy files: the loss of
    every step of the last timed loop (losses.npy) and every updated parameter (param.<name>.npy; tensors larger than
    DUMP_SAMPLE elements as the same fixed, seeded sample of positions in every run).  About 15 MB for the base model."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    arrays = {"losses": np.asarray(losses, dtype=np.float32)}
    for name, p in model.named_parameters():
        flat = p.detach().float().flatten()
        if flat.numel() > DUMP_SAMPLE:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            flat = flat[idx.to(flat.device)]
        arrays[f"param.{name}"] = flat.cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, total
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="per-GPU batch (default = BASELINE config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-step", action="store_true", help="skip the extra 'train step incl. VQ encode' measurement")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip decode steps/s, the tokenizer round trip, torch-eager-on-this-GPU and the per-kernel rooflines")
    ap.add_argument("--no-cuda-graph", action="store_true",
                    help="launch the kernels of each step one by one instead of replaying the captured step (N=1 default: graph)")
    ap.add_argument("--ddp-graph", type=int, default=int(os.environ.get("MUSE_B200_DDP_GRAPH", "1")),
                    help="N>1: capture the whole DDP step (NCCL bucket all-reduces included) in one CUDA graph")
    ap.add_argument("--nccl-sms", type=int, default=int(os.environ.get("MUSE_B200_NCCL_SMS", "0")),
                    help="N>1: SMs left to NCCL (NCCL_MAX_NCHANNELS is capped to the same number); 0 = full GEMM grids, NCCL default")
    ap.add_argument("--nccl-channels", type=int, default=0,
                    help="N>1 diagnostic: cap NCCL_MAX_NCHANNELS without shrinking the GEMM grids (0 = NCCL default)")
    ap.add_argument("--ddp-no-sync", action="store_true",
                    help="N>1 DIAGNOSTIC ONLY (invalid as a result): DDP wrapper with the gradient all-reduce skipped, to "
                         "separate launch overhead from NCCL contention")
    ap.add_argument("--optimizer", default="torch", choices=["torch", "fused"],
                    help="torch.optim.AdamW(fused=True) or open_muse_b200.FusedAdamW (AdamW + bf16 operand packing in one pass)")
    ap.add_argument("--pdl", type=int, default=None, choices=[0, 1],
                    help="programmatic dependent launch for the library's kernels (default: the library's own default / MUSE_B200_PDL)")
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"],
                    help="--impl reference only: cpu (the reference arm) or cuda (same eager ops under bf16 autocast, informational)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the losses of the last timed loop and (a seeded sample of) the updated "
                         "parameters as DIR/<name>.npy (float32), to compare two builds output for output")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from open_muse_b200 import ops
    from open_muse_b200.modeling_transformer import MaskGitTransformer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.pdl is not None:
        ops.set_pdl(bool(args.pdl))
    ddp_graph = world > 1 and bool(args.ddp_graph) and not args.no_cuda_graph
    if world > 1:
        if ddp_graph:  # graph capture of NCCL collectives: the watchdog must not poll events while the stream is capturing
            os.environ["TORCH_NCCL_ASYNC_ERROR_HANDLING"] = "0"
        if args.nccl_sms > 0:
            # the gradient all-reduce needs ~11 GB/s here (144 MB per 13 ms of backward): a few NCCL channels (= CTAs = SMs)
            # are plenty on NVLink 5, and the persistent GEMMs give exactly those SMs up instead of stalling behind them
            os.environ.setdefault("NCCL_MAX_NCHANNELS", str(args.nccl_sms))
            os.environ.setdefault("NCCL_MIN_NCHANNELS", str(min(2, args.nccl_sms)))
            ops.reserve_sms(args.nccl_sms)
        elif args.nccl_channels > 0:
            os.environ["NCCL_MAX_NCHANNELS"] = str(args.nccl_channels)
            os.environ["NCCL_MIN_NCHANNELS"] = str(min(2, args.nccl_channels))
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(3, args.warmup)
    B = args.batch

    torch.manual_seed(0)
    model = MaskGitTransformer(**BASE_CFG).to(dev).train()
    net = model
    if world > 1:
        if ddp_graph:  # DDP constructed on a side stream (torch's recipe for capturing a DDP step)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True)
            torch.cuda.current_stream().wait_stream(side)
        else:
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True)
    use_graph = (world == 1 or ddp_graph) and not args.no_cuda_graph
    if args.optimizer == "fused":
        from open_muse_b200 import FusedAdamW

        opt = FusedAdamW(model.parameters(), lr=1e-4, weight_decay=0.01, model=model)
    else:
        opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, fused=True, capturable=use_graph)
    gen = None if use_graph else torch.Generator(device=dev).manual_seed(100 + rank)  # graph capture: default generator
    torch.cuda.manual_seed(100 + rank)
    n_buf = 4
    host_tok = [torch.randint(0, 1024, (B, 256), generator=torch.Generator().manual_seed(1000 * rank + i)).pin_memory() for i in range(n_buf)]
    host_cls = [torch.randint(0, 1000, (B,), generator=torch.Generator().manual_seed(2000 * rank + i)).pin_memory() for i in range(n_buf)]
    dev_tok = [t.to(dev) for t in host_tok]
    dev_cls = [t.to(dev) for t in host_cls]

    import contextlib

    no_sync = net.no_sync if (world > 1 and args.ddp_no_sync) else contextlib.nullcontext

    def step(tokens, cls):
        inp, lab = mask_batch(tokens, cls, 2024, 1024, gen=gen)
        with no_sync():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                _, loss = net(inp, labels=lab)
            loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / n

    for i in range(warmup):
        step(dev_tok[i % n_buf], dev_cls[i % n_buf])
    torch.cuda.synchronize()
    l_eager = ops.launches()
    step(dev_tok[0], dev_cls[0])
    launches_per_step = ops.launches() - l_eager  # kernels of this package per step (a replayed graph launches the same)
    run = step
    if use_graph:  # the whole step (masking, fwd, loss, bwd, AdamW) captured once, replayed per step
        from open_muse_b200.graphs import GraphedStep

        try:
            # DDP: >= 11 eager warm-up iterations before capture (torch's documented requirement), thread-local capture mode
            run = GraphedStep(step, (dev_tok[0], dev_cls[0]), warmup=12 if world > 1 else 2,
                              capture_error_mode="thread_local" if world > 1 else "global")
            for i in range(2):
                run(dev_tok[i % n_buf], dev_cls[i % n_buf])
        except Exception as e:  # same kernels launched one by one (reported in config.cuda_graph)
            print(f"bench: CUDA graph capture failed ({type(e).__name__}: {e}); timing the eager launch path", file=sys.stderr)
            torch.cuda.synchronize()
            run, use_graph = step, False
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev = timed(lambda i: run(dev_tok[i % n_buf], dev_cls[i % n_buf]), args.steps)
    launches = launches_per_step * args.steps

    # e2e: every step copies its inputs from pinned host memory and copies its loss back to pinned host memory; the host
    # consumes the loss of step i-1 while step i runs (lagged logging, the usual training-loop practice), so the device
    # never idles behind a host round trip.  The last losses are consumed before the closing barrier.
    loss_host = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_evt = [torch.cuda.Event() for _ in range(2)]
    seen = []

    # inputs: step i+1's tokens are copied host -> device on a copy stream (two staging slots) while step i computes
    copy_stream = torch.cuda.Stream()
    stage = [(torch.empty_like(dev_tok[0]), torch.empty_like(dev_cls[0])) for _ in range(2)]
    staged, consumed = [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)]
    for ev in consumed:
        ev.record()

    def prefetch(i):
        k = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k])  # the slot's previous occupant (step i-2) has been read by its step
            stage[k][0].copy_(host_tok[i % n_buf], non_blocking=True)
            stage[k][1].copy_(host_cls[i % n_buf], non_blocking=True)
            staged[k].record(copy_stream)

    def e2e_step(i):
        if i == 0:
            prefetch(0)
        k = i & 1
        torch.cuda.current_stream().wait_event(staged[k])
        loss = run(stage[k][0], stage[k][1])
        consumed[k].record()
        if i + 1 < args.steps:
            prefetch(i + 1)
        slot = i & 1
        if i >= 2:  # the slot's previous occupant (step i-2) has certainly landed: consume it on the host
            loss_evt[slot].synchronize()
            seen.append(float(loss_host[slot]))
        loss_host[slot].copy_(loss.detach(), non_blocking=True)  # device->host read of this step's loss
        loss_evt[slot].record()
        if i == args.steps - 1:  # drain: every step's loss has been read by the host inside the timed region
            for k in ((i - 1) & 1, slot) if i >= 1 else (slot,):
                loss_evt[k].synchronize()
                seen.append(float(loss_host[k]))

    ms_e2e = timed(e2e_step, args.steps)
    assert len(seen) == args.steps and all(math.isfinite(v) for v in seen), seen
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before the profiled steps below move the parameters again
        dump_outputs(args.dump_outputs, model, seen)
    model._packed.key = None  # graph replays update the parameters without bumping their version counters: re-pack for eager use

    # ---- roofline of the dominant kernel (tcgen05 GEMM), measured live with CUDA events around every launch
    peak_tf, peak_hbm, peak_src = measured_peaks()
    ops.profile_gemms(True)
    for i in range(2):
        step(dev_tok[i % n_buf], dev_cls[i % n_buf])
    torch.cuda.synchronize()
    gemm_ms, gemm_flops, gemm_n = ops.profile_gemms(False)
    roof = None
    if gemm_n:
        ach = gemm_flops / (gemm_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all Linear fwd/dgrad/wgrad GEMMs of the step)",
                "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "traffic": gemm_traffic_from_profile(), "algorithmic_flops_per_launch": gemm_flops / gemm_n,
                "peak_source": peak_src, "launches_per_step": gemm_n // 2,
                "gemm_share_of_step": (gemm_ms / 2) / ms_dev}

    # ---- BASELINE config 2 (ii): the same train step fed from pixels, i.e. including the frozen MaskGitVQGAN tokeniser
    # (train_maskgit_imagenet.py:357-369: fp32, no autocast) in front of the transformer step.  N=1 only, informational.
    full = None
    if world == 1 and not args.no_full_step:
        from open_muse_b200 import MaskGitVQGAN

        torch.manual_seed(1)
        vq = MaskGitVQGAN().to(dev).eval()
        pix = torch.rand(B, 3, 256, 256, device=dev)
        chunk = 64

        def tokenise():
            return torch.cat([vq.get_code(pix[j:j + chunk]) for j in range(0, B, chunk)])

        def full_step(i):
            return step(tokenise(), dev_cls[i % n_buf])

        full_step(0)
        ms_full = timed(full_step, 3)
        ms_enc = timed(lambda i: tokenise(), 3)
        full = {"value": B / (ms_full * 1e-3), "unit": "images/s", "ms_per_step": ms_full, "vq_encode_ms": ms_enc,
                "vq_encode_images_per_s": B / (ms_enc * 1e-3),
                "note": "pixels resident in HBM -> MaskGitVQGAN f16-256 get_code (fp32-faithful bf16x3 tcgen05 convs) -> "
                        "masking -> train step; random-init tokeniser"}
        # fast tokenizer mode: single-pass bf16 convolutions (the accuracy class of the reference's own TF32 GPU path)
        with torch.no_grad():
            z0 = vq._encode_nhwc(pix[:chunk])
            vq.quantize.embedding.weight.copy_(torch.randn(1024, 256, device=dev) * z0.std())  # non-degenerate arg-min
        ids_exact = tokenise()
        vq.set_conv_precision("bf16")
        ids_fast = tokenise()
        full_step(0)
        ms_full_f = timed(full_step, 3)
        ms_enc_f = timed(lambda i: tokenise(), 3)
        vq.set_conv_precision("bf16x3")
        full["fast_tokenizer_mode"] = {
            "value": B / (ms_full_f * 1e-3), "unit": "images/s", "ms_per_step": ms_full_f, "vq_encode_ms": ms_enc_f,
            "vq_encode_images_per_s": B / (ms_enc_f * 1e-3),
            "token_id_agreement_with_exact_mode": float((ids_fast == ids_exact).float().mean()),
            "note": "MaskGitVQGAN.set_conv_precision('bf16'): one bf16 tensor-core product per fp32 product; codebook re-drawn "
                    "N(0, std(z)) for the agreement rate (random-init weights)"}
        del vq, pix
        torch.cuda.empty_cache()

    secondary = None
    if world == 1 and not args.no_secondary:
        secondary = secondary_metrics(dev, model, peak_tf, peak_hbm)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = cpu_threads()
        torch.set_num_threads(cores)
        cstep = cpu_reference_step_fn(CPU_SAMPLE_BATCH)
        cstep()
        t0 = time.perf_counter()
        n = 0
        while n < 2 or (time.perf_counter() - t0 < 15 and n < 12):
            cstep(); n += 1
        cdt = (time.perf_counter() - t0) / n
        cpu = {"value": CPU_SAMPLE_BATCH / cdt, "unit": "images/s", "cores": cores, "kind": reference_kind(),
               "sample": f"{n} steps x batch {CPU_SAMPLE_BATCH} of the same train step, fp32 torch eager on {cores} host threads, "
                         + ("unmodified reference modules (oracle/_ref)" if reference_kind() == "reference" else "oracle port")}

    if rank == 0:
        gb = B * world
        out = {
            "metric": METRIC, "value": gb / (ms_dev * 1e-3), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "MaskGitTransformer base (8x512, nh8, I2048, seq 257, vocab 2025) class-cond train step: "
                                   "masking + fwd + loss + bwd + AdamW, pre-tokenised synthetic ImageNet batch",
                       "global_batch": gb, "per_gpu_batch": B, "seq_len": 257,
                       "parallelism": f"dp{world}" if world > 1 else "single",
                       "l2": "no explicit flush: per-step working set (~15 GB activations + 0.5 GB weights/grads/optimizer) >> 126 MB L2",
                       "cuda_graph": bool(use_graph), "pdl": ops.get_pdl(), "optimizer": args.optimizer,
                       "nccl_sms_reserved": args.nccl_sms if world > 1 else 0,
                       **({"nccl_max_channels": args.nccl_channels} if world > 1 and args.nccl_channels else {}),
                       **({"DIAGNOSTIC_no_allreduce": True} if world > 1 and args.ddp_no_sync else {})},
            "e2e": {"value": gb / (ms_e2e * 1e-3), "unit": "images/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": world * (B * 256 * 8 + B * 8), "d2h_bytes_per_step": world * 4,
                    "api": "MaskGitTransformer.forward / loss.backward / optimizer.step (the captured step); every step's tokens "
                           "are copied from pinned host memory on a copy stream while the previous step computes (double "
                           "buffered), its loss is copied to pinned host memory and read by the host one step later"},
            "gpu_launches": launches,
            "tflops_per_gpu_model": 3 * FWD_GFLOP_PER_IMG * B / ms_dev,
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "full_step_incl_vq_encode": full,
        }
        if secondary:
            out.update(secondary)
        print(json.dumps(out))
    if world > 1:
        run = None  # drop the captured graph (its NCCL nodes) before the process group goes away
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
