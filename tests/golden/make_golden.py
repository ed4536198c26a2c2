#!/usr/bin/env python
"""Generates the golden fixtures in this directory by running the UNMODIFIED reference
(huggingface/open-muse @ 64e1afe, mounted at /root/reference) on CPU in fp32.

The reference has no tests, goldens or known-answer vectors of its own (SURVEY.md section 4), so
these outputs of the reference itself are what pins oracle/ (and, through the oracle, the CUDA path).
Run from the repo root, in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

`accelerate` is not installed; the reference imports two symbols from it that are only used by
`from_pretrained(low_cpu_mem_usage=True)`, so a two-symbol in-memory stub is registered (SURVEY 8c).
"""
import contextlib
import math
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("MUSE_REFERENCE", "/root/reference")


def import_reference():
    import transformers  # noqa: F401  (must be imported before the accelerate stub is registered)

    if "accelerate" not in sys.modules:
        acc = types.ModuleType("accelerate")
        acc.init_empty_weights = contextlib.nullcontext
        accu = types.ModuleType("accelerate.utils")
        accu.set_module_tensor_to_device = lambda *a, **k: None
        acc.utils = accu
        acc.__spec__ = None
        sys.modules["accelerate"] = acc
        sys.modules["accelerate.utils"] = accu
    sys.path.insert(0, REF)
    import muse  # the reference package

    assert os.path.realpath(muse.__file__).startswith(os.path.realpath(REF)), muse.__file__
    return muse


MICRO = dict(vocab_size=72, hidden_size=64, num_hidden_layers=2, num_attention_heads=1, intermediate_size=128,
             hidden_dropout=0.0, attention_dropout=0.0, max_position_embeddings=17, codebook_size=64,
             num_vq_tokens=16, num_classes=7, layer_norm_eps=1e-6)
MICRO_T2I = dict(vocab_size=72, hidden_size=64, num_hidden_layers=2, num_attention_heads=1, intermediate_size=128,
                 hidden_dropout=0.0, attention_dropout=0.0, max_position_embeddings=16, codebook_size=64,
                 num_vq_tokens=16, add_cross_attention=True, encoder_hidden_size=32, norm_type="rmsnorm",
                 use_normformer=False, layer_norm_eps=1e-6, use_codebook_size_for_output=True)
MICRO_T2I_PROJ = dict(vocab_size=72, hidden_size=64, num_hidden_layers=2, num_attention_heads=1, intermediate_size=128,
                      hidden_dropout=0.0, attention_dropout=0.0, max_position_embeddings=16, codebook_size=64,
                      num_vq_tokens=16, add_cross_attention=True, encoder_hidden_size=32,
                      project_encoder_hidden_states=True, norm_type="layernorm", use_normformer=True, layer_norm_eps=1e-6)
MICRO_V2 = dict(hidden_size=128, num_attention_heads=2, in_channels=64, block_out_channels=(64,), block_num_heads=1,
                num_res_blocks=1, num_hidden_layers=2, intermediate_size=128, vocab_size=72, codebook_size=64,
                encoder_hidden_size=32, cond_embed_dim=16, micro_cond_encode_dim=8, micro_cond_embed_dim=40,
                norm_type="rmsnorm")
TINY = dict(vocab_size=2025, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
            hidden_dropout=0.0, attention_dropout=0.0, max_position_embeddings=257, codebook_size=1024,
            num_vq_tokens=256, num_classes=1000)
MICRO_VQ = dict(resolution=32, num_channels=3, hidden_channels=32, channel_mult=(1, 2), num_res_blocks=1,
                z_channels=16, num_embeddings=64, quantized_embed_dim=16)


def masked_batch(gen, B, S, codebook, n_classes, mask_id):
    """The masking recipe of training/train_maskgit_imagenet.py:375-393 (class-conditional)."""
    tokens = torch.randint(0, codebook, (B, S), generator=gen)
    class_ids = torch.randint(0, n_classes, (B,), generator=gen)
    timesteps = torch.rand(B, generator=gen)
    mask_prob = torch.cos(timesteps * math.pi * 0.5).clip(0.0)
    n_mask = (S * mask_prob).round().clamp(min=1)
    rand = torch.rand(B, S, generator=gen)
    perm = rand.argsort(dim=-1)
    mask = perm < n_mask.unsqueeze(-1)
    input_ids = torch.where(mask, mask_id, tokens)
    labels = torch.where(mask, tokens, -100)
    input_ids = torch.cat([(class_ids + codebook).unsqueeze(-1), input_ids], dim=-1)
    labels = torch.cat([torch.full((B, 1), -100), labels], dim=-1)
    return dict(tokens=tokens, class_ids=class_ids, timesteps=timesteps, rand=rand, input_ids=input_ids, labels=labels)


def grads_of(model):
    return {n: p.grad.detach().clone() for n, p in model.named_parameters()}


def make_f16_256(muse):
    """(9) BASELINE config 3 at its own size: MaskGitVQGAN f16-256 (class defaults, modeling_maskgit_vqgan.py:353-367),
    default init from a seed (no weights stored: construction order == RNG order, checked through per-tensor signatures),
    codebook re-drawn N(0, std(z)) so that the arg-min is not degenerate (SURVEY H1), two rand images.  Stores the encoder
    output, the token ids with their top-2 distance margins, the quantised latents and the reconstruction."""
    torch.manual_seed(60)
    v = muse.MaskGitVQGAN()
    v.eval()
    init_sig = {k: (float(x.double().sum()), float(x.double().norm())) for k, x in v.state_dict().items()}
    img = torch.rand(2, 3, 256, 256, generator=torch.Generator().manual_seed(61))
    with torch.no_grad():
        z = v.encoder(img)
        cb = torch.randn(1024, 256, generator=torch.Generator().manual_seed(62)) * z.std()
        v.quantize.embedding.weight.copy_(cb)
        zq, ids = v.encode(img)
        rec = v.decode_code(ids)
        d = v.quantize.compute_distances(z.permute(0, 2, 3, 1).contiguous())
        top2 = d.topk(2, dim=1, largest=False).values
    margin = top2[:, 1] - top2[:, 0]
    rel = margin / top2[:, 0].abs()
    print("f16-256 vqgan: z std", float(z.std()), "min top-2 margin", float(margin.min()), "relative", float(rel.min()),
          "rows with relative margin < 1e-4:", int((rel < 1e-4).sum()), "of", rel.numel(), "distinct ids", ids.unique().numel())
    torch.save(dict(seed=60, image_seed=61, codebook_seed=62, init_signature=init_sig, codebook=cb.clone(), z=z.clone(),
                    ids=ids.clone(), z_q=zq.clone(), recon=rec.clone(), dmin=top2[:, 0].clone(), margin=margin.clone()),
               os.path.join(HERE, "f16_256_vqgan.pt"))


def make_signatures(muse):
    """(10) the public call signatures of the boundary (parameter names, order and defaults), as JSON."""
    import inspect
    import json

    from muse.modeling_transformer_v2 import MaskGiTUViT_v2
    from muse.modeling_taming_vqgan import VQGANModel

    def sig(fn):
        out = []
        for name, p in inspect.signature(fn).parameters.items():
            d = p.default
            if d is inspect.Parameter.empty:
                d = "<required>"
            elif callable(d):
                d = f"<callable {getattr(d, '__name__', type(d).__name__)}>"
            elif isinstance(d, tuple):
                d = list(d)
            out.append([name, str(p.kind), d])
        return out

    table = {
        "MaskGitTransformer.__init__": sig(muse.MaskGitTransformer.__init__),
        "MaskGitTransformer.forward": sig(muse.MaskGitTransformer.forward),
        "MaskGitTransformer.generate2": sig(muse.MaskGitTransformer.generate2),
        "MaskGiTUViT_v2.forward": sig(MaskGiTUViT_v2.forward),
        "MaskGiTUViT_v2.generate2": sig(MaskGiTUViT_v2.generate2),
        "MaskGitVQGAN.__init__": sig(muse.MaskGitVQGAN.__init__),
        "MaskGitVQGAN.encode": sig(muse.MaskGitVQGAN.encode),
        "MaskGitVQGAN.get_soft_code": sig(muse.MaskGitVQGAN.get_soft_code),
        "VQGANModel.__init__": sig(VQGANModel.__init__),
        "PipelineMuse.__init__": sig(muse.PipelineMuse.__init__),
        "PipelineMuse.__call__": sig(muse.PipelineMuse.__call__),
        "PipelineMuseInpainting.__call__": sig(muse.PipelineMuseInpainting.__call__),
        "EMAModel.__init__": sig(muse.EMAModel.__init__),
    }
    with open(os.path.join(HERE, "signatures.json"), "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
    print("signatures:", ", ".join(f"{k} ({len(v)})" for k, v in table.items()))


def make_uvit_downup(muse):
    """MaskGiTUViT_v2 with force_down_up_sample=True (modeling_transformer_v2.py:505-583): Norm2D + k2s2 conv before the down
    block, Norm2D + ConvTranspose2d(2, 2) after the up block.  8x8 tokens -> 4x4 inside the network.  Same re-draw of the
    zero-initialised tensors as fixture (6)."""
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    cfg = dict(MICRO_V2, force_down_up_sample=True)
    torch.manual_seed(60)
    v2 = MaskGiTUViT_v2(**cfg)
    init_sig = {k: (float(x.double().sum()), float(x.double().norm())) for k, x in v2.state_dict().items()}
    g = torch.Generator().manual_seed(61)
    with torch.no_grad():
        for k, x in v2.state_dict().items():
            if "adaLN_modulation.mapper" in k or k.endswith("gamma") or k.endswith("beta") or k == "mlm_layer.conv1.weight":
                x.copy_(torch.randn(x.shape, generator=g) * 0.05)
            elif k.endswith("norm.weight"):
                x.copy_(1.0 + 0.1 * torch.randn(x.shape, generator=g))
    v2.eval()
    B, S = 2, 64
    ids = torch.randint(0, 64, (B, S), generator=g)
    mask = torch.rand(B, S, generator=g) < 0.6
    inp = torch.where(mask, 71, ids)
    lab = torch.where(mask, ids, -100)
    enc = torch.randn(B, 5, 32, generator=g)
    ce = torch.randn(B, 16, generator=g)
    mc = torch.tensor([[256.0, 256.0, 0.0, 0.0, 6.0], [512.0, 384.0, 10.0, 20.0, 5.5]])
    stages = {}
    hooks = [v2.down_blocks[0].downsample.register_forward_hook(lambda m, i, o: stages.__setitem__("downsample", o.detach().clone())),
             v2.up_blocks[0].upsample.register_forward_hook(lambda m, i, o: stages.__setitem__("upsample", o.detach().clone()))]
    with torch.no_grad():
        logits, loss = v2(inp, enc, ce, mc, labels=lab, label_smoothing=0.1)
    for h in hooks:
        h.remove()
    empty_e, empty_c = torch.randn(1, 5, 32, generator=g), torch.randn(1, 16, generator=g)
    with torch.no_grad():
        gen_ids = v2.generate2(enc, ce, mc, empty_e, empty_c, temperature=(2.0, 0.0), timesteps=4,
                               guidance_scale=3.0, seq_len=S, generator=torch.Generator().manual_seed(62))
    torch.save(dict(config=cfg, seed=60, init_signature=init_sig, empty_embeds=empty_e, empty_cond_embeds=empty_c,
                    state_dict={k: x.clone() for k, x in v2.state_dict().items()}, input_ids=inp, labels=lab,
                    encoder_hidden_states=enc, cond_embeds=ce, micro_conds=mc, logits=logits.detach(), loss=loss.detach(),
                    stages=stages, gen_seed=62, gen_ids=gen_ids.clone()),
               os.path.join(HERE, "micro_uvit_v2_downup.pt"))
    print("micro uvit v2 down/up: loss", float(loss), "logits std", float(logits.std()),
          "downsample", tuple(stages["downsample"].shape), "upsample", tuple(stages["upsample"].shape))


HD48 = dict(vocab_size=2048, hidden_size=768, num_hidden_layers=2, num_attention_heads=16, intermediate_size=3072,
            hidden_dropout=0.0, attention_dropout=0.0, max_position_embeddings=264, codebook_size=1024, num_vq_tokens=256,
            num_classes=1000, layer_norm_eps=1e-6, use_encoder_layernorm=True, use_mlm_layer=True, use_mlm_layernorm=True)


def make_hd48(muse):
    """(12) head_dim 48: configs/imagenet.yaml (hidden 768, 16 heads, intermediate 3072 -- the config
    training/train_maskgit_imagenet.py is written for) at its own widths with 2 of its 24 layers; seed-constructed
    (weights not stored); logits slice, loss and every gradient's norm / first elements from the unmodified reference."""
    torch.manual_seed(70)
    t = muse.MaskGitTransformer(**HD48)
    t.train()
    g = torch.Generator().manual_seed(71)
    batch = masked_batch(g, 2, 256, 1024, 1000, t.config.mask_token_id)
    logits, loss = t(batch["input_ids"], labels=batch["labels"], label_smoothing=0.1)
    loss.backward()
    gr = grads_of(t)
    torch.save(dict(config=HD48, seed=70, batch=batch, label_smoothing=0.1, loss=loss.detach(),
                    logits_slice=logits.detach()[:, ::8, ::16].clone(), logits_mean=logits.mean().detach(),
                    logits_std=logits.std().detach(),
                    param_norms={k: v.norm().clone() for k, v in t.state_dict().items()},
                    grad_norms={k: v.norm() for k, v in gr.items()},
                    grad_heads={k: v.flatten()[:8].clone() for k, v in gr.items()}),
               os.path.join(HERE, "hd48_transformer.pt"))
    print("head_dim 48 transformer: loss", float(loss))


MICRO_CONV = dict(vocab_size=72, hidden_size=64, embedding_size=32, num_hidden_layers=2, num_attention_heads=1,
                  intermediate_size=128, hidden_dropout=0.0, attention_dropout=0.0, max_position_embeddings=16,
                  codebook_size=64, num_vq_tokens=64, add_cross_attention=True, encoder_hidden_size=32, norm_type="rmsnorm",
                  use_normformer=False, layer_norm_eps=1e-6, use_codebook_size_for_output=True, use_conv_in_out=True,
                  patch_size=2)


def make_conv_in_out(muse):
    """use_conv_in_out=True (ConvEmbed / ConvMlmLayer, muse/modeling_transformer.py:988-1080), the wiring of
    configs/imagenet_text2image_movq_conv.yaml and cc12m_movq.yaml at micro widths: 8x8 tokens outside, 4x4 inside.  Those
    two yaml files leave ``embedding_size`` unset, with which the reference raises a TypeError in nn.Embedding(vocab, None)
    (recorded below); the flag only constructs with an explicit embedding_size."""
    try:
        muse.MaskGitTransformer(**{k: v for k, v in MICRO_CONV.items() if k != "embedding_size"})
        unset = "constructs"
    except TypeError as e:
        unset = "TypeError: " + str(e)[:60]
    torch.manual_seed(80)
    m = muse.MaskGitTransformer(**MICRO_CONV)
    m.train()
    with torch.no_grad():  # non-trivial norm weights (they are ones at init)
        for n, p in m.named_parameters():
            if p.dim() == 1:
                p.copy_(torch.rand_like(p) + 0.5)
    g = torch.Generator().manual_seed(81)
    ids = torch.randint(0, 64, (2, 64), generator=g)
    mask = torch.rand(2, 64, generator=g) < 0.5
    input_ids = torch.where(mask, m.config.mask_token_id, ids)
    labels = torch.where(mask, ids, -100)
    enc = torch.randn(2, 5, 32, generator=g)
    logits, loss = m(input_ids, encoder_hidden_states=enc, labels=labels, label_smoothing=0.1)
    loss.backward()
    torch.manual_seed(80)
    init = {k: float(v.double().norm()) for k, v in muse.MaskGitTransformer(**MICRO_CONV).state_dict().items()}
    torch.save(dict(config=MICRO_CONV, seed=80, init_norms=init, embedding_size_unset=unset,
                    state_dict={k: v.clone() for k, v in m.state_dict().items()}, input_ids=input_ids, labels=labels,
                    encoder_hidden_states=enc, label_smoothing=0.1, logits=logits.detach(), loss=loss.detach(),
                    grads=grads_of(m)), os.path.join(HERE, "micro_conv_transformer.pt"))
    print("micro conv in/out transformer: loss", float(loss), "| embedding_size unset ->", unset)


def make_pipeline(muse):
    """The reference's PipelineMuse end to end (pipeline_muse.py:66-252) on the micro U-ViT + micro taming VQGAN fixtures'
    weights: precomputed text states / pooled embeddings (the text encoder is out of scope; a stub only supplies ``.dtype``),
    explicit negative embeddings, classifier-free guidance, 4 steps -> PIL images.  Stores the display bytes and the token
    ids the same generator seed produces."""
    import numpy as np
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2
    from muse.sampling import cosine_schedule

    gu = torch.load(os.path.join(HERE, "micro_uvit_v2.pt"), weights_only=False)
    gv = torch.load(os.path.join(HERE, "micro_taming_vqgan.pt"), weights_only=False)
    tr = MaskGiTUViT_v2(**gu["config"])
    tr.load_state_dict(gu["state_dict"])
    vae = muse.VQGANModel(**gv["config"])
    vae.load_state_dict(gv["state_dict"])
    tr.eval(), vae.eval()

    class _Enc:
        dtype = torch.float32

    pipe = muse.PipelineMuse(vae=vae, transformer=tr, text_encoder=_Enc())
    g = torch.Generator().manual_seed(90)
    B = 2
    inputs = dict(prompt_embeds=torch.randn(B, 5, 32, generator=g), pooled_embeds=torch.randn(B, 16, generator=g),
                  negative_prompt_embeds=torch.randn(B, 5, 32, generator=g), negative_pooled_embeds=torch.randn(B, 16, generator=g))
    call = dict(timesteps=4, guidance_scale=3.0, temperature=(2, 0), transformer_seq_len=16, orig_size=(256, 256),
                crop_coords=(0, 0), aesthetic_score=6.0)
    images = pipe(text=["a", "b"], negative_text=None, generator=torch.Generator().manual_seed(91), use_tqdm=False,
                  **inputs, **call)
    micro = torch.tensor([[256, 256, 0, 0, 6.0]])
    with torch.no_grad():
        tokens = tr.generate2(encoder_hidden_states=inputs["prompt_embeds"], cond_embeds=inputs["pooled_embeds"],
                              negative_embeds=inputs["negative_prompt_embeds"],
                              negative_cond_embeds=inputs["negative_pooled_embeds"], empty_embeds=None, empty_cond_embeds=None,
                              micro_conds=micro, timesteps=4,
                              guidance_scale=3.0, temperature=(2, 0), generator=torch.Generator().manual_seed(91),
                              noise_schedule=cosine_schedule, seq_len=16, use_tqdm=False)
        decoded = vae.decode_code(tokens)
    torch.save(dict(inputs=inputs, call=call, seed=91, tokens=tokens, decoded=decoded,
                    images=torch.from_numpy(np.stack([np.asarray(im) for im in images]))),
               os.path.join(HERE, "micro_pipeline.pt"))
    print("micro pipeline:", len(images), "images", images[0].size, "tokens", tokens.tolist()[0][:8])


def _yaml_numbers(d):
    """PyYAML reads "1e-6" as a string where OmegaConf (what the training scripts use) reads a float"""
    out = {}
    for k, v in d.items():
        if isinstance(v, str):
            try:
                v = float(v)
            except ValueError:
                pass
        out[k] = v
    return out


def make_config_audit(muse):
    """Every configs/*.yaml of the reference: the model class training/train_muse.py:358 would pick for it
    (``architecture`` "transformer" -> MaskGitTransformer, anything else -> MaskGiTUViT = MaskGiTUViT_v2) constructed on the
    meta device with its ``model.transformer`` section, recording either the exception class or the parameter names / shapes
    (sha1 of the ordered list) and the parameter count -- what a drop-in constructor has to reproduce."""
    import hashlib
    import json

    import yaml
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    out = {}
    cdir = os.path.join(REF, "configs")
    for f in sorted(os.listdir(cdir)):
        if not f.endswith(".yaml"):
            continue
        y = yaml.safe_load(open(os.path.join(cdir, f)))
        if not isinstance(y, dict) or "model" not in y:  # e.g. a prompt list
            continue
        model = y.get("model", {})
        tr = _yaml_numbers(dict(model.get("transformer", {})))
        arch = model.get("architecture", "transformer")
        entry = dict(architecture=arch, transformer=tr, vq_model=dict(model.get("vq_model", {})).get("type"))
        for cls_name, cls in (("MaskGitTransformer", muse.MaskGitTransformer), ("MaskGiTUViT_v2", MaskGiTUViT_v2)):
            try:
                with torch.device("meta"):
                    m = cls(**tr)
                shapes = [(n, list(p.shape)) for n, p in m.named_parameters()]
                res = dict(ok=True, n_params=sum(p.numel() for p in m.parameters()), n_tensors=len(shapes),
                           sha1=hashlib.sha1(json.dumps(shapes).encode()).hexdigest())
            except Exception as e:  # noqa: BLE001
                res = dict(ok=False, error=type(e).__name__)
            entry[cls_name] = res
        entry["script_class"] = "MaskGitTransformer" if arch == "transformer" else "MaskGiTUViT_v2"
        out[f] = entry
    with open(os.path.join(HERE, "configs.json"), "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
    for f, e in out.items():
        print(f"{f:48s} {e['script_class']:20s} v1 {e['MaskGitTransformer'].get('n_params', e['MaskGitTransformer'].get('error'))}"
              f"  v2 {e['MaskGiTUViT_v2'].get('n_params', e['MaskGiTUViT_v2'].get('error'))}")


def make_uvit_intermediate(muse):
    """MaskGiTUViT_v2.generate2(return_intermediate=True) on the micro_uvit_v2.pt weights and inputs, same generator seed as
    that fixture's ``gen_ids``: the per-step RAW multinomial samples the reference collects before it re-inserts the known
    tokens (modeling_transformer_v2.py:446-449)."""
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    g = torch.load(os.path.join(HERE, "micro_uvit_v2.pt"), weights_only=False)
    v2 = MaskGiTUViT_v2(**g["config"])
    v2.load_state_dict(g["state_dict"])
    v2.eval()
    with torch.no_grad():
        ids, inter = v2.generate2(g["encoder_hidden_states"], g["cond_embeds"], g["micro_conds"][:1], g["empty_embeds"],
                                  g["empty_cond_embeds"], temperature=(2.0, 0.0), timesteps=4, guidance_scale=3.0, seq_len=16,
                                  generator=torch.Generator().manual_seed(g["gen_seed"]), return_intermediate=True)
    assert torch.equal(ids, g["gen_ids"])
    torch.save(dict(intermediate=[t.clone() for t in inter], final=ids.clone()),
               os.path.join(HERE, "micro_uvit_v2_intermediate.pt"))
    print("micro uvit v2 intermediates:", len(inter), "steps; differ from the final-path ids at",
          int(sum((a != b).sum() for a, b in zip(inter[1:], [ids] * 3))), "positions")


def make_uvit_grads(muse):
    """Gradient signatures of the UNMODIFIED MaskGiTUViT_v2 on the micro_uvit_v2.pt / micro_uvit_v2_downup.pt weights and
    batches (label smoothing 0.1; for the first also the loss_weight form): per-parameter norm and the first 8 elements, which
    pin the oracle's autograd -- and through it the hand-written backward -- to the reference's own gradients."""
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    out = {}
    for name in ("micro_uvit_v2", "micro_uvit_v2_downup"):
        g = torch.load(os.path.join(HERE, name + ".pt"), weights_only=False)
        forms = {"plain": dict(label_smoothing=0.1)}
        if "loss_weight" in g:
            forms["loss_weight"] = dict(loss_weight=g["loss_weight"])
        for form, kw in forms.items():
            v2 = MaskGiTUViT_v2(**g["config"])
            v2.load_state_dict(g["state_dict"])
            v2.train()
            _, loss = v2(g["input_ids"], g["encoder_hidden_states"], g["cond_embeds"], g["micro_conds"], labels=g["labels"], **kw)
            loss.backward()
            gr = grads_of(v2)
            out[f"{name}/{form}"] = dict(loss=loss.detach().clone(), norms={k: v.norm().clone() for k, v in gr.items()},
                                         heads={k: v.flatten()[:8].clone() for k, v in gr.items()})
            print(name, form, "loss", float(loss), "tensors", len(gr))
    torch.save(out, os.path.join(HERE, "micro_uvit_v2_grads.pt"))


def make_pipeline_text(muse):
    """The reference's PipelineMuse with the text encoder run INSIDE the pipeline (pipeline_muse.py:113-197): a tiny random CLIP
    text encoder with projection + tokenizer (tests/train_script_harness.make_tiny_clip, seeded), the micro U-ViT and taming
    VQGAN fixtures' weights.  Two calls: default ``negative_text=""`` (negative prompt encoded, layer -2) and
    ``negative_text=None`` (guidance against the encoded empty prompt).  Stores images, the token ids handed to the
    detokeniser and a signature of the CLIP weights (the test rebuilds the same encoder from the same seed)."""
    import tempfile

    import numpy as np
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2
    from transformers import CLIPTextModelWithProjection, CLIPTokenizer

    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from tests.train_script_harness import make_tiny_clip

    gu = torch.load(os.path.join(HERE, "micro_uvit_v2.pt"), weights_only=False)
    gv = torch.load(os.path.join(HERE, "micro_taming_vqgan.pt"), weights_only=False)
    tr = MaskGiTUViT_v2(**gu["config"])
    tr.load_state_dict(gu["state_dict"])
    vae = muse.VQGANModel(**gv["config"])
    vae.load_state_dict(gv["state_dict"])
    tr.eval(), vae.eval()
    with tempfile.TemporaryDirectory() as d:
        make_tiny_clip(d, projection_dim=gu["config"]["cond_embed_dim"], weight_std=0.3)
        clip = CLIPTextModelWithProjection.from_pretrained(d).eval()
        tok = CLIPTokenizer.from_pretrained(d)
    seen, fed = [], []
    decode, gen2 = vae.decode_code, tr.generate2
    vae.decode_code = lambda ids: (seen.append(ids.clone()), decode(ids))[1]

    def spy(**kw):  # what the pipeline hands to generate2: the text side of the pipeline, tensor by tensor
        fed.append({k: v.clone() for k, v in kw.items() if torch.is_tensor(v)})
        return gen2(**kw)

    tr.generate2 = spy
    pipe = muse.PipelineMuse(vae=vae, transformer=tr, text_encoder=clip, tokenizer=tok)
    call = dict(timesteps=4, guidance_scale=3.0, temperature=(2, 0), transformer_seq_len=16, orig_size=(256, 256))
    text = ["a cat", "dog on a log"]
    out = {}
    for name, kw in (("negative_default", {}), ("negative_none", dict(negative_text=None)), ("clip_skip", dict(clip_skip=2))):
        images = pipe(text=text, generator=torch.Generator().manual_seed(92), use_tqdm=False, **call, **kw)
        out[name] = dict(images=torch.from_numpy(np.stack([np.asarray(im) for im in images])), tokens=seen[-1], fed=fed[-1])
    sig = float(sum(v.double().abs().sum() for v in clip.state_dict().values()))
    torch.save(dict(text=text, call=call, seed=92, clip_signature=sig, runs=out), os.path.join(HERE, "micro_pipeline_text.pt"))
    print("micro pipeline (text inside):", {k: v["tokens"][0, :6].tolist() for k, v in out.items()})


def make_inpainting_text(muse):
    """The reference's PipelineMuseInpainting (pipeline_muse.py:372-512) with MaskGiTUViT_v2, the taming VQGAN and the tiny
    seeded CLIP of make_pipeline_text: PIL image -> Resize / CenterCrop / ToTensor -> tokens, masked positions overwritten,
    text + explicit negative text, generate2 from the start tokens, decode.  Stores the image bytes, the mask, what the
    pipeline handed to generate2, the generated token ids and the output images."""
    import tempfile

    import numpy as np
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2
    from PIL import Image
    from transformers import CLIPTextModelWithProjection, CLIPTokenizer

    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from tests.train_script_harness import make_tiny_clip

    gu = torch.load(os.path.join(HERE, "micro_uvit_v2.pt"), weights_only=False)
    gv = torch.load(os.path.join(HERE, "micro_taming_vqgan.pt"), weights_only=False)
    tr = MaskGiTUViT_v2(**gu["config"])
    tr.load_state_dict(gu["state_dict"])
    vae = muse.VQGANModel(**gv["config"])
    vae.load_state_dict(gv["state_dict"])
    tr.eval(), vae.eval()
    with tempfile.TemporaryDirectory() as d:
        make_tiny_clip(d, projection_dim=gu["config"]["cond_embed_dim"], weight_std=0.3)
        clip = CLIPTextModelWithProjection.from_pretrained(d).eval()
        tok = CLIPTokenizer.from_pretrained(d)
    seen, fed = [], []
    decode, gen2 = vae.decode_code, tr.generate2
    vae.decode_code = lambda ids: (seen.append(ids.clone()), decode(ids))[1]

    def spy(**kw):
        fed.append({k: v.clone() for k, v in kw.items() if torch.is_tensor(v)})
        return gen2(**kw)

    tr.generate2 = spy
    pipe = muse.PipelineMuseInpainting(vae=vae, transformer=tr, text_encoder=clip, tokenizer=tok)
    pixels = (np.random.RandomState(3).rand(10, 12, 3) * 255).astype(np.uint8)  # resized (shorter side 8) and centre-cropped
    mask = torch.zeros(16, dtype=torch.bool)
    mask[5:13] = True
    out = {}
    for name, kw in (("negative_text", dict(negative_text="dog")), ("no_negative", {})):
        images = pipe(Image.fromarray(pixels), mask, text="a cat", timesteps=3, guidance_scale=2.0, temperature=1.0,
                      num_images_per_prompt=1, image_size=8, generator=torch.Generator().manual_seed(93), **kw)
        out[name] = dict(images=torch.from_numpy(np.stack([np.asarray(im) for im in images])), tokens=seen[-1], fed=fed[-1])
    torch.save(dict(pixels=torch.from_numpy(pixels), mask=mask, seed=93, runs=out), os.path.join(HERE, "micro_inpainting_text.pt"))
    print("micro inpainting (text):", {k: v["tokens"][0].tolist() for k, v in out.items()})


def make_uvit_schedules(muse):
    """MaskGiTUViT_v2.generate2 variants on the micro_uvit_v2.pt weights: guidance_schedule "linear" / "cosine", a scalar
    temperature (annealed to 0.01), explicit negative embeddings, start tokens, guidance off -- the final ids of each."""
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    g = torch.load(os.path.join(HERE, "micro_uvit_v2.pt"), weights_only=False)
    v2 = MaskGiTUViT_v2(**g["config"])
    v2.load_state_dict(g["state_dict"])
    v2.eval()
    gen = torch.Generator().manual_seed(94)
    neg_e, neg_c = torch.randn(3, 5, 32, generator=gen), torch.randn(3, 16, generator=gen)
    start = torch.full((3, 16), 71, dtype=torch.long)
    start[:, :6] = torch.randint(0, 64, (3, 6), generator=gen)
    base = dict(encoder_hidden_states=g["encoder_hidden_states"], cond_embeds=g["cond_embeds"], micro_conds=g["micro_conds"],
                empty_embeds=g["empty_embeds"], empty_cond_embeds=g["empty_cond_embeds"], timesteps=5, seq_len=16)
    variants = {
        "linear": dict(guidance_scale=4.0, guidance_schedule="linear", temperature=(2.0, 0.0)),
        "cosine": dict(guidance_scale=4.0, guidance_schedule="cosine", temperature=(2.0, 0.0)),
        "scalar_temperature": dict(guidance_scale=2.0, temperature=1.5),
        "negative": dict(guidance_scale=3.0, temperature=(1.0, 0.5), negative_embeds=neg_e, negative_cond_embeds=neg_c),
        "start_tokens": dict(guidance_scale=3.0, temperature=(2.0, 0.0), input_ids=start.clone()),
    }
    out = {}
    with torch.no_grad():
        for name, kw in variants.items():
            out[name] = v2.generate2(**base, **kw, generator=torch.Generator().manual_seed(95)).clone()
    torch.save(dict(negative_embeds=neg_e, negative_cond_embeds=neg_c, start=start, ids=out, seed=95),
               os.path.join(HERE, "micro_uvit_v2_schedules.pt"))
    print("micro uvit v2 generate2 variants:", {k: v[0, :5].tolist() for k, v in out.items()})


def make_sampling(muse):
    """muse/sampling.py function by function on seeded inputs (tests/test_sampling_helpers_cpu.py): the public names, every
    mask schedule of get_mask_chedule (or the exception it raises), mask_by_random_topk, top_k, log and the Gumbel helpers."""
    import importlib

    ref = importlib.import_module("muse.sampling")
    names = sorted(n for n in dir(ref) if not n.startswith("_") and callable(getattr(ref, n)) and n not in ("partial",))
    t = torch.linspace(0, 1, 21)
    schedules = {}
    for method in ("cosine", "linear", "sigmoid", "pow2", "pow3", "pow0.5", "pow", "log", "nonsense"):
        try:
            schedules[method] = ref.get_mask_chedule(method)(t)
        except Exception as e:  # noqa: BLE001
            schedules[method] = type(e).__name__
    g = torch.Generator().manual_seed(0)
    probs = torch.rand(3, 16, generator=g)
    mask_len = torch.tensor([[3], [5], [1]])
    x = torch.randn(2, 5, 16, generator=g)
    t9 = torch.rand(9, generator=g)
    out = dict(
        mask_by_random_topk={temp: ref.mask_by_random_topk(mask_len, probs, temperature=temp,
                                                           generator=torch.Generator().manual_seed(1))
                             for temp in (0.0, 0.7, 4.0)},
        top_k_07=ref.top_k(x, 0.7), top_k=ref.top_k(x), log=ref.log(probs),
        gumbel_noise=ref.gumbel_noise(probs, generator=torch.Generator().manual_seed(2)),
        gumbel_sample=ref.gumbel_sample(x, temperature=0.5, generator=torch.Generator().manual_seed(3)),
        cosine_schedule=ref.cosine_schedule(t9), linear_schedule=ref.linear_schedule(t9),
        sigmoid_schedule=ref.sigmoid_schedule(t9), pow=ref.pow(t9, "pow2.5"))
    torch.save(dict(public_names=names, schedule_t=t, schedules=schedules, probs=probs, mask_len=mask_len, x=x, t=t9,
                    outputs=out), os.path.join(HERE, "ref_sampling.pt"))
    print("sampling:", len(names), "public names,", {k: v for k, v in schedules.items() if isinstance(v, str)})


def make_lr_schedulers(muse):
    """muse/lr_schedulers.py: 12 steps of every schedule name through get_scheduler (3 warm-up of 10 training steps) and of
    the named constructors with non-default arguments, plus the SchedulerType values (tests/test_train_script_cpu.py)."""
    import importlib
    import json

    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from tests.test_train_script_cpu import LR_CASES, _lr_sequence

    ref = importlib.import_module("muse.lr_schedulers")
    names = [e.value for e in ref.SchedulerType]
    by_name = {n: _lr_sequence(lambda o: ref.get_scheduler(n, optimizer=o, num_warmup_steps=3, num_training_steps=10))
               for n in names}
    cases = [[fn, kw, _lr_sequence(lambda o: getattr(ref, fn)(o, **kw))] for fn, kw in LR_CASES]
    with open(os.path.join(HERE, "ref_lr_schedulers.json"), "w") as f:
        json.dump(dict(scheduler_types=names, get_scheduler=by_name, constructors=cases), f, indent=1)
    print("lr schedulers:", names)


def make_training_utils(muse):
    """muse/training_utils.py: the logging diagnostics train_muse.py computes from the logits, on a seeded batch whose
    masking rate spans every bucket (tests/test_train_muse_script_cpu.py)."""
    import importlib

    ref = importlib.import_module("muse.training_utils")
    g = torch.Generator().manual_seed(0)
    B, S, V = 12, 40, 16
    logits = torch.randn(B, S, V, generator=g)
    ids = torch.randint(0, V, (B, S), generator=g)
    mask = torch.rand(B, S, generator=g) < torch.linspace(0.02, 1.0, B)[:, None]
    mask[:, 0] = True
    inp, lab = torch.where(mask, V, ids), torch.where(mask, ids, -100)
    df = ref.token_probability_distributions_per_percent_masked_bucket(logits, inp, V)
    torch.save(dict(mask_id=V, label_smoothing=0.1, logits=logits, input_ids=inp, labels=lab,
                    buckets=ref.input_ids_to_masked_buckets(inp, V),
                    pixel_entropy=ref.pixel_entropy_per_percent_masked_bucket(logits.clone(), inp.clone(), V),
                    image_entropy=ref.image_entropy_per_percent_masked_bucket(logits.clone(), inp.clone(), V),
                    cross_entropy=ref.cross_entropy_per_percent_masked_bucket(logits.clone(), lab.clone(), inp.clone(), V, V, 0.1),
                    token_probs={"columns": list(df.columns), "dtypes": [str(d) for d in df.dtypes],
                                 "values": {c: df[c].to_numpy() for c in df.columns}}),
               os.path.join(HERE, "ref_training_utils.pt"))
    print("training utils: token-probability rows", len(df))


def make_interchange(muse):
    """Checkpoints written by the reference's save_pretrained for the four model classes of
    tests/test_checkpoint_interchange_cpu.py: its config.json verbatim, the state-dict keys / shapes / dtypes in the order
    torch.save wrote them, a SHA-256 of every tensor's bytes (the weights themselves are the seeded initialisation plus a
    seeded perturbation, which the test redraws and checks against the digests) and the reference's forward output on the
    test's seeded inputs."""
    import json
    import tempfile

    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from tests.test_checkpoint_interchange_cpu import KINDS, _digest, _inputs

    classes = {"MaskGitTransformer": muse.MaskGitTransformer, "MaskGiTUViT_v2": MaskGiTUViT_v2,
               "MaskGitVQGAN": muse.MaskGitVQGAN, "VQGANModel": muse.VQGANModel}
    out = {}
    for kind, cfg in KINDS:
        torch.manual_seed(1234)
        r = classes[kind](**cfg)
        with torch.no_grad():
            for p in r.parameters():
                p.add_((0.1 if p.dim() == 1 else 0.02) * torch.randn_like(p))
        r.eval()
        inputs = _inputs(kind)
        with tempfile.TemporaryDirectory() as d:
            r.save_pretrained(d)
            config_json = open(os.path.join(d, "config.json")).read()
            saved = torch.load(os.path.join(d, "pytorch_model.bin"))
        with torch.no_grad():
            if kind == "MaskGitTransformer":
                y = r(inputs["input_ids"])
            elif kind == "MaskGiTUViT_v2":
                y = r(inputs["input_ids"], inputs["enc"], inputs["cond"], inputs["micro"])
            else:
                y = r.decode_code(r.get_code(inputs["image"]))
        out[kind] = dict(config=cfg, config_json=json.loads(config_json),
                         keys=[(k, list(v.shape), str(v.dtype), _digest(v)) for k, v in saved.items()],
                         output=y.clone())
    torch.save(out, os.path.join(HERE, "ref_interchange.pt"))
    print("interchange:", {k: len(v["keys"]) for k, v in out.items()})


def make_surface(muse):
    """The public surface of the reference classes (tests/test_checkpoint_interchange_cpu.py): public class attributes beyond
    torch.nn.Module's, public instance attributes, config keys in order and the module tree (names, order)."""
    import json

    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    base = set(dir(torch.nn.Module))
    v1 = dict(vocab_size=72, hidden_size=64, num_hidden_layers=1, num_attention_heads=1, intermediate_size=128,
              add_cross_attention=True, encoder_hidden_size=32, project_encoder_hidden_states=True)
    v2 = dict(hidden_size=128, num_attention_heads=2, in_channels=64, block_out_channels=(64,), block_num_heads=1,
              num_res_blocks=1, num_hidden_layers=1, intermediate_size=128, vocab_size=72, codebook_size=64,
              encoder_hidden_size=32, cond_embed_dim=16, micro_cond_encode_dim=8, micro_cond_embed_dim=40)
    vq = dict(resolution=32, hidden_channels=32, channel_mult=(1, 2), num_res_blocks=1, z_channels=16, num_embeddings=64,
              quantized_embed_dim=16)
    table = {}
    for name, cls, kw in (("MaskGitTransformer", muse.MaskGitTransformer, v1), ("MaskGiTUViT_v2", MaskGiTUViT_v2, v2),
                          ("MaskGitVQGAN", muse.MaskGitVQGAN, vq), ("VQGANModel", muse.VQGANModel, vq),
                          ("EMAModel", muse.EMAModel, None), ("PipelineMuse", muse.PipelineMuse, None),
                          ("PipelineMuseInpainting", muse.PipelineMuseInpainting, None)):
        row = {"class_attributes": sorted({a for a in dir(cls) if not a.startswith("_")} - base), "kwargs": kw}
        if kw is not None:
            with torch.device("meta"):
                m = cls(**kw)
            row["instance_attributes"] = sorted(k for k in vars(m) if not k.startswith("_"))
            row["config_keys"] = list(m.config.keys())
            row["module_tree"] = [n for n, _ in m.named_modules()]
        table[name] = row
    with open(os.path.join(HERE, "ref_surface.json"), "w") as f:
        json.dump(table, f, indent=1)
    print("surface:", {k: len(v["class_attributes"]) for k, v in table.items()})


def main():
    muse = import_reference()
    torch.set_num_threads(4)
    out = {}
    only = [a.split("=", 1)[1].split(",") for a in sys.argv[1:] if a.startswith("--only=")]
    if only:  # regenerate a subset: --only=f16,signatures
        if "f16" in only[0]:
            make_f16_256(muse)
        if "signatures" in only[0]:
            make_signatures(muse)
        if "uvit_downup" in only[0]:
            make_uvit_downup(muse)
        if "hd48" in only[0]:
            make_hd48(muse)
        if "conv_in_out" in only[0]:
            make_conv_in_out(muse)
        if "pipeline" in only[0]:
            make_pipeline(muse)
        if "configs" in only[0]:
            make_config_audit(muse)
        if "pipeline_text" in only[0]:
            make_pipeline_text(muse)
        if "inpainting_text" in only[0]:
            make_inpainting_text(muse)
        if "uvit_intermediate" in only[0]:
            make_uvit_intermediate(muse)
        if "uvit_grads" in only[0]:
            make_uvit_grads(muse)
        if "uvit_schedules" in only[0]:
            make_uvit_schedules(muse)
        if "sampling" in only[0]:
            make_sampling(muse)
        if "lr_schedulers" in only[0]:
            make_lr_schedulers(muse)
        if "training_utils" in only[0]:
            make_training_utils(muse)
        if "interchange" in only[0]:
            make_interchange(muse)
        if "surface" in only[0]:
            make_surface(muse)
        return

    # ---- (1) micro class-conditional transformer: weights + inputs + logits/loss/all grads
    torch.manual_seed(0)
    m = muse.MaskGitTransformer(**MICRO)
    m.train()
    g = torch.Generator().manual_seed(1)
    batch = masked_batch(g, 3, 16, 64, 7, m.config.mask_token_id)
    logits, loss = m(batch["input_ids"], labels=batch["labels"], label_smoothing=0.1)
    loss.backward()
    torch.save(dict(config=MICRO, state_dict={k: v.clone() for k, v in m.state_dict().items()}, batch=batch,
                    label_smoothing=0.1, logits=logits.detach(), loss=loss.detach(), grads=grads_of(m)),
               os.path.join(HERE, "micro_transformer.pt"))
    print("micro transformer: loss", float(loss))

    # ---- (1b) generate2 trace on the micro model (final ids; the generator stream is torch's own)
    m.eval()
    for steps in (4, 7):
        cls = torch.tensor([1, 5, 0, 3])
        gen = torch.Generator().manual_seed(7)
        ids = m.generate2(class_ids=cls.clone(), timesteps=steps, temperature=1.0, generator=gen)
        out[f"micro_generate2_steps{steps}"] = ids.clone()
    torch.save(dict(class_ids=torch.tensor([1, 5, 0, 3]), seed=7, temperature=1.0,
                    ids={k: v for k, v in out.items() if k.startswith("micro_generate2")}),
               os.path.join(HERE, "micro_generate2.pt"))

    # ---- (2) micro text-conditional variant: cross-attention + rmsnorm + no normformer
    torch.manual_seed(2)
    mt = muse.MaskGitTransformer(**MICRO_T2I)
    mt.train()
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(0, 64, (2, 16), generator=g)
    enc = torch.randn(2, 5, 32, generator=g)
    mask = torch.rand(2, 16, generator=g) < 0.5
    inp = torch.where(mask, mt.config.mask_token_id, ids)
    lab = torch.where(mask, ids, -100)
    logits, loss = mt(inp, encoder_hidden_states=enc, labels=lab)
    loss.backward()
    torch.save(dict(config=MICRO_T2I, state_dict={k: v.clone() for k, v in mt.state_dict().items()},
                    input_ids=inp, labels=lab, encoder_hidden_states=enc, logits=logits.detach(), loss=loss.detach(),
                    grads=grads_of(mt)), os.path.join(HERE, "micro_t2i_transformer.pt"))
    print("micro t2i transformer: loss", float(loss))
    # generate2 with classifier-free guidance (zeros as the unconditional states, then explicit negative embeds) and a
    # partially given start sequence
    mt.eval()
    neg = torch.randn(2, 5, 32, generator=g)
    start = torch.full((2, 16), mt.config.mask_token_id, dtype=torch.long)
    start[:, :3] = torch.tensor([[4, 9, 1], [60, 2, 33]])
    with torch.no_grad():
        cfg_ids = mt.generate2(encoder_hidden_states=enc, timesteps=4, guidance_scale=3.0, generator=torch.Generator().manual_seed(5))
        neg_ids = mt.generate2(input_ids=start.clone(), encoder_hidden_states=enc, negative_embeds=neg, timesteps=3,
                               guidance_scale=1.5, temperature=0.7, generator=torch.Generator().manual_seed(6))
    mt.train()
    torch.save(dict(encoder_hidden_states=enc, negative_embeds=neg, start=start, cfg_ids=cfg_ids, neg_ids=neg_ids),
               os.path.join(HERE, "micro_t2i_generate2.pt"))

    # ---- (2b) text-conditional with encoder_proj + encoder_proj_layer_norm (:1154-1157,1239-1241), layernorm + normformer
    torch.manual_seed(12)
    mp = muse.MaskGitTransformer(**MICRO_T2I_PROJ)
    mp.train()
    g = torch.Generator().manual_seed(13)
    ids = torch.randint(0, 64, (3, 16), generator=g)
    enc = torch.randn(3, 7, 32, generator=g)
    mask = torch.rand(3, 16, generator=g) < 0.6
    inp = torch.where(mask, mp.config.mask_token_id, ids)
    lab = torch.where(mask, ids, -100)
    logits, loss = mp(inp, encoder_hidden_states=enc, labels=lab)
    loss.backward()
    torch.save(dict(config=MICRO_T2I_PROJ, seed=12, state_dict={k: v.clone() for k, v in mp.state_dict().items()},
                    input_ids=inp, labels=lab, encoder_hidden_states=enc, logits=logits.detach(), loss=loss.detach(),
                    grads=grads_of(mp)), os.path.join(HERE, "micro_t2i_proj_transformer.pt"))
    print("micro t2i (projected encoder states) transformer: loss", float(loss))

    # ---- (3) BASELINE config 1 (tiny, seed-constructed: no weights stored)
    torch.manual_seed(0)
    t = muse.MaskGitTransformer(**TINY)
    t.train()
    g = torch.Generator().manual_seed(1)
    batch = masked_batch(g, 2, 256, 1024, 1000, t.config.mask_token_id)
    logits, loss = t(batch["input_ids"], labels=batch["labels"])
    loss.backward()
    gr = grads_of(t)
    torch.save(dict(config=TINY, seed=0, batch=batch, loss=loss.detach(),
                    logits_slice=logits.detach()[:, ::16, ::25].clone(), logits_mean=logits.mean().detach(),
                    logits_std=logits.std().detach(),
                    param_norms={k: v.norm().clone() for k, v in t.state_dict().items()},
                    grad_norms={k: v.norm() for k, v in gr.items()},
                    grad_heads={k: v.flatten()[:8].clone() for k, v in gr.items()}),
               os.path.join(HERE, "tiny_transformer.pt"))
    print("tiny transformer (config 1): loss", float(loss))

    # ---- (4) vector quantiser: distances/ids on a margin-screened batch (small codebook)
    torch.manual_seed(4)
    vq = muse.modeling_maskgit_vqgan.VectorQuantizer(128, 64, 0.25)
    z = torch.randn(2, 64, 8, 8)
    with torch.no_grad():
        vq.embedding.weight.copy_(torch.randn(128, 64) * z.std())
        zq, ids, _ = vq(z)
        d = vq.compute_distances(z.permute(0, 2, 3, 1).contiguous())
        top2 = d.topk(2, dim=1, largest=False).values
        margin = (top2[:, 1] - top2[:, 0])
        code = vq.get_code(z)
        entry = vq.get_codebook_entry(ids)
    assert torch.equal(code, ids)
    print("vq: min top-2 margin", float(margin.min()), "relative", float((margin / top2[:, 0].abs()).min()))
    torch.save(dict(z=z, codebook=vq.embedding.weight.detach().clone(), ids=ids, z_q=zq, dmin=top2[:, 0].clone(),
                    margin=margin, entry=entry.clone()), os.path.join(HERE, "vq_quantizer.pt"))

    # ---- (4b) soft codes (get_soft_code, :327-340): deterministic and stochastic (multinomial through torch's RNG)
    with torch.no_grad():
        soft, code = vq.get_soft_code(z, temp=0.5, stochastic=False)
        torch.manual_seed(9)
        soft_s, code_s = vq.get_soft_code(z, temp=2.0, stochastic=True)
    assert torch.equal(code, ids)
    torch.save(dict(z=z, codebook=vq.embedding.weight.detach().clone(), temp=0.5, soft=soft.clone(), code=code.clone(),
                    temp_s=2.0, seed_s=9, soft_s=soft_s.clone(), code_s=code_s.clone()),
               os.path.join(HERE, "vq_soft_code.pt"))

    # ---- (5) micro MaskGitVQGAN: encode / decode_code round trip
    torch.manual_seed(5)
    v = muse.MaskGitVQGAN(**MICRO_VQ)
    v.eval()
    img = torch.rand(2, 3, 32, 32, generator=torch.Generator().manual_seed(6))
    with torch.no_grad():
        zenc = v.encoder(img)
        v.quantize.embedding.weight.copy_(torch.randn(64, 16, generator=torch.Generator().manual_seed(8)) * zenc.std())
        zq, ids = v.encode(img)
        rec = v.decode_code(ids)
        d = v.quantize.compute_distances(zenc.permute(0, 2, 3, 1).contiguous())
        top2 = d.topk(2, dim=1, largest=False).values
    print("micro vqgan: min top-2 margin", float((top2[:, 1] - top2[:, 0]).min()))
    torch.save(dict(config=MICRO_VQ, state_dict={k: x.clone() for k, x in v.state_dict().items()}, image=img,
                    z=zenc, ids=ids, z_q=zq, recon=rec, margin=(top2[:, 1] - top2[:, 0])),
               os.path.join(HERE, "micro_vqgan.pt"))

    # ---- (6) MaskGiTUViT_v2 (modeling_transformer_v2.py): micro config; the zero-initialised tensors (adaLN mappers, GRN
    # gamma/beta, mlm conv1) are re-drawn so that every branch contributes to the fixture
    from muse.modeling_transformer_v2 import MaskGiTUViT_v2

    torch.manual_seed(30)
    v2 = MaskGiTUViT_v2(**MICRO_V2)
    init_sig = {k: (float(x.double().sum()), float(x.double().norm())) for k, x in v2.state_dict().items()}
    g = torch.Generator().manual_seed(31)
    with torch.no_grad():
        for k, x in v2.state_dict().items():
            if "adaLN_modulation.mapper" in k or k.endswith("gamma") or k.endswith("beta") or k == "mlm_layer.conv1.weight":
                x.copy_(torch.randn(x.shape, generator=g) * 0.05)
            elif k.endswith("norm.weight"):
                x.copy_(1.0 + 0.1 * torch.randn(x.shape, generator=g))
    v2.train()
    ids = torch.randint(0, 64, (3, 16), generator=g)
    mask = torch.rand(3, 16, generator=g) < 0.6
    inp = torch.where(mask, 71, ids)
    lab = torch.where(mask, ids, -100)
    enc = torch.randn(3, 5, 32, generator=g)
    ce = torch.randn(3, 16, generator=g)
    mc = torch.tensor([[256.0, 256.0, 0.0, 0.0, 6.0], [512.0, 384.0, 10.0, 20.0, 5.5], [128.0, 256.0, 3.0, 0.0, 7.25]])
    logits, loss = v2(inp, enc, ce, mc, labels=lab, label_smoothing=0.1)
    lw = torch.rand(3, 16, generator=g)
    _, loss_w = v2(inp, enc, ce, mc, labels=lab, loss_weight=lw)
    v2.eval()
    empty_e, empty_c = torch.randn(1, 5, 32, generator=g), torch.randn(1, 16, generator=g)
    with torch.no_grad():
        gen_ids = v2.generate2(enc, ce, mc[:1], empty_e, empty_c, temperature=(2.0, 0.0), timesteps=4,
                               guidance_scale=3.0, seq_len=16, generator=torch.Generator().manual_seed(32))
    torch.save(dict(config=MICRO_V2, seed=30, init_signature=init_sig, empty_embeds=empty_e, empty_cond_embeds=empty_c,
                    state_dict={k: x.clone() for k, x in v2.state_dict().items()}, input_ids=inp, labels=lab,
                    encoder_hidden_states=enc, cond_embeds=ce, micro_conds=mc, logits=logits.detach(), loss=loss.detach(),
                    loss_weight=lw, loss_weighted=loss_w.detach(), gen_seed=32, gen_ids=gen_ids.clone()),
               os.path.join(HERE, "micro_uvit_v2.pt"))
    print("micro uvit v2: loss", float(loss), "weighted", float(loss_w), "logits std", float(logits.std()))

    # ---- (7) taming VQGANModel (modeling_taming_vqgan.py), micro config with attention at the last level and in the mid block
    from muse.modeling_taming_vqgan import VQGANModel

    TAMING = dict(resolution=32, num_channels=3, hidden_channels=32, channel_mult=(1, 2), num_res_blocks=2,
                  attn_resolutions=(16,), z_channels=16, num_embeddings=64, quantized_embed_dim=16)
    torch.manual_seed(40)
    tv = VQGANModel(**TAMING)
    tv.eval()
    init_sig = {k: (float(x.double().sum()), float(x.double().norm())) for k, x in tv.state_dict().items()}
    img = torch.rand(2, 3, 32, 32, generator=torch.Generator().manual_seed(41))
    with torch.no_grad():
        z = tv.quant_conv(tv.encoder(img))
        tv.quantize.embedding.weight.copy_(torch.randn(64, 16, generator=torch.Generator().manual_seed(42)) * z.std())
        zq, ids = tv.encode(img)
        rec = tv.decode_code(ids)
        d = tv.quantize.compute_distances(z.permute(0, 2, 3, 1).contiguous())
        top2 = d.topk(2, dim=1, largest=False).values
    print("micro taming vqgan: min top-2 margin", float((top2[:, 1] - top2[:, 0]).min()), "attn blocks",
          sum(1 for k in tv.state_dict() if k.endswith("proj_out.weight")))
    torch.save(dict(config=TAMING, seed=40, init_signature=init_sig,
                    state_dict={k: x.clone() for k, x in tv.state_dict().items()}, image=img, z=z, ids=ids, z_q=zq,
                    recon=rec, margin=(top2[:, 1] - top2[:, 0])), os.path.join(HERE, "micro_taming_vqgan.pt"))

    # ---- (8) EMAModel (modeling_ema.py): shadow parameters after a scripted sequence of updates, both decay schedules
    ema_out = {}
    for warm in (False, True):
        gq = torch.Generator().manual_seed(50)
        ps = [torch.nn.Parameter(torch.randn(5, 7, generator=gq)), torch.nn.Parameter(torch.randn(11, generator=gq)),
              torch.nn.Parameter(torch.randn(3, 2, generator=gq), requires_grad=False)]
        ema = muse.EMAModel(ps, decay=0.999, update_after_step=2, update_every=2, use_ema_warmup=warm, inv_gamma=2.0, power=0.75)
        decays = []
        for _ in range(40):
            with torch.no_grad():
                for q in ps:
                    q.add_(torch.randn(q.shape, generator=gq) * 0.1)
            ema.step(ps)
            decays.append(ema.cur_decay_value)
        ema_out[warm] = dict(shadow=[s.clone() for s in ema.shadow_params], decays=decays, step=ema.optimization_step)
    torch.save(dict(seed=50, runs=ema_out), os.path.join(HERE, "ema_model.pt"))

    make_f16_256(muse)
    make_signatures(muse)
    make_uvit_downup(muse)
    make_hd48(muse)
    make_conv_in_out(muse)
    make_pipeline(muse)
    make_config_audit(muse)
    make_uvit_intermediate(muse)
    make_uvit_grads(muse)
    make_uvit_schedules(muse)
    make_pipeline_text(muse)
    make_inpainting_text(muse)
    make_sampling(muse)
    make_lr_schedulers(muse)
    make_training_utils(muse)
    make_interchange(muse)
    make_surface(muse)

    for f in sorted(os.listdir(HERE)):
        if f.endswith(".pt"):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
