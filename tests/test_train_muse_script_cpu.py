"""CPU: the UNMODIFIED reference script training/train_muse.py (text-to-image: CLIP text encoder with projection, VQGAN
tokenizer, MaskGiTUViT = MaskGiTUViT_v2 with pooled + micro conditioning, classifier-free-guidance dropout through the
encoded empty prompt, name-based no-decay optimizer groups, EMA, checkpoints, validation) runs against the drop-in ``muse``
package for a few optimizer steps with the kernels replaced by their NUMERIC torch restatements (tests/cpu_math_ops.py,
precision-recipe mode) -- so the loss it logs is a real loss and has to fall.  The wiring is the one that runs end to end
upstream at this commit (quirk Q12: ``cond_embeds`` is only bound when cond_dropout_prob > 0, which needs
use_empty_embeds_for_uncond and a projection text encoder)."""
import json
import math
import os

import pytest
import torch

from tests import cpu_math_ops
from tests.train_script_harness import find_script, make_muse_config, run_script

SCRIPT = find_script("train_muse.py")
needs_script = pytest.mark.skipif(SCRIPT is None, reason="reference training script not available")


@needs_script
@pytest.mark.parametrize("use_ema", [False, True])
def test_reference_train_muse_script_runs_unchanged(monkeypatch, tmp_path, use_ema):
    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    steps = 5
    # (log_token_probability_distributions_every stays off: upstream indexes the BATCH with the bucket number there --
    # muse/training_utils.py:373-381 -- an IndexError for any batch smaller than 10, reproduced by the drop-in)
    extra = {"log_pixel_entropy_every": 2, "log_image_entropy_every": 2, "log_cross_entropy_every": 2,
             "checkpoints_total_limit": 1}
    cfg, out = make_muse_config(str(tmp_path), steps=steps, batch=4, mixed_precision="no", save_every=2,
                                extra_experiment=extra, use_ema=use_ema)
    acc = run_script(SCRIPT, cfg)
    losses = [v["step_loss"] for v, s in acc.logged if "step_loss" in v]
    assert len(losses) == steps and all(math.isfinite(x) for x in losses)
    assert abs(losses[0] - math.log(64)) < 0.6 and losses[-1] < losses[0]  # ~uniform at init, AdamW lr 1e-3 moves it
    assert any("eval_loss" in v for v, _ in acc.logged)
    assert any(k.startswith("grad_norm/") for v, _ in acc.logged for k in v)
    keys = {k for v, _ in acc.logged for k in v}
    assert any("entropy" in k for k in keys) and any("cross entropy" in k or "cross_entropy" in k for k in keys), sorted(keys)[:40]
    # checkpoints_total_limit = 1: checkpoint-2 was rotated out by checkpoint-4, the end-of-training one follows the same rule
    cks = sorted(d for d in os.listdir(out) if d.startswith("checkpoint"))
    assert len(cks) == 1 and json.load(open(os.path.join(out, cks[0], "metadata.json")))["global_step"] == steps
    assert os.path.exists(os.path.join(out, cks[0], "unwrapped_model", "pytorch_model.bin"))
    if use_ema:
        assert os.path.isdir(os.path.join(out, cks[0], "ema_model"))
    cfg_json = json.load(open(os.path.join(out, cks[0], "unwrapped_model", "config.json")))
    assert cfg_json["_class_name"] == "MaskGiTUViT_v2" and cfg_json["add_micro_cond_embeds"] is True


def test_training_utils_diagnostics_match_reference():
    """compat muse.training_utils (the logging diagnostics train_muse.py computes from the returned logits) against the
    reference's module, value for value -- including the upstream behaviour of scattering per-token cross-entropies with a
    per-image index (the reference's values are stored in tests/golden/ref_training_utils.pt by
    make_golden.py::make_training_utils)"""
    import sys

    import numpy as np

    ref = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_training_utils.pt"),
                     weights_only=False)
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "open_muse_b200", "compat"))
    try:
        for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
            del sys.modules[k]
        from muse import training_utils as mine
    finally:
        sys.path.pop(0)
    logits, inp, lab, V = ref["logits"], ref["input_ids"], ref["labels"], ref["mask_id"]
    assert torch.equal(ref["buckets"], mine.input_ids_to_masked_buckets(inp, V))
    for key, name, args in (("pixel_entropy", "pixel_entropy_per_percent_masked_bucket", (logits, inp, V)),
                            ("image_entropy", "image_entropy_per_percent_masked_bucket", (logits, inp, V)),
                            ("cross_entropy", "cross_entropy_per_percent_masked_bucket",
                             (logits, lab, inp, V, V, ref["label_smoothing"]))):
        m = getattr(mine, name)(*[a.clone() if torch.is_tensor(a) else a for a in args])
        torch.testing.assert_close(m, ref[key], rtol=1e-5, atol=1e-6)
    r = ref["token_probs"]
    m = mine.token_probability_distributions_per_percent_masked_bucket(logits, inp, V)
    assert list(m.columns) == r["columns"] and [str(d) for d in m.dtypes] == r["dtypes"] and len(m) > 0
    for c in r["columns"]:
        assert np.array_equal(m[c].to_numpy(), r["values"][c]), c
    for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
        del sys.modules[k]


@needs_script
def test_reference_train_muse_script_generates_and_inpaints_during_training(monkeypatch, tmp_path):
    """``experiment.generate_every`` of the unmodified train_muse.py: ``generate_images`` (16 validation prompts through the
    text encoder, classifier-free guidance against the encoded empty prompt, per-sample micro conditions, generate2 -> clamp ->
    decode_code -> PIL -> wandb) and ``generate_inpainting_images`` (reads ./inpainting_validation/<prompt>/{image, mask},
    tokenises, masks at latent resolution with its hard-coded /16, generate2 from those start tokens) both run against the
    drop-in classes in the middle of training, EMA weights swapped in and out around them."""
    from PIL import Image

    import numpy as np

    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    monkeypatch.setenv("MUSE_B200_CUDA_GRAPH", "0")
    from open_muse_b200 import MaskGiTUViT_v2

    monkeypatch.setattr(MaskGiTUViT_v2, "device", property(lambda self: torch.device("cpu")), raising=False)
    work = tmp_path / "cwd"
    rs = np.random.RandomState(0)
    for prompt in ("a red cube", "two dogs"):
        d = work / "inpainting_validation" / prompt
        os.makedirs(d)
        Image.fromarray((rs.rand(64, 64, 3) * 255).astype(np.uint8)).save(d / "image.png")
        m = np.zeros((64, 64), dtype=np.uint8)
        m[16:48, 16:48] = 255
        Image.fromarray(m).save(d / "mask.png")
    monkeypatch.chdir(work)
    cfg, out = make_muse_config(str(tmp_path), steps=2, batch=2, mixed_precision="no", save_every=1000, use_ema=True,
                                f16_tokenizer=True, extra_experiment={"generate_every": 2})
    log = tmp_path / "wandb.jsonl"
    monkeypatch.setenv("MUSE_SHIM_WANDB_LOG", str(log))
    acc = run_script(SCRIPT, cfg)
    assert [s for v, s in acc.logged if "step_loss" in v] == [1, 2]
    rows = [json.loads(l) for l in open(log)]
    gen = [r for r in rows if "generated_images" in r["keys"]]
    inp = [r for r in rows if "generated_inpainting_images" in r["keys"]]
    assert len(gen) == 1 and gen[0]["step"] == 2 and gen[0]["keys"]["generated_images"] == 16
    assert gen[0]["captions"][0] == "jay" and all(s == [64, 64] for s in gen[0]["sizes"])
    assert len(inp) == 1 and inp[0]["keys"]["generated_inpainting_images"] == 2
    assert sorted(inp[0]["captions"]) == ["a red cube", "two dogs"] and all(s == [64, 64] for s in inp[0]["sizes"])


@needs_script
def test_train_muse_script_cannot_train_the_v1_text_conditional_transformer_upstream(monkeypatch, tmp_path):
    """``architecture: transformer`` in train_muse.py = the text-conditional MaskGitTransformer (the model class of BASELINE
    config 4).  At this commit the UNMODIFIED script stops in its own code on both target modes, before or right after the
    first forward (SURVEY quirk Q12, extended): with hard targets it references ``cond_embeds`` before assignment
    (train_muse.py:747; bound only when cond_dropout_prob > 0, which in turn needs the U-ViT-only empty-prompt embeddings),
    with soft targets its ``soft_target_cross_entropy`` drops a class token that text-conditional batches do not have
    (:121-125: 255 logits rows against 256 soft-target rows).  The drop-in model is constructed, moved, wrapped and called
    with the script's keywords in both cases -- the failures are the script's, and are the same with the reference model."""
    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    cfg, _ = make_muse_config(str(tmp_path / "soft"), steps=1, batch=2, mixed_precision="no", v1_soft_targets=True)
    with pytest.raises(RuntimeError, match="must match the size of tensor"):
        run_script(SCRIPT, cfg)
    cfg, _ = make_muse_config(str(tmp_path / "hard"), steps=1, batch=2, mixed_precision="no", v1_soft_targets=True)
    with pytest.raises((NameError, UnboundLocalError), match="cond_embeds"):
        run_script(SCRIPT, cfg, extra_cli=("training.use_soft_code_target=False",))


@needs_script
def test_reference_train_muse_script_resumes_with_ema(monkeypatch, tmp_path):
    """resume of the unmodified train_muse.py with EMA: ``accelerator.load_state`` runs the script's load hook
    (``EMAModel.from_pretrained(checkpoint/ema_model, model_cls=...)`` -> ``ema.load_state_dict`` -> ``ema.to``), the model /
    optimizer / scheduler states come back, the step counter continues from the directory name."""
    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    cfg, out = make_muse_config(str(tmp_path), steps=2, batch=2, mixed_precision="no", save_every=2, use_ema=True)
    acc = run_script(SCRIPT, cfg)
    assert [s for v, s in acc.logged if "step_loss" in v] == [1, 2] and os.path.isdir(os.path.join(out, "checkpoint-2", "ema_model"))
    ema2 = torch.load(os.path.join(out, "checkpoint-2", "ema_model", "pytorch_model.bin"))
    acc = run_script(SCRIPT, cfg, extra_cli=("experiment.resume_from_checkpoint=latest", "training.max_train_steps=4"))
    assert [s for v, s in acc.logged if "step_loss" in v] == [3, 4]
    ema4 = torch.load(os.path.join(out, "checkpoint-4", "ema_model", "pytorch_model.bin"))
    k = "transformer_layers.0.ffn.wi_0.weight"
    assert set(ema2) == set(ema4) and not torch.equal(ema2[k], ema4[k])
    opt = torch.load(os.path.join(out, "checkpoint-4", "optimizer.bin"))
    assert int(next(iter(opt["state"].values()))["step"]) == 4
