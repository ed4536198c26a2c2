"""Checkpoints cross the boundary in BOTH directions (no GPU): a model saved by this package's ``save_pretrained`` writes the
config.json and the state-dict keys, shapes and dtypes the UNMODIFIED reference class writes for the same configuration (so
its ``from_pretrained`` consumes every key), and a model saved by the reference loads here -- ``config.json`` keys,
``pytorch_model.bin`` names and shapes are the compatibility contract (SURVEY 8b).  What the reference wrote is stored in
tests/golden/ref_interchange.pt (make_golden.py::make_interchange): its config.json, its state-dict layout with a SHA-256 of
every tensor, and its forward output.  Its weights are the seeded initialisation plus a seeded perturbation; they are redrawn
here, checked against the digests and written in the reference's key order.  The forward of the loaded weights is compared
numerically: the reference's own CPU forward against this package's host code on the kernels' torch restatements."""
import hashlib
import json
import os

import pytest
import torch

from tests import cpu_math_ops

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

V1 = dict(vocab_size=72, hidden_size=64, num_hidden_layers=2, num_attention_heads=1, intermediate_size=128, hidden_dropout=0.0,
          attention_dropout=0.0, max_position_embeddings=17, codebook_size=64, num_vq_tokens=16, num_classes=7)
V2 = dict(hidden_size=128, num_attention_heads=2, in_channels=64, block_out_channels=[64], block_num_heads=1, num_res_blocks=1,
          num_hidden_layers=2, intermediate_size=128, vocab_size=72, codebook_size=64, encoder_hidden_size=32, cond_embed_dim=16,
          micro_cond_encode_dim=8, micro_cond_embed_dim=40, norm_type="rmsnorm", force_down_up_sample=True)
VQ = dict(resolution=32, num_channels=3, hidden_channels=32, channel_mult=[1, 2], num_res_blocks=1, z_channels=16,
          num_embeddings=64, quantized_embed_dim=16)
TVQ = dict(VQ, num_res_blocks=2, attn_resolutions=[16])


def _digest(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def _inputs(kind):
    g = torch.Generator().manual_seed(7)
    if kind == "MaskGitTransformer":
        return dict(input_ids=torch.randint(0, 72, (2, 17), generator=g))
    if kind == "MaskGiTUViT_v2":
        return dict(input_ids=torch.randint(0, 72, (2, 64), generator=g), enc=torch.randn(2, 5, 32, generator=g),
                    cond=torch.randn(2, 16, generator=g), micro=torch.tensor([[256.0, 256.0, 0.0, 0.0, 6.0]] * 2))
    return dict(image=torch.rand(2, 3, 32, 32, generator=g))


KINDS = [("MaskGitTransformer", V1), ("MaskGiTUViT_v2", V2), ("MaskGitVQGAN", VQ), ("VQGANModel", TVQ)]


@pytest.fixture(scope="module")
def exchanged(tmp_path_factory):
    """this package saves one model per class and checks it against the reference's layout; the reference's checkpoint of
    each class is re-materialised from the golden file"""
    import open_muse_b200 as ours

    ref = torch.load(os.path.join(GOLDEN, "ref_interchange.pt"), weights_only=False)
    root = tmp_path_factory.mktemp("interchange")
    dirs = {}
    for kind, cfg in KINDS:
        r = ref[kind]
        assert r["config"] == cfg, kind
        base = str(root / kind)
        # (1) what this package saves is what the unmodified reference class saves and loads: config and state-dict layout
        torch.manual_seed(99)
        getattr(ours, kind)(**cfg).save_pretrained(os.path.join(base, "ours"))
        assert json.load(open(os.path.join(base, "ours", "config.json"))) == r["config_json"], kind
        saved = torch.load(os.path.join(base, "ours", "pytorch_model.bin"))
        assert [(k, list(v.shape), str(v.dtype)) for k, v in saved.items()] == [tuple(x[:3]) for x in r["keys"]], kind
        # (2) the reference's checkpoint: its weights redrawn bit for bit, its key order, its config.json
        torch.manual_seed(1234)
        m = getattr(ours, kind)(**cfg)
        with torch.no_grad():
            for p in m.parameters():  # every tensor non-trivial (norm weights are ones, adaLN mappers and GRN parameters zeros at init)
                p.add_((0.1 if p.dim() == 1 else 0.02) * torch.randn_like(p))
        sd = m.state_dict()
        assert [k for k, v in sd.items() if _digest(v) != dict((x[0], x[3]) for x in r["keys"]).get(k)] == [], kind
        dir_b = os.path.join(base, "theirs")
        os.makedirs(dir_b)
        torch.save({k: sd[k] for k, *_ in r["keys"]}, os.path.join(dir_b, "pytorch_model.bin"))
        with open(os.path.join(dir_b, "config.json"), "w") as f:
            json.dump(r["config_json"], f)
        torch.save(r["output"], os.path.join(dir_b, "reference_output.pt"))
        dirs[kind] = base
    return dirs


@pytest.mark.parametrize("kind,cfg", KINDS)
def test_checkpoints_are_interchangeable_with_the_unmodified_reference(exchanged, monkeypatch, kind, cfg):
    import open_muse_b200 as ours

    cls = getattr(ours, kind)
    dir_b = os.path.join(exchanged[kind], "theirs")
    inp = _inputs(kind)
    # (3) what the reference saved loads here: same keys / shapes / values, same config
    theirs = torch.load(os.path.join(dir_b, "pytorch_model.bin"))
    cpu_math_ops.install(monkeypatch, exact=True)
    monkeypatch.setenv("MUSE_B200_CUDA_GRAPH", "0")
    loaded = cls.from_pretrained(dir_b).eval()
    sd = loaded.state_dict()
    assert list(sd) == list(theirs) and all(torch.equal(sd[k], theirs[k]) for k in sd)
    ref_cfg = json.load(open(os.path.join(dir_b, "config.json")))
    for k, v in cfg.items():
        assert ref_cfg[k] == v and getattr(loaded.config, k) == (tuple(v) if isinstance(v, list) else v) or \
            list(getattr(loaded.config, k)) == list(v), k
    # (4) and computes what the reference computed with them
    want = torch.load(os.path.join(dir_b, "reference_output.pt"))
    with torch.no_grad():
        if kind == "MaskGitTransformer":
            got = loaded(inp["input_ids"])
        elif kind == "MaskGiTUViT_v2":
            got = loaded(inp["input_ids"], inp["enc"], inp["cond"], inp["micro"])
        else:
            got = loaded.decode_code(loaded.get_code(inp["image"]))
    assert got.shape == want.shape
    assert float((got.float() - want).norm() / want.norm()) < (5e-5 if "VQ" not in kind else 1e-3)


def test_public_surface_of_every_class_covers_the_reference():
    """every public class attribute / method, every public instance attribute, the config keys in order and the module tree
    (names, order) of the reference classes exist on the drop-in classes (the reference's surface is stored in
    tests/golden/ref_surface.json by make_golden.py::make_surface)"""
    import open_muse_b200 as ours

    with open(os.path.join(GOLDEN, "ref_surface.json")) as f:
        ref = json.load(f)
    base = set(dir(torch.nn.Module))
    bad = []
    for name, r in ref.items():
        o = getattr(ours, name)
        missing = set(r["class_attributes"]) - base - {a for a in dir(o) if not a.startswith("_")}
        if missing:
            bad.append((name, "class attributes", sorted(missing)))
        if r["kwargs"] is None:
            continue
        with torch.device("meta"):
            b = o(**r["kwargs"])
        missing = set(r["instance_attributes"]) - {k for k in vars(b) if not k.startswith("_")}
        if missing:
            bad.append((name, "instance attributes", sorted(missing)))
        if r["config_keys"] != list(b.config.keys()):
            bad.append((name, "config keys", sorted(set(r["config_keys"]) ^ set(b.config.keys()))))
        if r["module_tree"] != [n for n, _ in b.named_modules()]:
            bad.append((name, "module tree", "differs"))
    assert not bad, bad
