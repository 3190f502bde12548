"""Classification pretext models without a device: the oracle against the goldens written by the live reference
(oracle/make_classification_golden.py), each K-hot loss rule on hand-built logits, factories / configs, state-dict
interchange, gradient buckets and argument rejection by the new C entry points."""
import functools
import math
import os

import pytest
import torch

from oracle import classification_oracle as C

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ("clf_token_v10000_b4", "clf_multilabel_v81_b3", "clf_multilabel_v81_b3_empty")


@functools.lru_cache(maxsize=None)
def _case(name):
    """(golden, float64 oracle training output, grads, new buffers, float64 oracle eval output)."""
    g = torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)
    kind, vocab, seed, batch_kw = g["case"]
    state = C.synth_state(vocab, seed)
    batch = C.synth_label_batch(vocab=vocab, **batch_kw)
    out, grads, nb = C.loss_and_grads(state, batch, g["ignore"], dtype=torch.float64)
    ev, _, _ = C.loss_and_grads(state, batch, g["ignore"], dtype=torch.float64, training=False)
    return g, out, grads, nb, ev


def _same(a, b, rtol=1e-9, atol=1e-12):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return torch.allclose(a, b, rtol=rtol, atol=atol, equal_nan=True)


# ----------------------------------------------------------------------------------------------------------- goldens
@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name):
    """float64 oracle == float64 reference to round-off: loss, every gradient's norm and sum, probes, BN buffers,
    eval logits, and the top-10 exactly."""
    g, out, grads, nb, ev = _case(name)
    ref = g["f64"]
    assert _same(out["loss"], ref["loss"]), (out["loss"], ref["loss"])
    names = ref["grads"]["names"]
    assert sorted(grads) == names
    assert _same(torch.tensor([grads[n].norm().item() for n in names], dtype=torch.float64), ref["grads"]["norm"])
    sums = torch.tensor([grads[n].sum().item() for n in names], dtype=torch.float64)
    assert _same(sums, ref["grads"]["sum"], atol=1e-10)
    for k, v in ref["grad_probe"].items():
        assert _same(grads[k].flatten()[:64], v, atol=1e-14), k
    assert _same(nb["visual.cnn.layer4.2.bn3.running_mean"], ref["bn_running_mean_layer4"])
    assert _same(nb["visual.cnn.bn1.running_var"], ref["bn_running_var_stem"])
    assert int(nb["visual.cnn.bn1.num_batches_tracked"]) == int(ref["num_batches_tracked"])
    assert _same(ev["loss"], ref["eval_loss"])
    assert _same(ev["logits"][:, :96], ref["eval_logits"])
    assert torch.equal(ev["predictions"], ref["eval_top10"])
    assert _same(ev["logits"].gather(1, ev["predictions"]), ref["eval_top10_logits"])
    # the float32 reference agrees with the float64 one (the golden carries no float32-only artefact)
    assert torch.equal(g["f32"]["eval_top10"], ref["eval_top10"])


def test_empty_label_set_golden_is_nan_loss_with_finite_gradients():
    g, out, grads, _, _ = _case("clf_multilabel_v81_b3_empty")
    for tag in ("f64", "f32"):
        assert math.isnan(g[tag]["loss"].item())
        assert torch.isfinite(g[tag]["grads"]["norm"]).all()
    assert math.isnan(out["loss"].item())
    assert all(torch.isfinite(v).all() for v in grads.values())


# ---------------------------------------------------------------------------------------------- rules, hand-built
def reference_loop(logits, labels, ignore):
    """Inline restatement of the reference's per-image loop (virtex/models/classification.py:80-95)."""
    logp = torch.log_softmax(logits, dim=1)
    loss = logits.new_zeros(())
    for b in range(logits.shape[0]):
        keep = [int(l) for l in labels[b].unique() if int(l) not in ignore]
        loss = loss - logp[b, keep].mean()
    return loss / logits.shape[0]


def loop_counting_duplicates(logits, labels, ignore):
    """Planted mistake: no unique()."""
    logp = torch.log_softmax(logits, dim=1)
    loss = logits.new_zeros(())
    for b in range(logits.shape[0]):
        keep = [int(l) for l in labels[b] if int(l) not in ignore]
        loss = loss - logp[b, keep].mean()
    return loss / logits.shape[0]


def loop_keeping_ignored(logits, labels, ignore):
    """Planted mistake: the ignore list is not applied."""
    return reference_loop(logits, labels, ())


def agrees(fn_a, fn_b, logits, labels, ignore):
    """Comparator: loss and logit gradient of two implementations agree (NaN == NaN)."""
    outs = []
    for fn in (fn_a, fn_b):
        x = logits.clone().requires_grad_(True)
        loss = fn(x, labels, ignore)
        loss.backward()
        outs.append((loss.detach(), x.grad))
    (la, ga), (lb, gb) = outs
    return _same(la, lb, rtol=1e-12) and _same(ga, gb, rtol=1e-12, atol=1e-15)


def _logits(B, V, seed=0):
    return torch.randn(B, V, generator=torch.Generator().manual_seed(seed), dtype=torch.float64) * 3


def test_rule_duplicates_count_once():
    logits = _logits(2, 12)
    labels = torch.tensor([[5, 5, 5, 7, 0], [9, 4, 9, 0, 0]])
    assert agrees(C.khot_loss, reference_loop, logits, labels, (0,))
    assert not agrees(loop_counting_duplicates, reference_loop, logits, labels, (0,))


def test_rule_ignored_ids_and_padding_are_excluded():
    logits = _logits(2, 12, seed=1)
    labels = torch.tensor([[1, 6, 3, 2, 0, 0], [1, 8, 11, 2, 0, 0]])  # [SOS] ... [EOS] + [MASK] + 0-padding
    ignore = (0, 1, 2, 3)
    assert agrees(C.khot_loss, reference_loop, logits, labels, ignore)
    assert not agrees(loop_keeping_ignored, reference_loop, logits, labels, ignore)
    assert C.label_sets(labels, 12, ignore) == [[6], [8, 11]]


def test_rule_empty_set_gives_nan_loss_and_a_zero_gradient_row():
    logits = _logits(3, 10, seed=2)
    labels = torch.tensor([[4, 5], [0, 0], [7, 7]])
    assert agrees(C.khot_loss, reference_loop, logits, labels, (0,))
    x = logits.clone().requires_grad_(True)
    loss = C.khot_loss(x, labels, (0,))
    loss.backward()
    assert math.isnan(loss.item())
    assert torch.equal(x.grad[1], torch.zeros(10, dtype=torch.float64))
    # the other rows keep their gradient, still divided by the full batch size
    y = logits[[0, 2]].clone().requires_grad_(True)
    C.khot_loss(y, labels[[0, 2]], (0,)).backward()
    assert torch.allclose(x.grad[[0, 2]], y.grad * 2 / 3, rtol=1e-12)


def test_rule_out_of_range_ids_are_skipped():
    logits = _logits(2, 10, seed=3)
    labels = torch.tensor([[4, -1, 10, 123456, 6], [2, 2, -7, 0, 0]])
    in_range = torch.tensor([[4, 6, 0, 0, 0], [2, 2, 0, 0, 0]])
    assert agrees(C.khot_loss, lambda x, l, i: reference_loop(x, in_range, i), logits, labels, (0,))


def test_topk_order_nan_first_then_value_then_index():
    x = torch.tensor([[1.0, float("nan"), 3.0, 3.0, float("-inf"), float("nan"), 0.5]])
    assert C.topk(x, 5).tolist() == [[1, 5, 2, 3, 0]]
    ninf = torch.full((1, 12), float("-inf"))
    assert C.topk(ninf, 10).tolist() == [list(range(10))]
    r = torch.randn(4, 50, dtype=torch.float64)
    assert torch.equal(C.topk(r, 10), r.topk(10, dim=1).indices)


# ------------------------------------------------------------------------------------------- factories and configs
@pytest.mark.parametrize("cfg_name,cls_name,ignore,vocab", [
    ("task_ablations/token_classification_R_50.yaml", "TokenClassificationModel", [0, 1, 2, 3], 10000),
    ("task_ablations/multilabel_classification_R_50.yaml", "MultiLabelClassificationModel", [0], 81),
])
def test_configs_build_classification_models(cfg_name, cls_name, ignore, vocab):
    from virtex_b200.config import Config
    from virtex_b200.factories import PretrainingModelFactory, TextualHeadFactory, param_group_hparams
    from virtex_b200.modules import LinearTextualHead

    cfg = Config(cfg_name)
    model = PretrainingModelFactory.from_config(cfg)
    assert type(model).__name__ == cls_name
    assert model.ignore_indices == ignore
    assert isinstance(model.textual, LinearTextualHead)
    assert model.textual.output.weight.shape == (vocab, 2048) and model.textual.output.bias.shape == (vocab,)
    assert model.textual.hidden_size == 2048 and model.textual.textual_feature_size == 2048
    assert isinstance(TextualHeadFactory.create("none", visual_feature_size=2048, vocab_size=vocab), LinearTextualHead)
    # OPTIM.NO_DECAY "none" matches no parameter name: every parameter decays
    assert param_group_hparams(cfg, "textual.output.bias")[1] == cfg.OPTIM.WEIGHT_DECAY


def test_classification_model_rejects_other_heads_and_cpu_batches():
    from virtex_b200.models import TokenClassificationModel
    from virtex_b200.modules import LinearTextualHead, TorchvisionVisualBackbone, TransformerDecoderTextualHead

    visual = TorchvisionVisualBackbone("resnet50", 2048)
    with pytest.raises(ValueError):
        TokenClassificationModel(visual, TransformerDecoderTextualHead(2048, 100, 128, 1, 2, 256), [0])
    model = TokenClassificationModel(visual, LinearTextualHead(2048, 100), [0])
    with pytest.raises(KeyError):
        model({"image": torch.zeros(1, 3, 64, 64)})
    with pytest.raises(RuntimeError, match="no CPU path"):
        model({"image": torch.zeros(1, 3, 64, 64), "labels": torch.zeros(1, 3, dtype=torch.int64)})
    # the reference's topk(10) fails in eval mode below 10 classes: refused before any device work
    small = TokenClassificationModel(visual, LinearTextualHead(2048, 9), [0]).eval()
    with pytest.raises(ValueError, match="10 classes"):
        small({"image": torch.zeros(1, 3, 64, 64), "labels": torch.zeros(1, 3, dtype=torch.int64)})


# -------------------------------------------------------------------------------------------------------- state dict
@pytest.mark.parametrize("name,kind,vocab", [("clf_token_v10000_b4", "token", 10000),
                                             ("clf_multilabel_v81_b3", "multilabel", 81)])
def test_state_dict_keys_match_the_reference_and_load_strictly(name, kind, vocab):
    from virtex_b200.models import MultiLabelClassificationModel, TokenClassificationModel
    from virtex_b200.modules import LinearTextualHead, TorchvisionVisualBackbone

    g = torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)
    cls = TokenClassificationModel if kind == "token" else MultiLabelClassificationModel
    model = cls(TorchvisionVisualBackbone("resnet50", 2048), LinearTextualHead(2048, vocab), g["ignore"])
    assert list(model.state_dict().keys()) == g["state_dict_keys"]
    state = C.synth_state(vocab, 5)  # the reference checkpoint layout (what make_classification_golden loads)
    model.load_state_dict(state, strict=True)
    assert torch.equal(model.textual.output.weight, state["textual.output.weight"])


# ------------------------------------------------------------------------------------------------------------ buckets
def test_bucket_ranges_cover_every_classification_parameter_once():
    from virtex_b200.engine import Arena
    from virtex_b200.models import MultiLabelClassificationModel
    from virtex_b200.modules import LinearTextualHead, TorchvisionVisualBackbone
    from virtex_b200.trainer import bucket_ranges

    model = MultiLabelClassificationModel(TorchvisionVisualBackbone("resnet50", 2048), LinearTextualHead(2048, 81), [0])
    arena = Arena([("visual." + n, p) for n, p in model.visual.named_parameters()] +
                  [("textual." + n, p) for n, p in model.textual.named_parameters()], "cpu")
    r = bucket_ranges(arena.names, arena.offsets, arena.numels)
    assert r["head_b"] is None
    assert r["head"] == (arena.offsets["textual.output.weight"],
                         arena.offsets["textual.output.bias"] + arena.numels["textual.output.bias"])
    for n in arena.names:
        b, e = arena.offsets[n], arena.offsets[n] + arena.numels[n]
        owners = [k for k, v in r.items() if v is not None and v[0] <= b and e <= v[1]]
        assert len(owners) == 1, (n, owners)


# ------------------------------------------------------------------------------------------------ C argument checks
def _rc(name, *args):
    from virtex_b200 import ops
    return ops._get(name)(*args)


def test_classification_entry_points_reject_unsupported_sizes_before_touching_the_device():
    """Each call is invalid only in the one argument named; the library returns VTX_EINVAL (-1) while validating, so
    no pointer (all fake, 256) is dereferenced and no device is needed."""
    P = 256
    # K-hot loss: V > 65536 (8 KB bitmap), L > 1024, misaligned fp32 / bf16 leading dimensions
    assert _rc("vtx_khot_xent", P, 65544, P, 30, P, 4, 2, 65537, P, P, 65544, 0) == -1
    assert _rc("vtx_khot_xent", P, 10000, P, 1025, P, 4, 2, 10000, P, P, 10000, 0) == -1
    assert _rc("vtx_khot_xent", P, 82, P, 10, P, 1, 2, 81, P, P, 88, 0) == -1
    assert _rc("vtx_khot_xent", P, 88, P, 10, P, 1, 2, 81, P, P, 84, 0) == -1
    assert _rc("vtx_khot_xent", P, 80, P, 10, P, 1, 2, 81, P, P, 88, 0) == -1  # ldl < V
    # top-k: k > 16, k > N, ld < N
    assert _rc("vtx_topk_rows", P, 10000, 4, 10000, 17, P, 0) == -1
    assert _rc("vtx_topk_rows", P, 8, 4, 8, 10, P, 0) == -1
    assert _rc("vtx_topk_rows", P, 80, 4, 81, 10, P, 0) == -1
    # pooling: C % 8 != 0, S < 1
    assert _rc("vtx_avgpool_fwd", P, P, 4, 49, 2044, 0) == -1
    assert _rc("vtx_avgpool_fwd", P, P, 4, 0, 2048, 0) == -1
    assert _rc("vtx_avgpool_bwd", P, P, 4, 49, 2044, 0) == -1
    assert _rc("vtx_avgpool_bwd", P, P, 4, 0, 2048, 0) == -1
