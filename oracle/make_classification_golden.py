"""Generate tests/golden/clf_*.pt by running the UNMODIFIED reference's classification models -- build container only.

    python -m oracle.make_classification_golden

Each case builds the reference `TokenClassificationModel` / `MultiLabelClassificationModel` with a `LinearTextualHead`,
loads `classification_oracle.synth_state`, and records in float64 and float32: the training-mode loss, the norm and
sum of every gradient, gradient probes, BN running statistics after the step, the eval-mode logits and top-10, and the
reference's state_dict key list.  The float64 oracle must reproduce the float64 reference to round-off.
"""
import os
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import classification_oracle as C, ref_shim, virtex_oracle as O  # noqa: E402
from oracle.make_golden import GOLDEN_DIR, grad_summary  # noqa: E402

# name: (model, vocab, state seed, batch kwargs)
CASES = {
    "clf_token_v10000_b4": ("token", 10000, 61, dict(kind="token", batch_size=4, seed=1, image_size=224)),
    "clf_multilabel_v81_b3": ("multilabel", 81, 62, dict(kind="multilabel", batch_size=3, seed=2, image_size=160)),
    "clf_multilabel_v81_b3_empty": ("multilabel", 81, 63, dict(kind="multilabel", batch_size=3, seed=3,
                                                               image_size=160, empty_rows=(1,))),
}
PROBES = ("visual.cnn.conv1.weight", "visual.cnn.layer4.2.conv3.weight", "textual.output.weight",
          "textual.output.bias")


def ignore_of(kind):
    return C.TOKEN_IGNORE if kind == "token" else C.MULTILABEL_IGNORE


def build_reference_model(kind, vocab):
    from virtex.models import MultiLabelClassificationModel, TokenClassificationModel
    from virtex.modules.textual_heads import LinearTextualHead
    from virtex.modules.visual_backbones import TorchvisionVisualBackbone

    cls = TokenClassificationModel if kind == "token" else MultiLabelClassificationModel
    return cls(TorchvisionVisualBackbone("resnet50", visual_feature_size=C.FEATURES),
               LinearTextualHead(C.FEATURES, vocab), ignore_indices=list(ignore_of(kind)))


def run_case(name):
    kind, vocab, seed, batch_kw = CASES[name]
    state = C.synth_state(vocab, seed)
    batch = C.synth_label_batch(vocab=vocab, **batch_kw)
    out = {"case": CASES[name], "ignore": list(ignore_of(kind))}
    for tag, dtype in (("f64", torch.float64), ("f32", torch.float32)):
        model = build_reference_model(kind, vocab)
        out["state_dict_keys"] = list(model.state_dict().keys())
        model.load_state_dict(state, strict=True)
        model = model.to(dtype).train()
        b = dict(batch)
        b["image"] = batch["image"].to(dtype)
        res = model(b)
        res["loss"].backward()
        named = dict(model.named_parameters())
        grads = {k: named[k].grad for k in named}
        bufs = dict(model.named_buffers())
        rec = {"loss": res["loss"].detach().double(),
               "grads": grad_summary(grads),
               "grad_probe": {k: grads[k].detach().flatten()[:64].clone() for k in PROBES},
               "bn_running_mean_layer4": bufs["visual.cnn.layer4.2.bn3.running_mean"].clone(),
               "bn_running_var_stem": bufs["visual.cnn.bn1.running_var"].clone(),
               "num_batches_tracked": bufs["visual.cnn.bn1.num_batches_tracked"].clone()}
        # eval mode with the original buffers
        model.load_state_dict(O.cast_state(state, dtype), strict=True)
        model.eval()
        with torch.no_grad():
            ev = model(b)
            logits = model.textual(model.visual(b["image"]))
        rec["eval_loss"] = ev["loss"].double()
        rec["eval_top10"] = ev["predictions"].clone()
        rec["eval_logits"] = logits[:, :96].clone()
        rec["eval_top10_logits"] = logits.gather(1, ev["predictions"]).clone()
        out[tag] = rec
        print(f"{name} [{tag}] loss {rec['loss'].item():.9f} eval {rec['eval_loss'].item():.9f}", flush=True)
    # the float64 oracle against the float64 reference
    ref = out["f64"]
    o, grads, nb = C.loss_and_grads(state, batch, ignore_of(kind), dtype=torch.float64)
    g = grad_summary(grads)
    assert g["names"] == ref["grads"]["names"]
    loss_err = (o["loss"] - ref["loss"]).abs().item() if torch.isfinite(ref["loss"]) else float(
        not torch.isnan(o["loss"]))
    norm_err = ((g["norm"] - ref["grads"]["norm"]).abs() / ref["grads"]["norm"].clamp_min(1e-300)).max().item()
    ev, _, _ = C.loss_and_grads(state, batch, ignore_of(kind), dtype=torch.float64, training=False)
    assert torch.equal(ev["predictions"], ref["eval_top10"]), name
    print(f"{name}: f64 oracle vs reference: |loss err| {loss_err:.3g}, max grad-norm rel err {norm_err:.3g}, "
          f"top-10 equal", flush=True)
    path = os.path.join(GOLDEN_DIR, name + ".pt")
    torch.save(out, path)
    print(f"-> {path}")


def main():
    if not ref_shim.available():
        raise SystemExit("reference tree not found; goldens can only be regenerated in the build container")
    warnings.filterwarnings("ignore")
    ref_shim.install()
    only = sys.argv[1:]
    for name in CASES:
        if not only or name in only:
            run_case(name)


if __name__ == "__main__":
    main()
