"""GPU tests of the classification pretext models: the kernels of csrc/classify.cu against fp64 references, the GEMM
quartet at the first vocabulary narrower than one GEMM tile (V = 81), and both models against the CPU oracle
(oracle/classification_oracle.py, pinned to the reference by tests/golden/clf_*.pt).

Tolerances:
  * pooled features (bf16): |err| <= 2^-8 |ref| + 2^-16 mean|x| per element -- one round-to-nearest bf16 rounding is
    at most half an ulp of an 8-bit significand, 2^-8 relative; the fp32 sum of at most 64 bf16 values adds
    < 64 * 2^-24 of sum|x|;
  * pool backward: bit-exact against torch's fp32 tensor-by-tensor division and bf16 rounding (the kernel performs the
    same two IEEE operations; torch divides by a Python scalar through its reciprocal, which is not the same);
  * K-hot loss (fp32): |err| <= 2e-5 (1 + mean |lse|) -- fp32 log-sum-exp over <= 16384 terms and a set mean over <= 1024
    logits stay near 1e-6 relative; dlogits (bf16): max |err| <= 2^-7 max |ref| per row (one bf16 rounding plus fp32
    softmax error);
  * top-k indices and every untouched sentinel: exact;
  * V = 81 GEMMs (bf16 operands, fp32 accumulation): |err| <= 1e-5 sum |a_k b_k| per output, the fp32 rounding of K
    products in any order;
  * models (bf16 backbone, bn3_gain 0.25 as in tests/test_gpu_parity.py): train loss 1e-3 relative; output-layer
    gradients cos >= 0.999; backbone gradients against the oracle with the CUDA path's bf16 rounding placement: worst
    cos >= 0.85 and median relative error <= 0.5, the bounds of the backbone parity test; BN running statistics 2e-2;
    eval top-10 identical to the oracle's at every rank whose fp64 oracle logit is more than 0.02 from both neighbours
    (the logit error is asserted below 0.01 first, so no two such logits can swap; the bf16 backbone moves the logits
    by ~0.005 here), and identical to the top-10 of the engine's own logits everywhere.  Random logits over 10000
    classes crowd the top-10 into gaps of ~0.004, so the models' states add staggered output biases to ten classes
    (`spread_top10`) to give the check ranks to bind on;
  * trajectory: losses 3e-3, gradient norm 10 %, the output layer's update cos >= 0.99; a backbone weight's update
    cos >= 0.85, the per-step backbone-gradient floor above.
"""
import math

import pytest
import torch

from oracle import classification_oracle as C

pytestmark = pytest.mark.gpu
BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64
LOGIT_BOUND = 0.02


def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _call(name, *args):
    from virtex_b200.ops import _stream, call
    call(name, *args, _stream())
    torch.cuda.synchronize()


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def cos(a, b):
    a, b = a.detach().double().cpu().flatten(), b.detach().double().cpu().flatten()
    return (a @ b / (a.norm() * b.norm() + 1e-30)).item()


# ------------------------------------------------------------------------------------------------------------ pooling
@pytest.mark.parametrize("B", [1, 256])
@pytest.mark.parametrize("S", [1, 49, 64])
def test_avgpool_forward_and_backward(B, S):
    _need_cuda()
    C_ = 2048
    g = torch.Generator(device="cuda").manual_seed(S * 1000 + B)
    feat = (torch.randn(B * S, C_, device="cuda", generator=g) * 2).to(BF16)
    pooled = torch.full((B + 1, C_), 7.0, device="cuda", dtype=BF16)  # last row: sentinel
    _call("vtx_avgpool_fwd", feat.data_ptr(), pooled.data_ptr(), B, S, C_)
    x = feat.double().view(B, S, C_)
    ref = x.mean(1)
    bound = 2.0 ** -8 * ref.abs() + 2.0 ** -16 * x.abs().mean(1)
    err = (pooled[:B].double() - ref).abs()
    print(f"pool fwd B={B} S={S}: worst err / bound {(err / bound).max().item():.3f}")
    assert (err <= bound).all()
    assert (pooled[B] == 7.0).all()
    dpooled = torch.randn(B, C_, device="cuda", generator=g, dtype=F32)
    dfeat = torch.full((B * S + 1, C_), 7.0, device="cuda", dtype=BF16)
    _call("vtx_avgpool_bwd", dpooled.data_ptr(), dfeat.data_ptr(), B, S, C_)
    want = (dpooled / torch.full_like(dpooled, S)).to(BF16).repeat_interleave(S, dim=0)
    assert torch.equal(dfeat[:B * S], want)
    assert (dfeat[B * S] == 7.0).all()


# ------------------------------------------------------------------------------------------------------ K-hot loss
def _khot_inputs(B, V, L, seed, empty_row=None):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, V, generator=g, dtype=F64) * 3
    labels = torch.randint(-3, V + 3, (B, L), generator=g)  # includes out-of-range ids
    if L > 2:
        labels[:, 1] = labels[:, 0]  # a duplicate in every row
        labels[:, -1] = 0            # padding / ignored
    if empty_row is not None:
        labels[empty_row] = 0
    return logits, labels


@pytest.mark.parametrize("V,ldl", [(81, 88), (10000, 10000), (16384, 16400)])
@pytest.mark.parametrize("L", [1, 30, 1024])
def test_khot_xent_against_fp64(V, ldl, L):
    _need_cuda()
    B = 8
    ignore = (0, 1, 2, 3)
    logits, labels = _khot_inputs(B, V, L, seed=V + L)
    for b in range(B):  # every row keeps at least one label
        labels[b, 0] = 4 + b
    lf = torch.full((B + 1, ldl), 123.0, dtype=F32)
    lf[:B, :V] = logits.float()
    lf = lf.cuda()
    lf0 = lf.clone()
    lab = labels.cuda()
    ign = torch.tensor(ignore, device="cuda")
    loss = torch.tensor([0.5], device="cuda")  # += semantics
    dl = torch.full((B + 1, ldl), -5.0, device="cuda", dtype=BF16)
    _call("vtx_khot_xent", lf.data_ptr(), ldl, lab.data_ptr(), L, ign.data_ptr(), len(ignore), B, V, loss.data_ptr(),
          dl.data_ptr(), ldl)
    x = lf[:B, :V].double().cpu().requires_grad_(True)
    ref = C.khot_loss(x, labels, ignore)
    ref.backward()
    lse = torch.logsumexp(x.detach(), 1)
    tol = 2e-5 * (1 + lse.abs().mean().item())
    assert abs(loss.item() - 0.5 - ref.item()) <= tol, (loss.item() - 0.5, ref.item(), tol)
    d = dl[:B, :V].double().cpu()
    row_err = (d - x.grad).abs().amax(1) / x.grad.abs().amax(1)
    print(f"khot V={V} L={L}: loss err {abs(loss.item() - 0.5 - ref.item()):.2e} (tol {tol:.1e}), "
          f"worst dlogits row err / max {row_err.max().item():.2e}")
    assert (row_err <= 2.0 ** -7).all()
    assert torch.equal(lf, lf0)  # logits are read only
    assert (dl[:B, V:] == -5.0).all() and (dl[B] == -5.0).all()
    # without dlogits only the loss is produced
    loss2 = torch.zeros(1, device="cuda")
    _call("vtx_khot_xent", lf.data_ptr(), ldl, lab.data_ptr(), L, ign.data_ptr(), len(ignore), B, V, loss2.data_ptr(),
          0, ldl)
    assert abs(loss2.item() - ref.item()) <= tol


def test_khot_xent_empty_label_set_is_nan_with_a_zero_gradient_row():
    _need_cuda()
    B, V, L = 4, 81, 12
    logits, labels = _khot_inputs(B, V, L, seed=5, empty_row=2)
    for b in (0, 1, 3):
        labels[b, 0] = 10 + b
    lf = torch.zeros(B, 88, dtype=F32)
    lf[:, :V] = logits.float()
    lf, lab, ign = lf.cuda(), labels.cuda(), torch.tensor([0], device="cuda")
    loss = torch.zeros(1, device="cuda")
    dl = torch.full((B, 88), -5.0, device="cuda", dtype=BF16)
    _call("vtx_khot_xent", lf.data_ptr(), 88, lab.data_ptr(), L, ign.data_ptr(), 1, B, V, loss.data_ptr(),
          dl.data_ptr(), 88)
    assert math.isnan(loss.item())
    assert (dl[2, :V] == 0).all()
    x = lf[:, :V].double().cpu().requires_grad_(True)
    C.khot_loss(x, labels, (0,)).backward()
    keep = [0, 1, 3]
    err = (dl[keep, :V].double().cpu() - x.grad[keep]).abs().amax(1) / x.grad[keep].abs().amax(1)
    assert (err <= 2.0 ** -7).all()


# ------------------------------------------------------------------------------------------------------------ top-k
def _topk_rows(N, seed):
    g = torch.Generator().manual_seed(seed)
    rows = [torch.randn(N, generator=g),
            torch.randint(0, 4, (N,), generator=g).float(),                  # heavy ties
            torch.full((N,), float("-inf")),                                 # all -inf
            torch.where(torch.rand(N, generator=g) < 0.5, torch.randn(N, generator=g), torch.tensor(float("-inf")))]
    r = torch.randn(N, generator=g)
    r[[N // 3, 5, N - 1]] = float("nan")
    rows.append(r)
    rows.append(torch.full((N,), float("nan")))
    return torch.stack(rows)


@pytest.mark.parametrize("k", [1, 10, 16])
@pytest.mark.parametrize("N,ld", [(81, 88), (10000, 10000), (16, 20)])
def test_topk_rows_against_reference_order(k, N, ld):
    _need_cuda()
    X = _topk_rows(N, seed=N + k)
    M = X.shape[0]
    buf = torch.full((M, ld), 1e30)
    buf[:, :N] = X
    out = torch.full((M + 1, k), -7, dtype=torch.int64, device="cuda")
    _call("vtx_topk_rows", buf.cuda().data_ptr(), ld, M, N, k, out.data_ptr())
    assert torch.equal(out[:M].cpu(), C.topk(X, k))
    assert (out[M] == -7).all()


# ------------------------------------------------------------------------------------------ V = 81 GEMM quartet
@pytest.mark.parametrize("B", [4, 256])
def test_v81_output_layer_gemms(B):
    """Forward (N = 81 < one tile, fp32 output with ld 88), wgrad (K = B), dgrad (K = 81) and the bias column sums, as
    the engine issues them, against fp64."""
    _need_cuda()
    from virtex_b200.engine import Engine
    from virtex_b200.ops import gemm
    V, ldl, C_ = 81, 88, 2048
    g = torch.Generator(device="cuda").manual_seed(B)
    pooled = torch.randn(B, C_, device="cuda", generator=g).to(BF16)
    W = (torch.randn(V, C_, device="cuda", generator=g) * 0.02).to(BF16)
    bias = torch.randn(V, device="cuda", generator=g) * 0.1
    logits = torch.full((B, ldl), 9.0, device="cuda")
    gemm(pooled, W, logits, B, V, C_, ldd=ldl, bias=bias)
    dlog = torch.full((B, ldl), 3.0, device="cuda", dtype=BF16)
    dlog[:, :V] = (torch.randn(B, V, device="cuda", generator=g) * 0.01).to(BF16)
    dW = torch.zeros(V, C_, device="cuda")
    Engine._wgrad(None, dlog[:, :V], pooled, dW, V, C_, B)
    dp = torch.zeros(B, C_, device="cuda")
    gemm(dlog[:, :V], W, dp, B, C_, V, b_mn=1)
    db = torch.zeros(V, device="cuda")
    _call("vtx_colsum", dlog.data_ptr(), ldl, B, V, db.data_ptr())
    torch.cuda.synchronize()
    P, Wd, D = pooled.double(), W.double(), dlog[:, :V].double()

    def check(out, ref, mag, what):
        ratio = ((out.double() - ref).abs() / (1e-5 * mag + 1e-30)).max().item()
        print(f"V=81 {what} B={B}: worst err / tol {ratio:.3f}")
        assert ratio <= 1.0, what

    check(logits[:, :V], P @ Wd.t() + bias.double(), P.abs() @ Wd.abs().t() + bias.double().abs(), "forward")
    assert (logits[:, V:] == 9.0).all()
    check(dW, D.t() @ P, D.abs().t() @ P.abs(), "wgrad")
    check(dp, D @ Wd, D.abs() @ Wd.abs(), "dgrad")
    check(db, D.sum(0), D.abs().sum(0), "colsum")


# ------------------------------------------------------------------------------------------------- models vs oracle
CASES = {  # kind, vocab, state seed, batch kwargs
    "token": ("token", 10000, 71, dict(kind="token", batch_size=4, seed=11, image_size=224)),
    "multilabel": ("multilabel", 81, 72, dict(kind="multilabel", batch_size=3, seed=12, image_size=160)),
}


def spread_top10(state, vocab, seed):
    """Ten classes with output biases 7.0, 6.5, ..., 2.5 above the rest, clear of the largest of the other 9990 random
    logits (std ~0.3): their order is set by the biases plus the image's own logit spread, with gaps far above the
    bf16 logit error at most ranks."""
    g = torch.Generator().manual_seed(seed)
    bias = state["textual.output.bias"].clone()
    bias[torch.randperm(vocab, generator=g)[:10]] += torch.linspace(7.0, 2.5, 10)
    state["textual.output.bias"] = bias
    return state


def build(kind, vocab, state, frozen=False):
    from virtex_b200.models import MultiLabelClassificationModel, TokenClassificationModel
    from virtex_b200.modules import LinearTextualHead, TorchvisionVisualBackbone
    cls = TokenClassificationModel if kind == "token" else MultiLabelClassificationModel
    ignore = list(C.TOKEN_IGNORE if kind == "token" else C.MULTILABEL_IGNORE)
    model = cls(TorchvisionVisualBackbone("resnet50", 2048, frozen=frozen), LinearTextualHead(2048, vocab), ignore)
    model.load_state_dict(state, strict=True)
    return model.cuda(), ignore


def to_cuda(batch):
    return {k: v.cuda() for k, v in batch.items()}


def _check_grads(named, grads, grads_emul, tag):
    for n in ("textual.output.weight", "textual.output.bias"):
        c = cos(named[n].grad, grads[n])
        assert c >= 0.999, (tag, n, c)
    worst = sorted((cos(named[n].grad, grads_emul[n]), rel(named[n].grad, grads_emul[n]), n)
                   for n in grads if n.startswith("visual."))
    med = sorted(r for _, r, _ in worst)[len(worst) // 2]
    print(f"{tag}: backbone grads vs bf16-placement oracle: worst cos {worst[0][0]:.4f} ({worst[0][2]}), "
          f"median rel {med:.3f}")
    assert all(torch.isfinite(named[n].grad).all() for n in grads)
    assert worst[0][0] >= 0.85, worst[:3]
    assert med <= 0.5, med


@pytest.mark.parametrize("name", sorted(CASES))
def test_model_train_step_and_eval_vs_oracle(name):
    _need_cuda()
    kind, vocab, seed, batch_kw = CASES[name]
    state = spread_top10(C.synth_state(vocab, seed), vocab, seed)
    batch = C.synth_label_batch(vocab=vocab, **batch_kw)
    model, ignore = build(kind, vocab, state)
    model.train()
    out = model(to_cuda(batch))
    ref, grads, nb = C.loss_and_grads(state, batch, ignore)
    _, grads_emul, _ = C.loss_and_grads(state, batch, ignore, emulate_bf16=True)
    r = abs(out["loss"].item() - ref["loss"].item()) / ref["loss"].item()
    print(f"{name}: train loss {out['loss'].item():.6f} oracle {ref['loss'].item():.6f} rel {r:.2e}")
    assert r <= 1e-3
    assert out["loss_components"]["classification"].item() == out["loss"].item()
    out["loss"].backward()
    named = dict(model.named_parameters())
    _check_grads(named, grads, grads_emul, name)
    for k, b in (("visual.cnn.layer4.2.bn3.running_mean", model.visual.cnn.layer4[2].bn3.running_mean),
                 ("visual.cnn.bn1.running_var", model.visual.cnn.bn1.running_var)):
        assert rel(b, nb[k]) <= 2e-2, k
    # eval: running statistics, loss computed too, top-10 predictions
    model.load_state_dict(state, strict=True)
    model.eval()
    with torch.no_grad():
        ev = model(to_cuda(batch))
    ref_e, _, _ = C.loss_and_grads(state, batch, ignore, dtype=F64, training=False)
    assert abs(ev["loss"].item() - ref_e["loss"].item()) <= 1e-3 * ref_e["loss"].item()
    eng = model.engine
    lg = eng._clf["logits"][:, :vocab].double().cpu()
    err = (lg - ref_e["logits"]).abs().max().item()
    assert err < LOGIT_BOUND / 2, err
    pred, pref = ev["predictions"].cpu(), ref_e["predictions"]
    assert pred.shape == (batch_kw["batch_size"], 10) and pred.dtype == torch.int64
    top = ref_e["logits"].topk(11, dim=1).values
    gap = top[:, :-1] - top[:, 1:]                     # gap[:, r] = l_r - l_{r+1}
    before = torch.cat([torch.full_like(gap[:, :1], math.inf), gap[:, :-1]], 1)
    sure = (gap > LOGIT_BOUND) & (before > LOGIT_BOUND)
    print(f"{name}: eval logits max err {err:.2e}; top-10 ranks checked {int(sure.sum())}/{sure.numel()}")
    assert sure.float().mean() >= 0.5
    assert torch.equal(pred[sure], pref[sure])
    assert torch.equal(pred, C.topk(lg.float(), 10))


def test_model_with_an_empty_label_set_gives_nan_loss_and_the_oracle_gradients():
    _need_cuda()
    vocab = 81
    state = C.synth_state(vocab, 73)
    batch = C.synth_label_batch("multilabel", 3, seed=13, vocab=vocab, image_size=160, empty_rows=(1,))
    model, ignore = build("multilabel", vocab, state)
    model.train()
    out = model(to_cuda(batch))
    assert math.isnan(out["loss"].item())
    out["loss"].backward()
    _, grads, _ = C.loss_and_grads(state, batch, ignore)
    _, grads_emul, _ = C.loss_and_grads(state, batch, ignore, emulate_bf16=True)
    _check_grads(dict(model.named_parameters()), grads, grads_emul, "empty row")


@pytest.mark.parametrize("name", sorted(CASES))
def test_trainer_step_matches_model_forward(name):
    """Trainer.step on a classification batch returns [loss, 0] equal to the oracle's loss, and its gradient arena
    equals the one `loss.backward()` leaves."""
    _need_cuda()
    from virtex_b200.config import Config
    from virtex_b200.trainer import Trainer
    kind, vocab, seed, batch_kw = CASES[name]
    state = C.synth_state(vocab, seed)
    batch = C.synth_label_batch(vocab=vocab, **batch_kw)
    model, ignore = build(kind, vocab, state)
    model.train()
    cfg = Config(f"task_ablations/{kind if kind == 'token' else 'multilabel'}_classification_R_50.yaml")
    tr = Trainer(model, cfg)
    loss = tr.step({"image": batch["image"].cuda(), "labels": batch["labels"].cuda()})
    ref, grads, _ = C.loss_and_grads(state, batch, ignore)
    assert loss.shape == (2,) and loss[1].item() == 0.0
    assert abs(loss[0].item() - ref["loss"].item()) <= 1e-3 * ref["loss"].item()
    g = model.engine.arena.g("textual.output.weight")
    assert cos(g, grads["textual.output.weight"]) >= 0.999


def test_trainer_trajectory_vs_oracle():
    _need_cuda()
    from virtex_b200.config import Config
    from virtex_b200.trainer import Trainer
    from oracle import virtex_oracle as O
    vocab = 81
    state = C.synth_state(vocab, 74)
    model, ignore = build("multilabel", vocab, state)
    model.train()
    over = ["OPTIM.WARMUP_STEPS", 3, "OPTIM.NUM_ITERATIONS", 20, "OPTIM.BATCH_SIZE", 4, "OPTIM.CNN_LR", 0.005]
    tr = Trainer(model, Config("task_ablations/multilabel_classification_R_50.yaml", over))
    ora = C.OracleTrainer(state, ignore, O.OptimCfg(warmup_steps=3, num_iterations=20, cnn_lr=0.005, no_decay="none"))
    for it in range(6):
        batch = C.synth_label_batch("multilabel", 4, seed=40 + it, vocab=vocab, image_size=160)
        loss = tr.step({"image": batch["image"].cuda(), "labels": batch["labels"].cuda()})[0].item()
        ref = ora.step(batch)
        assert abs(loss - ref["loss"].item()) < 3e-3 * ref["loss"].item(), (it, loss, ref["loss"].item())
        assert abs(tr.grad_norm.item() - ref["grad_norm"].item()) < 0.1 * ref["grad_norm"].item(), it
    for k, bound in (("textual.output.weight", 0.99), ("visual.cnn.layer4.2.conv3.weight", 0.85)):
        d_ours = dict(model.named_parameters())[k].detach().cpu() - state[k]
        d_ref = ora.state[k] - state[k]
        print(f"trajectory: {k} update cos {cos(d_ours, d_ref):.4f}")
        assert cos(d_ours, d_ref) > bound, (k, cos(d_ours, d_ref))


def test_frozen_backbone_updates_only_the_output_layer():
    _need_cuda()
    from virtex_b200.config import Config
    from virtex_b200.factories import PretrainingModelFactory
    from virtex_b200.trainer import Trainer
    cfg = Config("task_ablations/multilabel_classification_R_50.yaml",
                 ["MODEL.VISUAL.FROZEN", True, "OPTIM.WARMUP_STEPS", 1])
    model = PretrainingModelFactory.from_config(cfg)
    model.load_state_dict(C.synth_state(81, 75), strict=True)
    model = model.cuda().train()
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    tr = Trainer(model, cfg)
    for it in range(3):
        batch = C.synth_label_batch("multilabel", 4, seed=50 + it, vocab=81, image_size=160)
        loss = tr.step({"image": batch["image"].cuda(), "labels": batch["labels"].cuda()})
        assert math.isfinite(loss[0].item())
    for n, p in model.named_parameters():
        changed = not torch.equal(p.detach(), before[n])
        assert changed == n.startswith("textual.output."), n


def test_linear_head_module_forward():
    """`LinearTextualHead.forward` (module-level, like the reference's): (B, C, h, w) fp32 -> (B, V) logits."""
    _need_cuda()
    from virtex_b200.modules import LinearTextualHead
    head = LinearTextualHead(2048, 81).cuda()
    vf = torch.randn(3, 2048, 7, 7, device="cuda").relu()
    out = head(vf, None, None)
    assert out.shape == (3, 81) and out.dtype == F32
    ref = vf.double().mean((2, 3)) @ head.output.weight.double().t() + head.output.bias.double()
    assert (out.double() - ref).abs().max().item() < 2e-3


def test_full_size_token_classification_batch_256_vs_fp32_oracle():
    """The token classification task at its training size (batch 256, V = 10000, 224 x 224): training-mode loss against
    the fp32 oracle within 1e-3 relative."""
    _need_cuda()
    torch.set_num_threads(max(1, min(32, (torch.get_num_threads() or 1))))
    vocab = 10000
    state = C.synth_state(vocab, 76)
    batch = C.synth_label_batch("token", 256, seed=14, vocab=vocab)
    model, ignore = build("token", vocab, state)
    model.train()
    with torch.no_grad():
        out = model(to_cuda(batch))
        ref_loss = C.forward(state, batch, ignore, training=True)["loss"]
    r = abs(out["loss"].item() - ref_loss.item()) / ref_loss.item()
    print(f"B=256 token classification: loss {out['loss'].item():.6f} oracle {ref_loss.item():.6f} rel {r:.2e}")
    assert r < 1e-3
