"""GPU tests of beam-search decoding (csrc/decode.cu, Engine.decode, AutoRegressiveBeamSearch).

Tolerances, and why:
  * decode attention (bf16 q / k / v, fp32 softmax and accumulation, bf16 output) against fp64 on the same
    bf16-rounded inputs: |err| <= 2^-8 * max|v| + 1e-3 per (row, head) -- one bf16 rounding of the output (2^-9
    relative) plus fp32 exp / sum error, well inside twice that.
  * beam step against `oracle.decode_oracle.select` evaluating the kernel's formula in fp32 on identical logits:
    tokens, parents and the ended flag exactly; scores within 1e-5 * (1 + |score|) (the log-sum-exp is summed in
    another order: a few fp32 ulps).
  * incremental (KV-cached) logits against `Engine.head_logits` over the full prefix: max |diff| < 0.15, the bf16
    bound of the head-forward parity test (test_gpu_parity.py::test_head_forward_backward_vs_oracle).
  * end to end: each selection of Engine.decode is replayed through the fp64 oracle from the GPU's own state (its
    histories and running scores), so the candidates differ only by that step's log-probability error, MEASURED on the
    cached step's logits over each row's 16 best tokens: bound = 2 x error.  Where every margin of an image's
    selection exceeds the bound its tokens and parents must equal the oracle's; everywhere the GPU's choices must
    score within the bound of the oracle's.  The error itself is capped (0.3 per unit of logit scale: twice the
    head-forward bound) so that a wrong cache cannot widen its own bound.  The sharpened golden state is only a valid
    exact-match case when every margin exceeds the bound, which the test asserts before comparing beams.
"""
import functools
import os

import pytest
import torch

from oracle import decode_oracle as D, virtex_oracle as O
from oracle.make_decode_golden import case_inputs, decode_image

pytestmark = pytest.mark.gpu
F64 = torch.float64


def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _bf(x):
    return x.to(torch.bfloat16).to(F64)


def build_model(spec, state, eos, beam=5, per_node=2, max_steps=30):
    from virtex_b200.beam_search import AutoRegressiveBeamSearch
    from virtex_b200.models import VirTexModel
    from virtex_b200.modules import TorchvisionVisualBackbone, TransformerDecoderTextualHead
    visual = TorchvisionVisualBackbone(spec.backbone, visual_feature_size=spec.visual_feature_size)
    textual = TransformerDecoderTextualHead(
        visual_feature_size=spec.visual_feature_size, vocab_size=spec.vocab, hidden_size=spec.hidden,
        num_layers=spec.layers, attention_heads=spec.heads, feedforward_size=spec.ffn, dropout=0.0,
        norm_first=spec.norm_first, max_caption_length=spec.max_len, padding_idx=spec.pad)
    model = VirTexModel(visual, textual, sos_index=1, eos_index=eos,
                        decoder=AutoRegressiveBeamSearch(eos, max_steps=max_steps, beam_size=beam,
                                                         per_node_beam_size=per_node))
    model.load_state_dict(O.to_reference_state_dict(state, spec), strict=True)
    return model.cuda().eval()


# ------------------------------------------------------------------------------------------------ decode attention
def _attn_ref(q, keys, vals):
    """q [U, 64], keys / vals [U, Tk, 64] (fp64) -> [U, 64]."""
    s = torch.einsum("ud,utd->ut", q, keys) / 8.0
    return torch.einsum("ut,utd->ud", torch.softmax(s, -1), vals)


@pytest.mark.parametrize("H", [512, 768, 1024, 2048])
@pytest.mark.parametrize("t", [1, 2, 17, 29])
@pytest.mark.parametrize("beam", [1, 5])
def test_decode_attention_self_cache_vs_fp64(H, t, beam):
    _need_cuda()
    from virtex_b200.ops import call, _stream
    g = torch.Generator().manual_seed(H + 7 * t + beam)
    A, B, T_cache = H // 64, 3, 29
    rows = B * beam  # 3 or 15 rows: neither a multiple of the 8 warps of a block
    cache = _bf(torch.randn(T_cache, rows, 3 * H, generator=g, dtype=F64))
    table = torch.randint(0, rows, (rows, T_cache), generator=g, dtype=torch.int32)
    cache_d = cache.to(torch.bfloat16).cuda()
    table_d = table.cuda()
    out = torch.full((rows + 2, H), 7.0, dtype=torch.bfloat16, device="cuda")  # 2 sentinel rows
    pos = t - 1
    base = cache_d.data_ptr()
    call("vtx_decode_attn", cache_d[pos].data_ptr(), 3 * H, base + 2 * H, base + 4 * H, 3 * H, rows * 3 * H,
         table_d.data_ptr(), T_cache, 1, out.data_ptr(), H, rows, A, t, T_cache, _stream())
    torch.cuda.synchronize()
    phys = torch.cat([table[:, :t - 1], torch.arange(rows, dtype=torch.int32)[:, None]], 1).long()  # [rows, t]
    kv = cache[torch.arange(t)[None, :].expand(rows, t), phys]  # [rows, t, 3H]
    q = cache[pos, :, :H].reshape(rows * A, 64)
    keys = kv[..., H:2 * H].reshape(rows, t, A, 64).permute(0, 2, 1, 3).reshape(rows * A, t, 64)
    vals = kv[..., 2 * H:].reshape(rows, t, A, 64).permute(0, 2, 1, 3).reshape(rows * A, t, 64)
    ref = _attn_ref(q, keys, vals)
    got = out[:rows].double().cpu().view(rows * A, 64)
    tol = 2 ** -8 * vals.abs().amax(dim=(1, 2)) + 1e-3
    err = (got - ref).abs().amax(-1)
    assert bool((err <= tol).all()), f"worst (row, head) ratio {(err / tol).max().item():.3f}"
    assert bool((out[rows:] == 7.0).all()), "wrote past the output"


@pytest.mark.parametrize("H,beam", [(512, 5), (1024, 1), (2048, 5)])
def test_decode_attention_cross_vs_fp64(H, beam):
    _need_cuda()
    from virtex_b200.ops import call, _stream
    g = torch.Generator().manual_seed(H + beam)
    A, B, Sk = H // 64, 3, 49
    rows = B * beam
    kv = _bf(torch.randn(B * Sk, 2 * H, generator=g, dtype=F64))
    q = _bf(torch.randn(rows, H, generator=g, dtype=F64))
    kv_d, q_d = kv.to(torch.bfloat16).cuda(), q.to(torch.bfloat16).cuda()
    out = torch.full((rows + 1, H), 7.0, dtype=torch.bfloat16, device="cuda")
    call("vtx_decode_attn", q_d.data_ptr(), H, kv_d.data_ptr(), kv_d.data_ptr() + 2 * H, Sk * 2 * H, 2 * H, 0, 0,
         beam, out.data_ptr(), H, rows, A, Sk, Sk, _stream())
    torch.cuda.synchronize()
    img = torch.arange(rows) // beam
    kvr = kv.view(B, Sk, 2 * H)[img]  # [rows, Sk, 2H]
    keys = kvr[..., :H].reshape(rows, Sk, A, 64).permute(0, 2, 1, 3).reshape(rows * A, Sk, 64)
    vals = kvr[..., H:].reshape(rows, Sk, A, 64).permute(0, 2, 1, 3).reshape(rows * A, Sk, 64)
    ref = _attn_ref(q.view(rows * A, 64), keys, vals)
    err = (out[:rows].double().cpu().view(rows * A, 64) - ref).abs().amax(-1)
    tol = 2 ** -8 * vals.abs().amax(dim=(1, 2)) + 1e-3
    assert bool((err <= tol).all()), f"worst ratio {(err / tol).max().item():.3f}"
    assert bool((out[rows:] == 7.0).all())


# ----------------------------------------------------------------------------------------------------- beam step
def _run_beam_step(logits, V, B, beam_in, per_node, beam_out, eos, last, scores_in):
    from virtex_b200.ops import call, _stream
    rows_out = B * beam_out
    tok = torch.full((rows_out + 1,), -7, dtype=torch.int64, device="cuda")
    par = torch.full((rows_out + 1,), -7, dtype=torch.int64, device="cuda")
    sc = torch.full((rows_out + 1,), -7.0, dtype=torch.float32, device="cuda")
    ended = torch.zeros(1, dtype=torch.int32, device="cuda")
    call("vtx_beam_step", logits.data_ptr(), logits.stride(0), V, B, beam_in, per_node, beam_out, eos,
         last.data_ptr() if last is not None else 0, scores_in.data_ptr() if scores_in is not None else 0,
         tok.data_ptr(), par.data_ptr(), sc.data_ptr(), ended.data_ptr(), _stream())
    torch.cuda.synchronize()
    assert tok[-1].item() == -7 and par[-1].item() == -7 and sc[-1].item() == -7.0, "wrote past the outputs"
    return tok[:-1].cpu(), par[:-1].cpu(), sc[:-1].cpu(), bool(ended.item())


@pytest.mark.parametrize("V,ldl", [(10000, 10000), (10001, 10016)])
@pytest.mark.parametrize("per_node", [1, 2, 5])
def test_beam_step_vs_torch_rule(V, ldl, per_node):
    _need_cuda()
    g = torch.Generator().manual_seed(V + per_node)
    B, beam, eos = 7, 5, 2
    rows = B * beam
    x = torch.randn(rows, ldl, generator=g) * 3.0
    last = torch.randint(3, V, (rows,), generator=g)
    last[[1, 7, 8]] = eos                       # ended beams (image 1 keeps two live ones)
    last[10:15] = eos                           # image 2: every beam ended
    x[3, last[3]] = 50.0                        # the penalised token is the row's largest logit
    x[20, 100], x[20, 37] = 40.0, 40.0          # planted tie: token 37 wins
    x[25, 11] = float("nan")                    # NaN row: every lp NaN except the penalty
    scores = -torch.rand(rows, generator=g) * 10
    scores[30:35] = scores[30]                  # image 6: equal running scores
    x[30:35] = x[30]
    xd = x.cuda()
    tok, par, sc, ended = _run_beam_step(xd, V, B, beam, per_node, beam, eos, last.cuda(), scores.cuda())
    rtok, rpar, rsc, _ = D.select(D.log_softmax_f32(x[:, :V]), last, scores, eos, beam, per_node)
    assert torch.equal(tok, rtok.reshape(-1)), (tok.view(B, beam), rtok)
    assert torch.equal(par, rpar.reshape(-1))
    rsc = rsc.reshape(-1)
    fin = torch.isfinite(rsc)
    assert torch.equal(fin, torch.isfinite(sc)) and torch.equal(torch.isnan(rsc), torch.isnan(sc))
    assert bool(((sc[fin] - rsc[fin]).abs() <= 1e-5 * (1 + rsc[fin].abs())).all())
    assert not ended
    assert tok.view(B, beam)[2].tolist() == [eos] * beam     # forced
    assert tok.view(B, beam)[5, 0].item() == 0               # the NaN row's lowest id (image 5, row 25)


def test_beam_step_first_step_and_ended_flag():
    _need_cuda()
    g = torch.Generator().manual_seed(3)
    B, beam, eos, V = 9, 5, 2, 10000
    x = torch.randn(B, V, generator=g)
    tok, par, sc, ended = _run_beam_step(x.cuda(), V, B, 1, beam, beam, eos, None, None)
    rtok, rpar, rsc, _ = D.select(D.log_softmax_f32(x), None, None, eos, beam, beam)
    assert torch.equal(tok, rtok.reshape(-1)) and torch.equal(par, rpar.reshape(-1))
    assert torch.equal(par, torch.arange(B).repeat_interleave(beam))
    assert bool(((sc - rsc.reshape(-1)).abs() <= 1e-5 * (1 + rsc.reshape(-1).abs())).all())
    assert not ended
    # every row ended -> EOS everywhere, flag set
    last = torch.full((B * beam,), eos, dtype=torch.int64)
    xs = torch.randn(B * beam, V, generator=g).cuda()
    tok, par, sc, ended = _run_beam_step(xs, V, B, beam, 2, beam, eos, last.cuda(), torch.zeros(B * beam).cuda())
    assert ended and bool((tok == eos).all())


# --------------------------------------------------------------------------------------------------------- reorder
@pytest.mark.parametrize("n", [0, 1, 2, 17, 29])
def test_beam_reorder_vs_torch_gather(n):
    """n = tokens of history before the step = positions cached (n = 0: the first step, history only)."""
    _need_cuda()
    from virtex_b200.ops import call, _stream
    g = torch.Generator().manual_seed(n)
    rows, ldh, ldt = 15, 31, 30
    in_hist = torch.randint(0, 10000, (rows, ldh), generator=g)
    in_tab = torch.randint(0, rows, (rows, ldt), generator=g, dtype=torch.int32)
    parents = torch.randint(0, rows, (rows,), generator=g)
    tokens = torch.randint(0, 10000, (rows,), generator=g)
    out_hist = torch.full((rows + 1, ldh), -7, dtype=torch.int64, device="cuda")  # + a sentinel row
    out_tab = torch.full((rows + 1, ldt), -7, dtype=torch.int32, device="cuda")
    ih, it, pd, td = in_hist.cuda(), in_tab.cuda(), parents.cuda(), tokens.cuda()
    call("vtx_beam_reorder", pd.data_ptr(), td.data_ptr(), ih.data_ptr() if n else 0, out_hist.data_ptr(), ldh, n,
         it.data_ptr() if n > 1 else 0, out_tab.data_ptr() if n else 0, ldt, max(n, 1), rows, _stream())
    torch.cuda.synchronize()
    oh, ot = out_hist.cpu(), out_tab.cpu()
    assert torch.equal(oh[:rows, :n], in_hist[parents, :n])
    assert torch.equal(oh[:rows, n], tokens)
    assert bool((oh[:rows, n + 1:] == -7).all()) and bool((oh[rows:] == -7).all()), "wrote past the history"
    if n:
        assert torch.equal(ot[:rows, :n - 1], in_tab[parents, :n - 1])
        assert torch.equal(ot[:rows, n - 1], parents.to(torch.int32))
        assert bool((ot[:rows, n:] == -7).all()) and bool((ot[rows:] == -7).all()), "wrote past the table"
    else:
        assert bool((ot == -7).all())


# ----------------------------------------------------------------------------------------------- incremental = full
@pytest.mark.parametrize("layers,hidden,heads,ffn,norm_first", [(1, 128, 2, 256, False), (2, 256, 4, 512, True),
                                                                (4, 128, 2, 256, False), (2, 128, 2, 256, False)])
def test_incremental_logits_equal_full_prefix(layers, hidden, heads, ffn, norm_first):
    """Beams re-parented at random (within their image) every step through vtx_beam_reorder, as the search does:
    the cached step over the reordered cache index must give the logits of the full head over each row's history."""
    _need_cuda()
    from virtex_b200.ops import call, _stream
    spec = O.Spec(hidden=hidden, layers=layers, heads=heads, ffn=ffn, norm_first=norm_first)
    model = build_model(spec, O.synth_state(spec, 40 + layers, bn3_gain=0.25), eos=2)
    eng = model.engine
    eng.mark_weights_dirty()
    B, beam, T = 2, 3, 12
    rows = B * beam
    image = decode_image(B, 9).cuda()
    g = torch.Generator().manual_seed(layers)
    kvs, caches, Sk = eng.decode_setup(image, rows, T)
    vf = eng.visual_features(image).repeat_interleave(beam, 0)
    tab = [torch.zeros(rows, T + 1, dtype=torch.int32, device="cuda") for _ in range(2)]
    hst = [torch.zeros(rows, T + 2, dtype=torch.int64, device="cuda") for _ in range(2)]
    hist = torch.randint(3, spec.vocab, (rows, 1), generator=g)
    hst[0][:, 0] = hist[:, 0].cuda()
    cur, worst, moved = 0, 0.0, 0
    for t in range(1, T + 1):  # positions 0 .. t-1: t-1 holds each row's newest token, the rest are cached
        newest = hist[:, t - 1].contiguous().cuda()
        inc = eng._decode_logits(newest, rows, t - 1, beam, tab[cur] if t > 1 else None, kvs, caches, Sk, T).clone()
        full = eng.head_logits(vf, hist.cuda(), torch.full((rows,), t, device="cuda"))[:, -1]
        worst = max(worst, (inc - full).abs().max().item())
        parents = (torch.arange(rows) // beam) * beam + torch.randint(0, beam, (rows,), generator=g)
        new = torch.randint(3, spec.vocab, (rows,), generator=g)
        if t == 4:
            new[0] = 0  # a padding-id token inside a history: its embedding is zeroed on both paths
        moved += int((parents != torch.arange(rows)).sum())
        parents_d, new_d = parents.cuda(), new.cuda()  # kept alive until the kernel has run
        call("vtx_beam_reorder", parents_d.data_ptr(), new_d.data_ptr(), hst[cur].data_ptr(),
             hst[1 - cur].data_ptr(), T + 2, t, tab[cur].data_ptr() if t > 1 else 0, tab[1 - cur].data_ptr(), T + 1,
             t, rows, _stream())
        torch.cuda.synchronize()
        hist = torch.cat([hist[parents], new[:, None]], 1)
        cur = 1 - cur
        assert torch.equal(hst[cur][:, :t + 1].cpu(), hist)
    assert moved > T  # the cache index really was permuted
    assert worst < 0.15, worst


# ------------------------------------------------------------------------------------------------------ end to end
def _oracle_step(P, spec, image):
    vf = O.backbone_forward(P, image.double(), spec, training=False)
    B = image.shape[0]

    def step(partial):
        if partial.dim() == 1:
            partial = partial.unsqueeze(1)
        rows, T = partial.shape
        return O.head_forward(P, vf.repeat_interleave(rows // B, 0), partial,
                              torch.full((rows,), T, dtype=torch.int64), spec)[:, -1]
    return step


def _replay(monkeypatch, model, P, spec, image, eos, dec_kw, err_cap):
    """Run Engine.decode with every selection recorded (the GPU's cached-step logits, and the state they were taken
    in), then replay each selection through the fp64 oracle from that same state: the oracle's logits of the GPU's
    own histories, the GPU's running scores.  The two candidate sets then differ only by this step's log-probability
    error `err` (measured over each row's 16 best tokens), so two candidates are ordered alike when their gap exceeds
    bound = 2 * err (+ fp32 rounding of the running sums).  Per step and image: where every margin (the image merge and
    its rows' top-k boundaries) exceeds the bound, the GPU's tokens and parents equal the oracle's; everywhere, the
    GPU's k-th choice scores, by the oracle, within the bound of the oracle's k-th best.  Returns the GPU's beams,
    scores and the per-step (smallest margin, bound, images whose selection was checked exactly)."""
    from virtex_b200 import beam_search as BS
    steps = []

    def recorded(orig):
        def select(self, logits):
            rec = {"logits": logits.double().cpu(), "length": self.length}
            if self.length:
                rec.update(hist=self.history.cpu().clone(), last=self.last_tokens.cpu().clone(),
                           scores=self.scores[self.cur].cpu().double())
            orig(self, logits)
            rec.update(tokens=self.last_tokens.cpu().clone(), parents=self.parents.cpu().clone(),
                       new_scores=self.scores[self.cur].cpu().double())
            steps.append(rec)
        return select

    monkeypatch.setattr(BS.BeamState, "first", recorded(BS.BeamState.first))
    monkeypatch.setattr(BS.BeamState, "step", recorded(BS.BeamState.step))
    beam, per_node, B = dec_kw["beam"], dec_kw["per_node"], image.shape[0]
    g_beams, g_scores = model.engine.decode(image.cuda(), 1, eos, beam, per_node, dec_kw["max_steps"],
                                            only_return_best=False)
    monkeypatch.undo()
    ostep = _oracle_step(P, spec, image)
    report = []
    for rec in steps:
        first = rec["length"] == 0
        o_logits = ostep(torch.full((B,), 1, dtype=torch.int64) if first else rec["hist"])
        lp_o, lp_g = torch.log_softmax(o_logits, -1), torch.log_softmax(rec["logits"], -1)
        top = lp_o.topk(16, dim=-1).indices
        err = (lp_g - lp_o).gather(1, top).abs().max().item()
        assert err <= err_cap, f"cached-step log-probabilities off by {err} (cap {err_cap})"
        last, scores = (None, None) if first else (rec["last"], rec["scores"])
        pn = beam if first else per_node
        o_tok, o_par, o_sc, m = D.select(lp_o, last, scores, eos, beam, pn)
        sc_abs = 0.0 if first else scores.abs().max().item()
        bound = 2 * err + 1e-5 * (1 + sc_abs)
        beam_in = 1 if first else beam
        decided = (m["image"] > bound) & (m["row"].view(B, beam_in).min(1).values > bound)
        g_tok, g_par = rec["tokens"].view(B, beam), rec["parents"].view(B, beam)
        assert torch.equal(g_tok[decided], o_tok[decided]) and torch.equal(g_par[decided], o_par[decided]), \
            (rec["length"], g_tok, o_tok)
        lp_pen = lp_o if first else D.penalise(lp_o, last, eos)
        base = torch.zeros(B * beam_in, dtype=F64) if first else scores
        g_oracle = lp_pen[g_par.reshape(-1), g_tok.reshape(-1)] + base[g_par.reshape(-1)]
        assert bool((g_oracle.view(B, beam) >= o_sc - bound).all()), (rec["length"], g_oracle, o_sc, bound)
        fin = torch.isfinite(g_oracle)
        assert bool(((rec["new_scores"][fin] - g_oracle[fin]).abs() <= bound).all())
        report.append((min(m["image"].min().item(), m["row"].min().item()), bound, int(decided.sum())))
    return g_beams.cpu(), g_scores.cpu(), report


def test_sharpened_state_every_beam_equals_oracle_and_reference(golden_dir, monkeypatch):
    _need_cuda()
    name = "decode_sharp_h128_beam5"
    spec, state, eos, dec_kw, image = case_inputs(name)
    golden = torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)
    P = {k: v.double() if v.is_floating_point() else v for k, v in state.items()}
    model = build_model(spec, state, eos, dec_kw["beam"], dec_kw["per_node"], dec_kw["max_steps"])
    g_beams, g_scores, report = _replay(monkeypatch, model, P, spec, image, eos, dec_kw, err_cap=0.3)
    bad = [(i, mg, bd) for i, (mg, bd, _) in enumerate(report) if not mg > bd]
    assert not bad, f"invalid case: selections (step, margin, bound) {bad} are within the GPU's error"
    o_beams, _, _ = D.decode(P, image.double(), spec, 1, eos, only_return_best=False, **dec_kw)
    assert 5 <= o_beams.shape[-1] < dec_kw["max_steps"]  # several steps, and it stops early
    assert sum(r[2] for r in report) == len(report) * image.shape[0]  # every selection was checked exactly
    assert torch.equal(g_beams, o_beams) and torch.equal(g_beams, golden["beams_f32"])
    pred = model({"image": image.cuda()})["predictions"].cpu()
    assert torch.equal(pred, golden["predictions_f32"])
    # the generic search over the model's own (full-prefix) decoding_step takes the same path
    vf = model.engine.visual_features(image.cuda())
    start = torch.full((image.shape[0],), 1, dtype=torch.int64, device="cuda")
    s_beams, _ = model.decoder.search(start, functools.partial(model.decoding_step, vf), only_return_best=False)
    assert torch.equal(s_beams.cpu(), g_beams)


@pytest.mark.parametrize("name", ["decode_h256_pre_l2_beam5", "decode_h128_beam1"])
def test_unsharpened_selections_replay_within_bound(name, monkeypatch):
    """Every selection of the GPU decode, replayed through the fp64 oracle from the GPU's own state, is the oracle's
    wherever the margin exceeds the GPU's error, and within that error of the oracle's choice everywhere."""
    _need_cuda()
    spec, state, eos, dec_kw, image = case_inputs(name)
    P = {k: v.double() if v.is_floating_point() else v for k, v in state.items()}
    model = build_model(spec, state, eos, dec_kw["beam"], dec_kw["per_node"], dec_kw["max_steps"])
    g_beams, _, report = _replay(monkeypatch, model, P, spec, image, eos, dec_kw, err_cap=0.3)
    assert g_beams.shape[:2] == (image.shape[0], dec_kw["beam"]) and len(report) == g_beams.shape[-1]
    exact = sum(r[2] for r in report[1:])
    print(f"{name}: {exact} of {image.shape[0] * (len(report) - 1)} selections after step 1 checked exactly; "
          f"bounds {min(r[1] for r in report):.2e} .. {max(r[1] for r in report):.2e}")
    assert exact >= 1, "no selection after the first step was decided by the math alone"


# ---------------------------------------------------------------------------------------------------- base config
def test_base_config_shape_runs():
    _need_cuda()
    from virtex_b200.config import Config
    from virtex_b200.factories import PretrainingModelFactory
    cfg = Config("_base_bicaptioning_R_50_L1_H1024.yaml", [])
    model = PretrainingModelFactory.from_config(cfg).cuda().eval()
    assert model.textual.hidden_size == 1024
    assert model.decoder.beam_size == 5 and model.decoder.max_steps == 30
    image = torch.randn(256, 3, 224, 224, device="cuda")
    pred = model({"image": image})["predictions"]
    assert pred.dtype == torch.int64 and pred.shape[0] == 256 and 1 <= pred.shape[1] <= 30
    assert int(pred.min()) >= 0 and int(pred.max()) < cfg.DATA.VOCAB_SIZE
    with pytest.raises(RuntimeError):
        model.train()({"image": image[:2]})


def test_decode_rejects_unsupported_sizes_before_device_work():
    _need_cuda()
    spec = O.Spec(hidden=128, layers=1, heads=2, ffn=256)
    model = build_model(spec, O.synth_state(spec, 3, bn3_gain=0.25), eos=2)
    eng = model.engine
    image = torch.randn(2, 3, 224, 224, device="cuda")
    for kw in (dict(beam_size=9), dict(beam_size=0), dict(per_node=17), dict(max_steps=66)):
        args = dict(beam_size=5, per_node=2, max_steps=30)
        args.update(kw)
        with pytest.raises(ValueError):
            eng.decode(image, 1, 2, **args)
    with pytest.raises(ValueError, match="visual tokens"):
        eng.decode(torch.randn(1, 3, 288, 288, device="cuda"), 1, 2)
