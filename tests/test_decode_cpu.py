"""CPU tests of beam-search captioning: the decode oracle against the reference's own outputs (tests/golden/decode_*.pt,
written by oracle/make_decode_golden.py from the live reference), each selection rule on hand-built logits, the
factory / config wiring, and the argument checks of the decode entry points (which must fail before any device work).
"""
import os
import warnings

import pytest
import torch

from oracle import decode_oracle as D
from oracle.make_decode_golden import CASES, case_inputs

V = 8
EOS = 2


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_decode_reproduces_reference_f64(golden_dir, name):
    g = torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)
    spec, state, eos, dec_kw, image = case_inputs(name)
    P = {k: v.double() if v.is_floating_point() else v for k, v in state.items()}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        beams, scores, margins = D.decode(P, image.double(), spec, g["sos"], eos, only_return_best=False, **dec_kw)
    assert beams.shape == g["beams_f64"].shape
    assert torch.equal(beams, g["beams_f64"])                  # every beam, as the reference's search returns them
    assert torch.equal(beams[:, 0], g["predictions_f64"])      # and what the reference model returns
    assert torch.allclose(scores, g["beam_scores_f64"], rtol=0, atol=1e-9)
    assert D.min_margin(margins) == pytest.approx(g["min_margin"], rel=1e-6)
    if name.startswith("decode_sharp"):
        assert 5 <= beams.shape[-1] < dec_kw["max_steps"]      # several steps, and it stops early
        assert len({tuple(b) for b in beams[0].tolist()}) == dec_kw["beam"]  # five different captions
        assert g["min_margin"] > 0.2
        assert torch.equal(g["beams_f32"], g["beams_f64"])


def _scripted(tables):
    """A step function replaying fixed logits: tables[i] is the [rows, V] logits of call i."""
    calls = []

    def step(partial):
        calls.append(partial.clone())
        return tables[len(calls) - 1].clone()
    return step, calls


def _lp(*rows):
    """Rows of logits given as {token: logit} over a floor of -20."""
    out = torch.full((len(rows), V), -20.0, dtype=torch.float64)
    for i, r in enumerate(rows):
        for t, v in r.items():
            out[i, t] = v
    return out


def test_step1_topk_and_history_without_sos():
    step, calls = _scripted([_lp({5: 3.0, 4: 2.0, 6: 1.0}),
                             _lp({6: 5.0}, {6: 5.0}), _lp({EOS: 5.0}, {EOS: 5.0})])
    pred, scores, _ = D.beam_search(torch.tensor([1]), step, EOS, max_steps=5, beam=2, per_node=1,
                                    only_return_best=False)
    assert calls[0].tolist() == [1]
    assert calls[1].tolist() == [[5], [4]]  # the start token is dropped after step 1
    assert calls[2].tolist() == [[5, 6], [4, 6]]
    assert pred.tolist() == [[[5, 6, EOS], [4, 6, EOS]]]
    assert scores.shape == (1, 2) and scores[0, 0] > scores[0, 1]


def test_repetition_penalty_is_exactly_minus_10000():
    # beam 1, per_node 1: the row's last token 5 is the best logit at step 2 but gets -10000
    step, _ = _scripted([_lp({5: 9.0}), _lp({5: 9.0, 3: 1.0})])
    pred, score, margins = D.beam_search(torch.tensor([1]), step, EOS, max_steps=2, beam=1, per_node=1)
    assert pred.tolist() == [[5, 3]]
    lp2 = torch.log_softmax(_lp({5: 9.0, 3: 1.0}), -1)[0]
    lp1 = torch.log_softmax(_lp({5: 9.0}), -1)[0]
    assert score.item() == pytest.approx((lp1[5] + lp2[3]).item(), abs=1e-12)
    # the row's second candidate is the next-best token, not the penalised one (-10000 is far below -20 - lse)
    assert margins[1]["row"].item() == pytest.approx((lp2[3] - lp2[0]).item(), abs=1e-12)


def test_ended_beam_is_forced_to_eos_with_unchanged_score():
    step, _ = _scripted([_lp({EOS: 3.0, 4: 2.9}), _lp({7: 8.0}, {7: 8.0}), _lp({EOS: 8.0}, {EOS: 8.0})])
    pred, scores, _ = D.beam_search(torch.tensor([1]), step, EOS, max_steps=4, beam=2, per_node=2,
                                    only_return_best=False)
    lp1 = torch.log_softmax(_lp({EOS: 3.0, 4: 2.9}), -1)[0]
    assert pred[0, 0].tolist() == [EOS, EOS, EOS]           # the ended beam repeats EOS at score + 0
    assert scores[0, 0].item() == pytest.approx(lp1[EOS].item(), abs=1e-12)
    assert pred[0, 1, :2].tolist() == [4, 7]


def test_per_node_limits_candidates_per_beam():
    # beam 0 has three equally good continuations (lp -log 3), beams 1 and 2 only flat rows (lp -log 8): without the
    # per_node limit all three survivors would descend from beam 0
    step, _ = _scripted([_lp({4: 2.0, 5: 1.9, 6: 1.8}), _lp({3: 5.0, 6: 5.0, 7: 5.0}, {}, {})])
    pred, _, _ = D.beam_search(torch.tensor([1]), step, EOS, max_steps=2, beam=3, per_node=2, only_return_best=False)
    assert pred[0].tolist() == [[4, 3], [4, 6], [5, 0]]


def test_ties_prefer_lower_token_and_lower_candidate():
    step, _ = _scripted([_lp({6: 1.0, 4: 1.0, 5: 1.0})])
    pred, _, _ = D.beam_search(torch.tensor([1]), step, EOS, max_steps=1, beam=2, per_node=2, only_return_best=False)
    assert pred[0, :, 0].tolist() == [4, 5]
    # image merge: two beams with equal scores and equal logits -> beam 0's candidates first
    step, _ = _scripted([_lp({4: 1.0, 5: 1.0}), _lp({6: 1.0, 7: 1.0}, {6: 1.0, 7: 1.0})])
    pred, _, _ = D.beam_search(torch.tensor([1]), step, EOS, max_steps=2, beam=2, per_node=2, only_return_best=False)
    assert pred[0].tolist() == [[4, 6], [4, 7]]


def test_nan_ranks_first_and_lowest_index_wins():
    x = torch.tensor([[1.0, float("nan"), 3.0, float("nan"), float("inf")]])
    assert D.rank(x)[0].tolist() == [1, 3, 4, 2, 0]


def test_beam1_all_eos_returns_after_step1_with_warning():
    step, calls = _scripted([_lp({EOS: 5.0}, {EOS: 5.0})])
    with pytest.warns(RuntimeWarning, match=D.EMPTY_WARNING):
        pred, scores, _ = D.beam_search(torch.tensor([1, 1]), step, EOS, max_steps=5, beam=1, per_node=2)
    assert pred.shape == (2, 1, 1) and scores.shape == (2, 1) and len(calls) == 1


def test_infinite_scores_warn_and_shapes():
    # V = 8 tokens with two finite logits, beam 4, per_node 1: two beams start at -inf and stay there
    x = torch.full((1, V), float("-inf"), dtype=torch.float64)
    x[0, 3], x[0, 4] = 1.0, 0.5
    step, _ = _scripted([x, x.repeat(4, 1)])
    with pytest.warns(RuntimeWarning, match=D.INF_WARNING):
        pred, scores, _ = D.beam_search(torch.tensor([1]), step, EOS, max_steps=2, beam=4, per_node=1,
                                        only_return_best=False)
    assert pred.shape == (1, 4, 2) and scores.shape == (1, 4)
    with pytest.warns(RuntimeWarning, match=D.INF_WARNING):
        best, best_score, _ = D.beam_search(torch.tensor([1]), _scripted([x, x.repeat(4, 1)])[0], EOS, max_steps=2,
                                            beam=4, per_node=1)
    assert best.shape == (1, 2) and best_score.shape == (1,)


def test_decoder_factory_and_alias():
    from virtex_b200.beam_search import AutoRegressiveBeamSearch
    from virtex_b200.config import Config
    from virtex_b200.factories import CaptionDecoderFactory
    import virtex.utils.beam_search as alias

    assert alias.AutoRegressiveBeamSearch is AutoRegressiveBeamSearch
    cfg = Config(None, ["MODEL.DECODER.BEAM_SIZE", 3, "MODEL.DECODER.MAX_DECODING_STEPS", 17, "DATA.EOS_INDEX", 2])
    dec = CaptionDecoderFactory.from_config(cfg)
    assert isinstance(dec, AutoRegressiveBeamSearch)
    assert (dec._eos_index, dec.max_steps, dec.beam_size, dec.per_node_beam_size) == (2, 17, 3, 2)
    cfg = Config(None, ["MODEL.DECODER.NAME", "nucleus_sampling"])
    with pytest.raises(NotImplementedError):
        CaptionDecoderFactory.from_config(cfg).search(torch.zeros(1), None)


def _rejects(name, *args):
    from virtex_b200 import lib, ops
    with pytest.raises(lib.VtxError, match=r"\(-1\)"):
        ops.call(name, *args)


FAKE = 1 << 40  # never dereferenced: every call below must be refused by its argument checks


def test_decode_entries_reject_bad_arguments_before_device_work():
    pytest.importorskip("ctypes")
    from virtex_b200 import lib
    try:
        lib.load()
    except lib.VtxError:
        pytest.skip("library not built")
    # attention: H % 128 != 0, Tk over the cache, cache over 64 keys, table narrower than the cache
    _rejects("vtx_decode_attn", FAKE, 192, FAKE, FAKE, 192, 192, 0, 0, 1, FAKE, 64, 4, 1, 1, 8, 0)
    _rejects("vtx_decode_attn", FAKE, 384, FAKE, FAKE, 384, 384, FAKE, 8, 1, FAKE, 128, 4, 2, 9, 8, 0)
    _rejects("vtx_decode_attn", FAKE, 384, FAKE, FAKE, 384, 384, 0, 0, 1, FAKE, 128, 4, 2, 65, 65, 0)
    _rejects("vtx_decode_attn", FAKE, 384, FAKE, FAKE, 384, 384, FAKE, 4, 1, FAKE, 128, 4, 2, 8, 8, 0)
    # beam step: per_node > V, per_node over 16, beams over one cluster, ldl < V, beam_out > candidates
    args = lambda ldl, V, imgs, bin_, pn, bout: (FAKE, ldl, V, imgs, bin_, pn, bout, 0, FAKE, FAKE, FAKE, FAKE, FAKE,
                                                  FAKE, 0)
    _rejects("vtx_beam_step", *args(8, 4, 2, 5, 5, 5))
    _rejects("vtx_beam_step", *args(10000, 10000, 2, 5, 17, 5))
    _rejects("vtx_beam_step", *args(10000, 10000, 2, 9, 2, 5))   # 9 beams: more blocks than one cluster holds
    _rejects("vtx_beam_step", *args(9999, 10000, 2, 5, 2, 5))
    _rejects("vtx_beam_step", *args(10000, 10000, 2, 2, 2, 5))
    # reorder: history past its row, in place
    _rejects("vtx_beam_reorder", FAKE, FAKE, FAKE, FAKE + 8, 30, 30, 0, 0, 31, 1, 10, 0)
    _rejects("vtx_beam_reorder", FAKE, FAKE, FAKE, FAKE, 31, 3, 0, 0, 31, 1, 10, 0)
