"""Generate tests/golden/decode_*.pt by running the UNMODIFIED reference's beam search -- build container only.

    python -m oracle.make_decode_golden

Each case builds the reference `VirTexModel` from `virtex_oracle.synth_state` (optionally sharpened), attaches the
reference `AutoRegressiveBeamSearch` and stores `model.eval(); model({"image": ...})["predictions"]` in float64 and in
float32, together with the selection margins of `oracle.decode_oracle.decode` (float64) on the same state.
"""
import functools
import os
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import decode_oracle as D, ref_shim, virtex_oracle as O  # noqa: E402
from oracle.make_golden import GOLDEN_DIR, build_reference_model  # noqa: E402

# name: (spec kwargs, state seed, sharpen, eos, eos bias, decoder kwargs, batch size, image seed, decode_state options)
#   sharpen scales textual.embedding.words.weight (the tied output projection; the embedding LayerNorm removes the
#   scale from the input side); eos bias is added to textual.output.bias[eos].
#   "decode_sharp_h128_beam5" is a designed state (`chain`): a 10-token vocabulary (every other token is held at a
#   -1e5 output bias) whose word embeddings are orthogonal and whose position embeddings point at one "next" and one
#   "alternative" token per position, with position-dependent weights, so that every row's two best continuations and
#   every image's five best candidates lie far apart.  The search runs 10 steps of 30 and ends when every beam has
#   reached EOS (the last chain token); the five beams are five different captions, and every selection margin is
#   at least 0.2 with logits within +-12, far above bf16 error.
CASES = {
    "decode_sharp_h128_beam5": (dict(hidden=128, layers=1, heads=2, ffn=256), 45, 1.0, 100 + 37 * 9, 0.0,
                                dict(beam=5, per_node=2, max_steps=30), 2, 0, {"chain": 0.6}),
    "decode_h256_pre_l2_beam5": (dict(hidden=256, layers=2, heads=4, ffn=512, norm_first=True), 32, 1.0, 2, 0.0,
                                 dict(beam=5, per_node=2, max_steps=12), 2, 1, {}),
    "decode_h128_beam1": (dict(hidden=128, layers=1, heads=2, ffn=256), 33, 1.0, 2, 0.0,
                          dict(beam=1, per_node=2, max_steps=30), 3, 2, {}),
}
SOS = 1


def _chain(state, scale):
    """The designed state of "decode_sharp_h128_beam5" (see CASES)."""
    K = 10
    toks = [100 + 37 * i for i in range(K)]
    g = torch.Generator().manual_seed(7)
    U = torch.linalg.qr(torch.randn(128, 2 * K + 2, generator=g, dtype=torch.float64))[0].T.float()
    amp = scale * 11.3
    words = state["textual.embedding.words.weight"]
    for i, t in enumerate(toks):
        words[t] = amp * U[i]
    words[SOS] = amp * U[K]
    pos = state["textual.embedding.positions.weight"]
    for p in range(pos.shape[0]):
        nxt, alt = min(p + 1, K - 1), (p + 4) % (K - 1)
        pos[p] = amp * ((0.6 + 0.07 * p) * U[nxt] + (0.35 + 0.05 * ((p * 7) % 5)) * U[alt])
    pos[0] = amp * sum(w * U[k] for w, k in zip((0.9, 0.72, 0.55, 0.4, 0.26), (1, 3, 5, 6, 8)))
    bias = torch.full_like(state["textual.output.bias"], -1e5)
    bias[toks] = 0.0
    state["textual.output.bias"] = bias


def decode_state(spec, seed, sharpen, eos, eos_bias, chain=None):
    state = O.synth_state(spec, seed, bn3_gain=0.25)
    state["textual.embedding.words.weight"] = state["textual.embedding.words.weight"] * sharpen
    if chain is not None:
        _chain(state, chain)
    state["textual.output.bias"] = state["textual.output.bias"].clone()
    state["textual.output.bias"][eos] += eos_bias
    return state


def decode_image(batch_size, seed):
    return torch.randn(batch_size, 3, 224, 224, generator=torch.Generator().manual_seed(5000 + seed))


def case_inputs(name):
    """(spec, state, eos, decoder kwargs, image) of a case."""
    spec_kw, seed, sharpen, eos, eos_bias, dec_kw, batch_size, image_seed, gains = CASES[name]
    spec = O.Spec(**spec_kw)
    return spec, decode_state(spec, seed, sharpen, eos, eos_bias, **gains), eos, dec_kw, decode_image(batch_size,
                                                                                                    image_seed)


def run_case(name):
    from virtex.utils.beam_search import AutoRegressiveBeamSearch

    spec, state, eos, dec_kw, image = case_inputs(name)
    out = {"case": CASES[name], "sos": SOS, "eos": eos}
    for dtype, tag in ((torch.float64, "f64"), (torch.float32, "f32")):
        model = build_reference_model(spec)
        model.load_state_dict(O.to_reference_state_dict(state, spec), strict=True)
        model.sos_index, model.eos_index = SOS, eos
        model.decoder = AutoRegressiveBeamSearch(eos, max_steps=dec_kw["max_steps"], beam_size=dec_kw["beam"],
                                                 per_node_beam_size=dec_kw["per_node"])
        model = model.to(dtype).eval()
        with torch.no_grad():
            out[f"predictions_{tag}"] = model({"image": image.to(dtype)})["predictions"].clone()
            # every beam, through the reference's own search and decoding_step
            vf = model.visual(image.to(dtype))
            start = torch.full((image.shape[0],), SOS, dtype=torch.int64)
            out[f"beams_{tag}"], out[f"beam_scores_{tag}"] = model.decoder.search(
                start, functools.partial(model.decoding_step, vf), only_return_best=False)
    P = {k: v.double() if v.is_floating_point() else v for k, v in state.items()}
    beams, scores, margins = D.decode(P, image.double(), spec, SOS, eos, only_return_best=False, **dec_kw)
    pred = beams[:, 0]
    assert torch.equal(pred, out["predictions_f64"]), (name, pred, out["predictions_f64"])
    assert torch.equal(beams, out["beams_f64"]), name
    out["scores_f64"] = scores[:, 0]
    out["min_margin"] = D.min_margin(margins)
    out["margins_image"] = [m["image"] for m in margins]
    out["margins_row"] = [m["row"] for m in margins]
    path = os.path.join(GOLDEN_DIR, name + ".pt")
    torch.save(out, path)
    print(f"{name}: L = {pred.shape[-1]}, min margin {out['min_margin']:.4g}, f32 == f64: "
          f"{torch.equal(out['predictions_f32'], out['predictions_f64'])} -> {path}")


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
