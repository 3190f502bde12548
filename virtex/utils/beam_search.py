from virtex_b200.beam_search import AutoRegressiveBeamSearch  # noqa: F401
