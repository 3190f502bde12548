from virtex_b200.modules import LinearTextualHead, TextualHead, TransformerDecoderTextualHead  # noqa: F401
