"""The reference's import paths (`virtex.*`) reach the classification pretext models, and its textual-head name
"none" builds their linear head."""


def test_virtex_aliases_expose_the_classification_models():
    from virtex.config import Config
    from virtex.factories import PretrainingModelFactory, TextualHeadFactory
    from virtex.models import MultiLabelClassificationModel, TokenClassificationModel
    from virtex.models.classification import ClassificationModel
    from virtex.modules.textual_heads import LinearTextualHead
    import virtex_b200.models as vm

    assert TokenClassificationModel is vm.TokenClassificationModel and ClassificationModel is vm.ClassificationModel
    assert issubclass(MultiLabelClassificationModel, ClassificationModel)
    assert {"token_classification", "multilabel_classification"} <= set(PretrainingModelFactory.PRODUCTS)
    head = TextualHeadFactory.create("none", visual_feature_size=2048, vocab_size=81)
    assert isinstance(head, LinearTextualHead) and head.output.weight.shape == (81, 2048)
    cfg = Config(None, ["MODEL.NAME", "token_classification", "MODEL.TEXTUAL.NAME", "none"])
    assert isinstance(TextualHeadFactory.from_config(cfg), LinearTextualHead)
    assert isinstance(PretrainingModelFactory.from_config(cfg), TokenClassificationModel)
