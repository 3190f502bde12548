from virtex_b200.models import ClassificationModel, MultiLabelClassificationModel, TokenClassificationModel  # noqa: F401
