from virtex_b200.models import (CaptioningModel, ForwardCaptioningModel, BidirectionalCaptioningModel,  # noqa: F401
                                VirTexModel, MaskedLMModel, ClassificationModel, TokenClassificationModel,
                                MultiLabelClassificationModel)
