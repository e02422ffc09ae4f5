"""``app/src/im2latex.py`` served by the B200 engine: same names, same signatures, same return values
(``load_model(model_path, vocab, device)``, ``predict(model, image_tensor, vocab, idx2char, device) ->
(formula, confidence)``), plus ``predict_batch`` for a tensor-batched ``/predict/batch`` and ``predict_nbest`` for ranked alternatives."""
import model_swin  # noqa: F401  (this directory's skeleton classes must be importable when torch.load un-pickles)
import preprocess as _preprocess
from handwritten_math_ocr_api_b200 import im2latex as _engine_api

predict = _engine_api.predict
predict_batch = _engine_api.predict_batch
predict_nbest = _engine_api.predict_nbest


def load_model(model_path: str, vocab, device):
    """/root/reference/app/src/im2latex.py:7-13.  ``device`` is what main.py computed ('cuda' on a GPU box; the
    engine has no CPU path and raises otherwise)."""
    model = _engine_api.load_model(model_path, vocab, device)
    _preprocess.bind_model(model)
    return model
