"""CPU-only: this package's plug-in mirror against the original project's OWN hot-path files.

`NLP_workloads/Anyscale_job/predictor.py:14-106` (HuggingFaceModelPredictor) and `utils.py:6-33`
(preprocess_function) of the original workshop project were run unmodified through the shim, on the inputs below,
and their outputs stored in tests/golden/reference_predictor.npz (tests/golden/make_reference_golden.py). What these
tests establish carries to the GPU through pinned equalities:

    reference predictor + HF model  ==  direct HF generate                    (stored; the mirror reproduces both here)
    reference predictor             ==  this package's mirror, same model      (here)
    mirror + B200 model             ==  B200 generate == HF on the same GPU    (tests/test_model_gpu.py)

Flow reproduced: flan-t5-batch-inference.py:119-138 (from_checkpoint -> predict -> to_pandas -> join).
"""
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
import torch

from anyscale_workshop_nyc_2023_b200 import rayshim
from anyscale_workshop_nyc_2023_b200.predictor import HuggingFaceModelPredictor as Mirror
from anyscale_workshop_nyc_2023_b200.preprocess import make_preprocess_function
from anyscale_workshop_nyc_2023_b200.workload import checkpoint_dir


@pytest.fixture(scope="module")
def gold():
    return np.load(Path(__file__).resolve().parent / "golden" / "reference_predictor.npz")


class HFOnCpu:
    """model_cls stand-in with from_pretrained(dir, **kw): the dependency's own model on CPU (what
    `T5ForConditionalGeneration` is in the reference script, minus the hub download)."""

    @staticmethod
    def from_pretrained(path, **kw):
        from oracle.hf_anchor import load_hf_model

        assert kw.get("torch_dtype") is torch.float16 and kw.get("device_map") == "auto"  # forwarded untouched (NB:881-882)
        return load_hf_model(path, dtype=torch.float32, device="cpu")


def test_reference_script_flow_with_the_unmodified_predictor_class(gold):
    """BatchPredictor.from_checkpoint(checkpoint=..., predictor_cls=..., model_cls=..., tokenizer=T5Tokenizer,
    use_gpu=..., device_map="auto", torch_dtype=torch.float16) -> predict(ds, num_gpus_per_worker=..., batch_size=...,
    max_new_tokens=...) -> to_pandas -> join, as flan-t5-batch-inference.py:119-138: the mirror class returns what the
    unmodified reference class returned in this flow."""
    rayshim.install()
    from ray.data.preprocessors import BatchMapper
    from ray.train.batch_predictor import BatchPredictor
    from transformers import T5Tokenizer

    from anyscale_workshop_nyc_2023_b200.rayshim.train import HuggingFaceCheckpoint
    from oracle.hf_anchor import hf_generate, load_hf_model

    ckpt = checkpoint_dir("tiny", seed=1)
    use_gpu = False
    rows = {c: gold[f"flow_{c}"].tolist() for c in ("instruction", "input", "output", "text")}
    validation_dataset = rayshim.data.from_huggingface(rows).limit(10)
    fn = make_preprocess_function(str(ckpt), max_length=32, lean=False)  # the reference's own tokenizer call
    checkpoint = HuggingFaceCheckpoint.from_directory(str(ckpt))
    checkpoint.set_preprocessor(BatchMapper(fn, batch_format="pandas", batch_size=4096))
    predictor = BatchPredictor.from_checkpoint(checkpoint=checkpoint, predictor_cls=Mirror, model_cls=HFOnCpu,
                                               tokenizer=T5Tokenizer, use_gpu=use_gpu, device_map="auto", torch_dtype=torch.float16)
    prediction = predictor.predict(validation_dataset, num_gpus_per_worker=int(use_gpu), batch_size=4, max_new_tokens=7)
    input_data_pd = validation_dataset.to_pandas()
    prediction_pd = prediction.to_pandas()
    outputs = input_data_pd.join(prediction_pd, how="inner").head(n=7)
    assert len(outputs) == 7 and "generated_output" in outputs.columns and "instruction" in outputs.columns
    assert prediction_pd["generated_output"].tolist() == gold["flow_generated_output"].tolist()
    # row for row what the dependency generates directly for the same tokenised prompts
    enc = fn(input_data_pd)
    model = load_hf_model(ckpt)
    tok = T5Tokenizer.from_pretrained(str(ckpt))
    want = []
    for lo in range(0, 10, 4):
        want += tok.batch_decode(hf_generate(model, enc["input_ids"][lo:lo + 4], enc["attention_mask"][lo:lo + 4], 7), skip_special_tokens=True)
    assert prediction_pd["generated_output"].tolist() == want


def test_mirror_predictor_equals_the_reference_predictor(gold):
    """Same model, same inputs, same kwargs as the reference class was given: identical DataFrames - for the
    dict-of-columns input of the hot path, with `labels` present (JOB/utils.py:31), with feature_columns, and for
    max_length-default calls."""
    from transformers import T5Tokenizer

    from oracle.hf_anchor import load_hf_model

    ckpt = checkpoint_dir("tiny", seed=1)
    model = load_hf_model(ckpt)
    tok = T5Tokenizer.from_pretrained(str(ckpt))
    ids, mask = gold["case_ids"], gold["case_mask"]
    mir = Mirror(model, tokenizer=tok)
    cases = [
        ({"input_ids": ids, "attention_mask": mask, "labels": ids.copy()}, dict(max_new_tokens=6)),
        ({"input_ids": ids, "attention_mask": mask, "labels": ids.copy(), "junk": ids}, dict(feature_columns=["input_ids", "attention_mask"], max_new_tokens=4)),
        ({"input_ids": ids, "attention_mask": mask}, dict()),  # GenerationConfig default max_length = 20
        ({"input_ids": ids, "attention_mask": mask}, dict(max_new_tokens=5, min_new_tokens=5)),
    ]
    for i, (data, kw) in enumerate(cases):
        b = mir._predict_numpy({k: v.copy() for k, v in data.items()}, **kw)
        assert list(b.columns) == ["generated_output"]
        assert b["generated_output"].tolist() == gold[f"case{i}_generated_output"].tolist(), i
    # the classmethod: same constructor contract (tokenizer class resolved through the checkpoint)
    from anyscale_workshop_nyc_2023_b200.rayshim.train import HuggingFaceCheckpoint

    ck = HuggingFaceCheckpoint.from_directory(str(ckpt))
    p = Mirror.from_checkpoint(ck, HFOnCpu, tokenizer=T5Tokenizer, use_gpu=False, device_map="auto", torch_dtype=torch.float16)
    assert [str(p.use_gpu), p.tokenizer.__class__.__name__, str(p.get_preprocessor())] == gold["from_checkpoint"].tolist()


def test_reference_preprocess_function_equals_the_mirror(gold):
    """utils.py:6-33 hard-codes `T5Tokenizer.from_pretrained("google/flan-t5-base")` (a hub download); with that one
    call pointed at the local tokenizer files the unmodified function produced the stored arrays, and this package's
    lean mirror produces them too."""
    from anyscale_workshop_nyc_2023_b200.workload import ASSETS

    batch = pd.DataFrame({"instruction": gold["pre_instruction"].tolist(), "input": gold["pre_input"].tolist()})
    mir = make_preprocess_function(str(ASSETS / "tokenizer"))(batch)
    assert set(mir) == {"input_ids", "attention_mask", "labels"}
    for k in mir:
        assert np.array_equal(gold[f"pre_{k}"], mir[k]), k
