"""Generates tests/golden/reference_predictor.npz: the outputs of the original workshop project's own plug-in files,
run unmodified through this package's Ray shim, for the inputs tests/test_reference_predictor_cpu.py feeds them.

    python tests/golden/make_reference_golden.py <checkout of the original project>

`NLP_workloads/Anyscale_job/predictor.py` (HuggingFaceModelPredictor) and `utils.py` (preprocess_function) are
plain Python whose only obstacle offline is `import ray`; with the shim registered under that name they import as
they are. The model behind the predictor is transformers' own T5ForConditionalGeneration (fp32, CPU) on the seeded
tiny synthetic checkpoint, so the fixture is environment-stamped (torch / transformers versions)."""
import importlib.util
import sys
from pathlib import Path

import numpy as np
import pandas as pd
import torch
import transformers

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from anyscale_workshop_nyc_2023_b200 import rayshim  # noqa: E402
from anyscale_workshop_nyc_2023_b200.preprocess import make_preprocess_function  # noqa: E402
from anyscale_workshop_nyc_2023_b200.synth import SPECS, synthetic_alpaca_rows, synthetic_token_batch  # noqa: E402
from anyscale_workshop_nyc_2023_b200.workload import ASSETS, checkpoint_dir  # noqa: E402
from oracle.hf_anchor import load_hf_model  # noqa: E402

OUT = Path(__file__).resolve().parent / "reference_predictor.npz"
COLUMNS = ("instruction", "input", "output", "text")


def load_unmodified(path: Path, name: str):
    spec = importlib.util.spec_from_file_location(name, str(path))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


class HFOnCpu:
    @staticmethod
    def from_pretrained(path, **kw):
        return load_hf_model(path, dtype=torch.float32, device="cpu")


def main(ref_root: Path):
    rayshim.install()
    from ray.data.preprocessors import BatchMapper
    from ray.train.batch_predictor import BatchPredictor
    from transformers import T5Tokenizer

    from anyscale_workshop_nyc_2023_b200.rayshim.train import HuggingFaceCheckpoint

    job = ref_root / "NLP_workloads" / "Anyscale_job"
    Ref = load_unmodified(job / "predictor.py", "_reference_anyscale_job_predictor").HuggingFaceModelPredictor
    utils = load_unmodified(job / "utils.py", "_reference_anyscale_job_utils")
    ckpt = checkpoint_dir("tiny", seed=1)
    res = {}

    # flan-t5-batch-inference.py:119-138 with the unmodified predictor class
    rows = synthetic_alpaca_rows(11)
    res.update({f"flow_{c}": np.array(rows[c]) for c in COLUMNS})
    ds = rayshim.data.from_huggingface(rows).limit(10)
    checkpoint = HuggingFaceCheckpoint.from_directory(str(ckpt))
    checkpoint.set_preprocessor(BatchMapper(make_preprocess_function(str(ckpt), max_length=32, lean=False),
                                            batch_format="pandas", batch_size=4096))
    bp = BatchPredictor.from_checkpoint(checkpoint=checkpoint, predictor_cls=Ref, model_cls=HFOnCpu, tokenizer=T5Tokenizer,
                                        use_gpu=False, device_map="auto", torch_dtype=torch.float16)
    res["flow_generated_output"] = np.array(bp.predict(ds, num_gpus_per_worker=0, batch_size=4, max_new_tokens=7)
                                            .to_pandas()["generated_output"].tolist())

    # _predict_numpy on the cases of test_mirror_predictor_equals_the_reference_predictor
    model = load_hf_model(ckpt)
    tok = T5Tokenizer.from_pretrained(str(ckpt))
    ids, mask = synthetic_token_batch(6, 20, SPECS["tiny"].vocab_size, seed=17, lengths="uniform")
    res["case_ids"], res["case_mask"] = ids, mask
    ref = Ref(model, tokenizer=tok)
    cases = [
        ({"input_ids": ids, "attention_mask": mask, "labels": ids.copy()}, dict(max_new_tokens=6)),
        ({"input_ids": ids, "attention_mask": mask, "labels": ids.copy(), "junk": ids}, dict(feature_columns=["input_ids", "attention_mask"], max_new_tokens=4)),
        ({"input_ids": ids, "attention_mask": mask}, dict()),
        ({"input_ids": ids, "attention_mask": mask}, dict(max_new_tokens=5, min_new_tokens=5)),
    ]
    for i, (data, kw) in enumerate(cases):
        df = ref._predict_numpy({k: v.copy() for k, v in data.items()}, **kw)
        assert list(df.columns) == ["generated_output"]
        res[f"case{i}_generated_output"] = np.array(df["generated_output"].tolist())
    p = Ref.from_checkpoint(HuggingFaceCheckpoint.from_directory(str(ckpt)), HFOnCpu, tokenizer=T5Tokenizer, use_gpu=False,
                            device_map="auto", torch_dtype=torch.float16)
    res["from_checkpoint"] = np.array([str(p.use_gpu), p.tokenizer.__class__.__name__, str(p.get_preprocessor())])

    # utils.py:6-33 with its hub download of google/flan-t5-base pointed at the local tokenizer files
    real = T5Tokenizer.from_pretrained
    utils.T5Tokenizer.from_pretrained = classmethod(lambda cls, name, *a, **k: real(str(ASSETS / "tokenizer"), *a, **k))
    batch = pd.DataFrame(synthetic_alpaca_rows(40, seed=5))[["instruction", "input"]]
    res["pre_instruction"], res["pre_input"] = np.array(batch["instruction"].tolist()), np.array(batch["input"].tolist())
    enc = utils.preprocess_function(batch)
    assert set(enc) == {"input_ids", "attention_mask", "labels"}
    res.update({f"pre_{k}": np.asarray(v) for k, v in enc.items()})

    res["meta"] = np.array([f"torch={torch.__version__} transformers={transformers.__version__}"])
    np.savez_compressed(OUT, **res)
    print(OUT, {k: v.shape for k, v in res.items()})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(Path(sys.argv[1]))
