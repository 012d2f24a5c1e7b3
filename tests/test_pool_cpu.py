"""CPU-only: the one-process-per-GPU scoring pool (rayshim/pool.py) with stand-in predictors - block order, in-worker
CPU stage, persistence across predict() calls, and loud failure when a worker dies natively."""
import os

import pandas as pd
import pytest

from anyscale_workshop_nyc_2023_b200 import rayshim
from anyscale_workshop_nyc_2023_b200.rayshim.pool import GpuWorkerPool, _visible_devices
from anyscale_workshop_nyc_2023_b200.rayshim.train import Predictor


class EchoPredictor(Predictor):
    """Reports which process scored each row; dies without a Python exception when asked to."""

    @classmethod
    def from_checkpoint(cls, checkpoint, use_gpu=False, **kw):
        return cls(preprocessor=checkpoint.get_preprocessor())

    def _predict_pandas(self, data, **kw):
        if (data["text"] == "die").any():
            os._exit(77)  # what a CUDA abort / segfault looks like from the driver: no exception, no message
        if (data["text"] == "raise").any():
            raise ValueError("bad row")
        return pd.DataFrame({"generated_output": [f"{t}:{kw.get('suffix', '')}" for t in data["text"]],
                             "pid": [os.getpid()] * len(data), "gpu": [os.environ.get("CUDA_VISIBLE_DEVICES")] * len(data)})


class Ckpt:
    def __init__(self, prep=None):
        self._prep = prep

    def get_preprocessor(self):
        return self._prep


def _upper(batch):
    return pd.DataFrame({"text": batch["text"].str.upper()})


def _blocks(n_blocks, rows=3):
    return [pd.DataFrame({"text": [f"b{i}r{j}" for j in range(rows)]}) for i in range(n_blocks)]


def test_visible_devices_are_passed_through_as_strings(monkeypatch):
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "GPU-aaaa,GPU-bbbb,MIG-cccc,3")
    assert _visible_devices(3, 1) == ["GPU-aaaa", "GPU-bbbb", "MIG-cccc"]
    assert _visible_devices(2, 2) == ["GPU-aaaa,GPU-bbbb", "MIG-cccc,3"]
    assert _visible_devices(6, 1)[4] == "GPU-aaaa"  # more workers than devices wrap around


@pytest.mark.timeout(300)
def test_pool_order_persistence_and_worker_side_cpu_stage(monkeypatch):
    # two devices for the two workers whatever this host has (the stand-in predictor never touches them)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "0,1")
    with GpuWorkerPool(2, Ckpt(), EchoPredictor, {}, True) as pool:
        outs = pool.map_ordered(_blocks(7), None, None, {"suffix": "x"})
        assert [o["generated_output"].tolist() for o in outs] == [[f"b{i}r{j}:x" for j in range(3)] for i in range(7)]
        pids = [o["pid"][0] for o in outs]
        assert pids[0] == pids[2] == pids[4] == pids[6] and pids[1] == pids[3] == pids[5] and pids[0] != pids[1]
        assert {o["gpu"][0] for o in outs} == {"0", "1"} or len({o["gpu"][0] for o in outs}) == 2
        # second call: the same processes (model load and graph capture are paid once per pool, not per call),
        # each tokenising its own raw blocks
        prep = rayshim.data.BatchMapper(_upper, batch_format="pandas")
        again = pool.map_ordered(_blocks(5), None, None, {}, prep=prep)
        assert [o["generated_output"][0] for o in again] == [f"B{i}R0:" for i in range(5)]
        assert {o["pid"][0] for o in again} == set(pids)
        # a Python exception in a worker surfaces with its traceback
        bad = _blocks(3)
        bad[1].loc[0, "text"] = "raise"
        with pytest.raises(RuntimeError, match="bad row"):
            pool.map_ordered(bad, None, None, {})


@pytest.mark.timeout(300)
def test_native_death_of_a_worker_is_reported_not_hung():
    pool = GpuWorkerPool(2, Ckpt(), EchoPredictor, {}, True)
    blocks = _blocks(4)
    blocks[3].loc[1, "text"] = "die"
    with pytest.raises(RuntimeError, match=r"died .* without reporting an exception .*77"):
        pool.map_ordered(blocks, None, None, {})
    assert pool.closed
    with pytest.raises(RuntimeError, match="shut down"):
        pool.map_ordered(_blocks(1), None, None, {})


def test_overlap_tail_keeps_order_overlaps_and_propagates_errors():
    """train._overlap_tail: results in input order, two calls in flight (the host tail of block i runs while the
    lock-serialised 'GPU part' of block i+1 does), an exception of any call surfaces at its position."""
    import threading
    import time

    from anyscale_workshop_nyc_2023_b200.rayshim.train import _overlap_tail

    gpu = threading.Lock()
    gpu_span, tail_span = {}, {}

    def fn(i):
        with gpu:                      # the model's lock: one generate at a time
            a = time.perf_counter()
            time.sleep(0.05)
            gpu_span[i] = (a, time.perf_counter())
        a = time.perf_counter()
        time.sleep(0.05)               # detokenise / DataFrame tail
        tail_span[i] = (a, time.perf_counter())
        return i * i

    t0 = time.perf_counter()
    assert list(_overlap_tail(fn, range(6))) == [i * i for i in range(6)]
    overlapped = time.perf_counter() - t0
    assert sorted(gpu_span) == list(range(6))
    spans = sorted(gpu_span.values())
    assert all(b[0] >= a[1] - 1e-4 for a, b in zip(spans, spans[1:]))  # the 'GPU parts' never overlap each other
    # ... but some block's tail ran while another block was generating
    assert any(min(tail_span[i][1], gpu_span[j][1]) - max(tail_span[i][0], gpu_span[j][0]) > 0.01
               for i in range(6) for j in range(6) if i != j)
    assert overlapped < 6 * 0.1 * 0.9  # sequential would be 0.6 s; two in flight ~0.35 s
    assert list(_overlap_tail(fn, range(3), enabled=False)) == [0, 1, 4]

    def boom(i):
        if i == 2:
            raise ValueError("block 2")
        return i

    got = []
    with pytest.raises(ValueError, match="block 2"):
        for v in _overlap_tail(boom, range(5)):
            got.append(v)
    assert got == [0, 1]


def test_predictor_hands_oversized_batches_over_in_host_memory():
    """predictor._predict_numpy: a batch larger than the model's pool of decode slots stays in host memory (the slot
    pool admits prompts from host buffers); `labels` is never passed on; smaller batches take the device path."""
    import numpy as np
    import torch

    from anyscale_workshop_nyc_2023_b200.predictor import HuggingFaceModelPredictor

    class Model:
        device = "cuda:0"
        seen = None

        def takes_host_batches(self, B, S):
            return B > 4

        def generate(self, **kw):
            Model.seen = kw
            return torch.zeros((kw["input_ids"].shape[0], 2), dtype=torch.long)

    class Tok:
        def batch_decode(self, out, skip_special_tokens=True):
            return ["x"] * len(out)

    pred = HuggingFaceModelPredictor(Model(), tokenizer=Tok())
    ids = np.arange(8 * 6, dtype=np.int64).reshape(8, 6)
    df = pred._predict_numpy({"input_ids": ids, "attention_mask": np.ones_like(ids), "labels": ids}, max_new_tokens=3)
    assert len(df) == 8 and set(Model.seen) == {"input_ids", "attention_mask", "max_new_tokens"}
    assert Model.seen["input_ids"].device.type == "cpu" and torch.equal(Model.seen["input_ids"], torch.from_numpy(ids))


class NumpyPredictor(Predictor):
    """`_predict_numpy` only, like the reference's HuggingFaceModelPredictor: must be handed the tokenised COLUMNS."""

    @classmethod
    def from_checkpoint(cls, checkpoint, use_gpu=False, **kw):
        return cls(preprocessor=checkpoint.get_preprocessor())

    def _predict_numpy(self, data, **kw):
        import numpy as np

        ids = data["input_ids"]
        assert isinstance(ids, np.ndarray) and ids.ndim == 2 and ids.dtype == np.int64 and "text" not in data
        return pd.DataFrame({"generated_output": [f"{int(r.sum())}" for r in ids]})


def _tokenise(batch):
    import numpy as np

    ids = np.array([[len(t), ord(t[1]), 0, 0] for t in batch["text"]], dtype=np.int64)
    return {"input_ids": ids, "attention_mask": (ids != 0).astype(np.int64), "labels": ids.copy()}


def test_tokenised_blocks_reach_the_predictor_as_numpy_columns():
    """The worker-side CPU stage hands the predictor the preprocessor's numpy columns as they are (no DataFrame of
    per-row array objects in between: that round trip cost more host time per 4096-row block than the GPU needs to
    score it), in the pool and in the single-worker path alike; keep_columns still works on such a block."""
    from anyscale_workshop_nyc_2023_b200.rayshim.train import _ScoringWorker, _model_batch

    prep = rayshim.data.BatchMapper(_tokenise, batch_format="pandas")
    want = [[str(len(f"b{i}r{j}") + ord("0") + i) for j in range(3)] for i in range(5)]
    with GpuWorkerPool(2, Ckpt(), NumpyPredictor, {}, True) as pool:
        outs = pool.map_ordered(_blocks(5), None, None, {}, prep=prep)
        assert [o["generated_output"].tolist() for o in outs] == want
    worker = _ScoringWorker(Ckpt(), NumpyPredictor, {}, True)
    block = _model_batch(prep.transform_batch(_blocks(1)[0]))
    assert isinstance(block, dict)
    out = worker(block, ["input_ids"], ["labels"], {})
    assert out["generated_output"].tolist() == want[0] and len(out["labels"]) == 3
    # a preprocessor that returns a DataFrame keeps the pandas path
    assert isinstance(_model_batch(_upper(_blocks(1)[0])), pd.DataFrame)
