#!/usr/bin/env python
"""bench.py - the reference's headline workload on B200: FLAN-T5 greedy batch inference,
512-token prompts -> 128 generated tokens, batch 256 (BASELINE.json configs[1]).

A "step" is one pass of the hot path over one 256-prompt batch (tokenised synthetic prompts,
seeded random FLAN-T5-base weights: no checkpoints or datasets exist offline).

  value      generated tokens/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        the same metric through the reference-facing plug-in call
             HuggingFaceModelPredictor._predict_numpy(host numpy batch) -> DataFrame of strings:
             pinned H2D copy + generate + D2H copy + detokenisation inside the timed region
  roofline   cross-attention decode kernel (85 % of decode bytes): algorithmic bytes / launch duration
             INSIDE the step graph (per-chain launches, %globaltimer stamps taken in an extra untimed
             pass) vs the measured HBM copy bandwidth; the isolated-launch figure, the whole decode
             loop's, the encoder's and the whole batch's fractions beside it
  parity     a sample of the LAST TIMED batch's rows against transformers' eager model in the same
             dtype on this GPU (outside the timed region)
  incumbent_hf_gpu  transformers eager bf16 generate on this GPU, same workload, same run
  cpu_baseline  the reference's CPU path (HF eager fp32 generate through the predictor plug-in),
             one 64-prompt batch of the same workload, thread count chosen by a 3-point sweep

python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
python bench.py --impl reference ...                     (reference arm: the CPU path only)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "generated tokens/sec (and prompts/sec) FLAN-T5-base 512->128"
UNIT = "tokens/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="flan-t5-base")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--seq", type=int, default=512)
    ap.add_argument("--new", type=int, default=128)
    ap.add_argument("--lengths", default="full", choices=["full", "alpaca", "uniform"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"],
                    help="numerics contract: bf16 (headline) or the notebook's literal torch_dtype=float16 (fp32 wo, fp32 residual stream)")
    ap.add_argument("--cpu-sample", type=int, default=64, help="prompts per CPU step (one batch of this size)")
    ap.add_argument("--cpu-timeout", type=int, default=420, help="seconds allowed for the in-run CPU baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--hf-gpu-batches", type=int, default=2, help="timed 256-prompt batches of the HF-eager-on-GPU incumbent (0 = skip)")
    ap.add_argument("--parity-rows", type=int, default=16, help="rows of the last timed batch checked against HF on this GPU (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the tokens generate() returned in the last timed step (rank 0) as "
                         "DIR/generated_tokens.npy (float32), so that two builds can be compared on identical seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return a


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def log(msg: str) -> None:
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def effective_cores() -> int:
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(n, 1)


def workload_name(a):
    # BASELINE.json: configs[1] = FLAN-T5-base, batch 256, 512-in/128-out on one B200 (the config the metric is
    # quoted on); configs[3] = the same shape with FLAN-T5-large (HBM-roofline report); configs[0] is the CPU case
    tag = {"flan-t5-base": "BASELINE configs[1]", "flan-t5-large": "BASELINE configs[3] shape", "flan-t5-small": "configs[0] model at the configs[1] shape"}
    std = a.batch == 256 and a.seq == 512 and a.new == 128 and a.lengths == "full"
    note = tag.get(a.model, "custom") if std else "custom shape"
    return f"{a.model} batch {a.batch} {a.seq}-in/{a.new}-out greedy, lengths={a.lengths} ({note})"


# --------------------------------------------------------------------------- clocks sampling
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, smax, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # samples under load = the upper half (idle samples at the edges pull the median down)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU path (reference arm / baseline)
def _cpu_predictor(a):
    """HF eager fp32 model behind this package's mirror of the reference's predictor plug-in (kind "port"; the
    arithmetic is the genuine dependency, and tests/test_reference_predictor_cpu.py pins the mirror to the
    reference's own class output for output)."""
    import torch
    from transformers import T5Tokenizer

    from anyscale_workshop_nyc_2023_b200.predictor import HuggingFaceModelPredictor
    from anyscale_workshop_nyc_2023_b200.workload import checkpoint_dir
    from oracle.hf_anchor import load_hf_model

    ckpt = checkpoint_dir(a.model, seed=0)
    model = load_hf_model(ckpt, dtype=torch.float32, device="cpu")
    tok = T5Tokenizer.from_pretrained(str(ckpt))
    return HuggingFaceModelPredictor(model, tokenizer=tok), "port"


def run_cpu_path(a, steps: int, warmup: int, sample: int):
    """The reference's CPU implementation of the path on the host cores: `steps` predictor calls, each ONE batch of
    `sample` prompts of the same workload. The intra-op thread count is chosen by a 3-point sweep on a short probe
    (eager generate is ~4k small ATen ops per decode step: more threads is not monotonically faster). Returns tokens/s."""
    import torch

    from anyscale_workshop_nyc_2023_b200.synth import SPECS, synthetic_token_batch

    spec = SPECS[a.model]
    cores = effective_cores()
    pred, kind = _cpu_predictor(a)
    ids0, mask0 = synthetic_token_batch(1, 16, spec.vocab_size, seed=1, lengths="full")
    pred._predict_numpy({"input_ids": ids0, "attention_mask": mask0}, max_new_tokens=2)  # lazy-init costs, untimed
    sweep = {}
    forced = os.environ.get("B200T5_CPU_THREADS")
    cands = [int(forced)] if forced else sorted({max(cores // 4, 1), max(cores // 2, 1), cores})
    pids, pmask = synthetic_token_batch(sample, a.seq, spec.vocab_size, seed=999, lengths=a.lengths)
    probe_new = 8
    for n in cands:
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        pred._predict_numpy({"input_ids": pids, "attention_mask": pmask, "labels": pids.copy()},
                            max_new_tokens=probe_new, min_new_tokens=probe_new)
        sweep[n] = time.perf_counter() - t0
        log(f"cpu path: thread sweep {n} threads -> {sweep[n]:.2f} s for {sample} prompts x {probe_new} tokens")
    threads = min(sweep, key=sweep.get)
    torch.set_num_threads(threads)
    log(f"cpu path [{kind}]: {threads} torch threads of {cores} usable (host reports {os.cpu_count()} cpus), {sample} prompts/step")
    times = []
    for s in range(warmup + steps):
        ids, mask = synthetic_token_batch(sample, a.seq, spec.vocab_size, seed=1000 + s, lengths=a.lengths)
        t0 = time.perf_counter()
        df = pred._predict_numpy({"input_ids": ids, "attention_mask": mask, "labels": ids.copy()},
                                 max_new_tokens=a.new, min_new_tokens=a.new)
        dt = time.perf_counter() - t0
        assert len(df) == sample
        log(f"cpu path step {s}: {dt:.1f} s")
        if s >= warmup:
            times.append(dt)
    total = sum(times)
    toks = steps * sample * a.new
    return {"value": toks / total, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{steps} step(s) x one batch of {sample} prompts of the same {a.seq}->{a.new} workload, HF transformers eager "
                      "fp32 generate via the predictor plug-in mirror, "
                      f"torch threads={threads} (3-point sweep {dict((k, round(v, 2)) for k, v in sweep.items())} s per probe; "
                      f"{cores} usable cores)",
            "prompts_per_s": steps * sample / total, "ms_per_step": 1e3 * total / steps,
            "thread_sweep_s": {str(k): v for k, v in sweep.items()}}


def main_reference(a):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    steps = a.steps
    warm = min(a.warmup, 1)  # CPU steps are seconds long; at most one warm-up pass
    # bounded: one 64-prompt batch per step for short runs, smaller batches when the driver asks for many steps
    sample = a.cpu_sample if steps <= 3 else max(8, min(a.cpu_sample, 16))
    base = run_cpu_path(a, steps, warm, sample)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "sampled_prompts_per_step": sample},
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "thread_sweep_s")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "prompts_per_s": base["prompts_per_s"],
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------- HF on the same GPU: parity + incumbent
def hf_gpu_legs(a, ckpt, spec, last_batch, last_out, dtype, model=None):
    """transformers' eager model in the same dtype on this GPU (torch 2.11 + cuBLAS: 'the existing Blackwell path').
    (1) parity of a sample of the last TIMED batch, (2) its own throughput on the same workload."""
    import numpy as np
    import torch

    from anyscale_workshop_nyc_2023_b200.synth import synthetic_token_batch
    from oracle.hf_anchor import hf_generate, hf_teacher_forced_logits, load_hf_model

    out = {}
    hf = load_hf_model(ckpt, dtype=dtype, device="cuda")
    T = a.new
    if a.parity_rows > 0:
        ids, mask = last_batch
        B = ids.shape[0]
        sub = np.linspace(0, B - 1, min(a.parity_rows, B)).round().astype(int)
        ref = hf_generate(hf, ids[sub], mask[sub], T, min_new_tokens=T)
        ours = last_out[sub]
        lg = hf_teacher_forced_logits(hf, ids[sub], mask[sub], ref[:, :-1])
        lg[:, :, spec.eos_token_id] = -np.inf
        top2 = np.partition(lg, -2, axis=-1)[:, :, -2:]
        margins = top2[:, :, 1] - top2[:, :, 0]
        tau = 0.13 if dtype == torch.bfloat16 else 0.03  # tests/test_model_gpu.py: TAU / TAU_FP16
        gated = full = 0
        for r in range(len(sub)):
            low = np.where(~(margins[r] > tau))[0]
            upto = 1 + (int(low[0]) if len(low) else T)
            gated += int((ours[r, :upto] == ref[r, :upto]).all())
            full += int((ours[r] == ref[r]).all())
        out["parity"] = {
            "anchor": f"transformers {__import__('transformers').__version__} eager {str(dtype).split('.')[-1]} generate on this GPU",
            "what": f"{len(sub)} rows of the last timed batch (forced length {T})", "rows": int(len(sub)),
            "rows_equal_up_to_first_near_tie": gated / len(sub), "tau": tau,
            "rows_fully_equal": full / len(sub), "token_agreement": float((ours == ref).mean()),
            "first_tokens_equal": float((ours[:, 1] == ref[:, 1]).mean()),
        }
        if model is not None:
            # every decision with HF's own tokens fed back (nothing excluded, no divergence to compound): the
            # B200 arg-max at each of the rows x T positions against HF's, and the logit error itself
            mine = model.decode_logits(ids[sub], mask[sub], ref[:, :-1]).float().cpu().numpy()
            mine[:, :, spec.eos_token_id] = -np.inf
            same = mine.argmax(-1) == lg.argmax(-1)
            clear = margins > tau
            fin = np.isfinite(lg) & np.isfinite(mine)
            out["parity"].update({
                "teacher_forced_decisions": int(same.size), "teacher_forced_argmax_agreement": float(same.mean()),
                "teacher_forced_agreement_outside_near_ties": float(same[clear].mean()) if clear.any() else None,
                "mean_abs_logit_error_vs_hf": float(np.abs(np.where(fin, mine - lg, 0.0)).mean()),
            })
        log(f"parity vs HF on this GPU: {out['parity']}")
        log(f"parity vs HF on this GPU: {out['parity']}")
    if a.hf_gpu_batches > 0:
        B = a.batch
        times = []
        for s in range(a.hf_gpu_batches + 1):  # first pass = warm-up
            ids, mask = synthetic_token_batch(B, a.seq, spec.vocab_size, seed=5000 + s, lengths=a.lengths)
            di, dm = torch.from_numpy(ids).cuda(), torch.from_numpy(mask).cuda()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            with torch.no_grad():
                o = hf.generate(input_ids=di, attention_mask=dm, max_new_tokens=T, min_new_tokens=T, do_sample=False, num_beams=1)
            e1.record()
            torch.cuda.synchronize()
            assert o.shape == (B, T + 1)
            if s > 0:
                times.append(e0.elapsed_time(e1))
            log(f"HF eager on this GPU, batch {s}: {e0.elapsed_time(e1):.0f} ms")
        ms = sum(times) / len(times)
        out["incumbent_hf_gpu"] = {"value": B * T / (ms / 1e3), "unit": UNIT, "ms_per_step": ms,
                                   "prompts_per_s": B / (ms / 1e3),
                                   "what": f"transformers eager {str(dtype).split('.')[-1]} T5ForConditionalGeneration.generate, torch "
                                           f"{torch.__version__}, same GPU, {a.hf_gpu_batches} timed batch(es) of {B} prompts after one "
                                           "warm-up, inputs resident, CUDA events"}
    del hf
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------- B200 arm
DUMP_LIMIT_BYTES = 60 << 20  # keeps a dump under 64 MB, .npy headers included


def dump_tokens(out_dir: Path, tokens):
    """Token ids (< 2**24, exact in float32) as out_dir/generated_tokens.npy; above DUMP_LIMIT_BYTES a fixed seeded
    sample of rows, in row order, with their indices in out_dir/generated_tokens_rows.npy."""
    import numpy as np

    out_dir.mkdir(parents=True, exist_ok=True)
    rows = DUMP_LIMIT_BYTES // (4 * tokens.shape[1] + 8)
    if tokens.shape[0] > rows:
        keep = np.sort(np.random.default_rng(0).choice(tokens.shape[0], rows, replace=False))
        tokens = tokens[keep]
        np.save(out_dir / "generated_tokens_rows.npy", keep.astype(np.float64))
    np.save(out_dir / "generated_tokens.npy", tokens.astype(np.float32))


def main_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist

    from anyscale_workshop_nyc_2023_b200 import roofline
    from anyscale_workshop_nyc_2023_b200.parallel import max_over_ranks
    from anyscale_workshop_nyc_2023_b200.synth import SPECS, synthetic_token_batch
    from anyscale_workshop_nyc_2023_b200.workload import checkpoint_dir, make_batch_predictor

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a B200; there is no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    spec = SPECS[a.model]
    B, S, T, K, W = a.batch, a.seq, a.new, a.steps, max(a.warmup, 3)

    # rank 0 of the node writes the synthetic checkpoint once; the others wait for it
    if local == 0:
        ckpt = checkpoint_dir(a.model, seed=0)
    if world > 1:
        dist.barrier()
    ckpt = checkpoint_dir(a.model, seed=0)

    log(f"rank {rank}/{world}: checkpoint at {ckpt}; loading the model")
    tdtype = torch.float16 if a.dtype == "fp16" else torch.bfloat16
    os.environ.setdefault("B200T5_GC_FREEZE", "1")  # this process is a dedicated scoring process, like a pool worker
    bp = make_batch_predictor(ckpt, device_map="auto", torch_dtype=tdtype)
    from anyscale_workshop_nyc_2023_b200.rayshim.train import _ScoringWorker

    worker = _ScoringWorker(bp._checkpoint, bp._predictor_cls, {**bp._predictor_kwargs, "use_gpu": True}, False)
    predictor = worker.predictor
    model = predictor.model
    # the bench times the named configuration: one static batch per step, whatever its size (larger batches would
    # otherwise be routed through the slot pool, whose occupancy-dependent work is measured by tools/bench_stream.py)
    model.pool_size = max(model.pool_size, a.batch)

    # every rank owns its own shard of batches (dataset sharded by block index, no collective)
    def host_batch(step):
        return synthetic_token_batch(B, S, spec.vocab_size, seed=7919 * (rank + 1) + step, lengths=a.lengths)

    host = [host_batch(s) for s in range(W + K)]
    dev_batches = [(torch.from_numpy(i).to(dev), torch.from_numpy(m).to(dev)) for i, m in host]
    gen_kw = dict(max_new_tokens=T, min_new_tokens=T)  # fixed-length timing: every row emits exactly T tokens

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: inputs resident in HBM, CUDA events
    for s in range(W):
        t_w = time.perf_counter()
        model.generate(input_ids=dev_batches[s][0], attention_mask=dev_batches[s][1], **gen_kw)
        torch.cuda.synchronize()
        if rank == 0:
            log(f"warm-up step {s}: {1e3 * (time.perf_counter() - t_w):.1f} ms {model.stats()}")
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    enc_ms = dec_ms = 0.0
    dec_bytes = enc_flops = 0.0
    out = None
    e0.record()
    for s in range(W, W + K):
        out = model.generate(input_ids=dev_batches[s][0], attention_mask=dev_batches[s][1], **gen_kw)
        st = model.stats()
        launches += st["kernel_launches"]
        enc_ms += st["encoder_ms"]
        dec_ms += st["decode_ms"]
        dec_bytes += st["decode_algo_bytes"]
        enc_flops += st["encoder_flops"]
        xattn_kernel, row_chains = int(st["xattn_kernel"]), int(st["row_chains"])
        assert out.shape == (B, T + 1)
    e1.record()
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    last_out = out.cpu().numpy()  # the last TIMED batch's tokens: checked against HF below, outside the timed region
    if a.dump_outputs and rank == 0:
        dump_tokens(Path(a.dump_outputs), last_out)

    if rank == 0:
        log(f"device-resident: {elapsed_ms / K:.1f} ms/step")
    # ---------------- e2e: host numpy batch -> DataFrame of strings through the plug-in
    for s in range(min(W, 2)):
        predictor._predict_numpy({"input_ids": host[s][0], "attention_mask": host[s][1], "labels": host[s][0]}, **gen_kw)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = []
    for s in range(W, W + K):
        ts = time.perf_counter()
        df = predictor._predict_numpy({"input_ids": host[s][0], "attention_mask": host[s][1], "labels": host[s][0]}, **gen_kw)
        assert len(df) == B and isinstance(df["generated_output"].iloc[0], str)
        e2e_steps.append(1e3 * (time.perf_counter() - ts))  # (the DataFrame of strings is on the host: the step is complete)
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    barrier()

    # ---------------- roofline of the dominant kernel (cross-attention decode): inside the step graph, then alone
    model.set_option("profile_xattn", 1)  # re-captures the step graph with %globaltimer stamps; untimed passes only
    for s in (0, 1):
        model.generate(input_ids=dev_batches[s][0], attention_mask=dev_batches[s][1], **gen_kw)
    prof = model.xattn_profile()
    model.set_option("profile_xattn", 0)
    model.generate(input_ids=dev_batches[0][0], attention_mask=dev_batches[0][1], **gen_kw)  # plan for the calls below
    full_bytes = roofline.cross_attention_bytes_per_launch(spec, host[0][1].sum(axis=1).tolist())
    n_chains = max(1, row_chains)
    rows_per_launch = (B + n_chains - 1) // n_chains
    ca_chain = model.bench_cross_attention(reps=5, rows_per_launch=rows_per_launch)
    ca_full = model.bench_cross_attention(reps=5, rows_per_launch=0)

    elapsed_ms = max_over_ranks(elapsed_ms, dev)
    e2e_ms = max_over_ranks(e2e_ms, dev)

    peaks_file = ROOT / "MEASURED_PEAKS.json"
    if peaks_file.exists():
        pk = json.loads(peaks_file.read_text())
        hbm_peak, tf_peak, peak_src = float(pk["hbm_gbs"]), float(pk.get("bf16_tflops_sustained", 1458.8)), "measured (MEASURED_PEAKS.json)"
    else:
        hbm_peak, tf_peak, peak_src = 6650.0, 1400.0, "fallback (B200_PROFILING.md)"
    # DRAM bytes per launch of the roofline kernel from the committed `ncu --set full` capture (per batch row, scaled
    # to the rows one in-situ launch covers): only valid for the captured configuration (base, S=512, full-length)
    traffic = None
    tf = ROOT / "profiles" / "cross_attn_traffic.json"
    if tf.exists() and a.model == "flan-t5-base" and (S, a.lengths) == (512, "full"):
        tj = json.loads(tf.read_text()).get("attn_cross_stream_kernel" if xattn_kernel else "attn_decode_kernel<false>")
        if tj:
            traffic = tj["dram_bytes_per_launch"] * rows_per_launch / float(tj["rows_per_launch"])

    kv_gb = roofline.cross_attention_bytes_per_launch(spec, [S] * B) * spec.num_decoder_layers / 1e9
    w_gb = 2.0 * roofline.step_weight_elements(spec) / 1e9

    if rank == 0:
        tokens = world * K * B * T
        value = tokens / (elapsed_ms / 1e3)
        gbs = lambda nbytes, ms: nbytes / (ms / 1e3) / 1e9  # noqa: E731
        ach_launch = gbs(prof["bytes_per_launch"], prof["us_per_launch"] / 1e3) if prof["launches"] else None
        ach_situ = gbs(prof["bytes_per_layer"], prof["busy_us_per_layer"] / 1e3) if prof["busy_us_per_layer"] > 0 else ach_launch
        ach_chain = gbs(ca_chain["bytes_per_launch"], ca_chain["ms_per_launch"])
        ach_full = gbs(ca_full["bytes_per_launch"], ca_full["ms_per_launch"])
        dec_frac = dec_bytes / (dec_ms / 1e3) / 1e9 / hbm_peak
        enc_frac = enc_flops / (enc_ms / 1e3) / 1e12 / tf_peak
        roof_ms = (dec_bytes / K) / (hbm_peak * 1e9) * 1e3 + (enc_flops / K) / (tf_peak * 1e12) * 1e3
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": a.dtype, "data": "synthetic",
            "config": {"workload": workload_name(a), "global_batch": world * B, "prompts_per_rank_step": B,
                       "parallelism": f"dataset sharded over {world} replica(s), no collective",
                       "l2": f"inputs exceed L2 (cross-KV arena {kv_gb:.1f} GB and {w_gb:.2f} GB of decoder weights "
                             "are streamed every step vs 126 MB L2)",
                       "forced_length": "min_new_tokens == max_new_tokens", "row_chains": n_chains,
                       "host": "dedicated scoring process: gc.freeze() after the model is loaded, as rayshim/pool.py workers do"},
            "prompts_per_s": world * K * B / (elapsed_ms / 1e3),
            "e2e": {"value": tokens / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": 2 * B * S * 8,
                    "d2h_bytes_per_step": B * (T + 1) * 8, "ms_per_step": e2e_ms / K,
                    "ms_per_step_min_median_max": [min(e2e_steps), sorted(e2e_steps)[len(e2e_steps) // 2], max(e2e_steps)],
                    "api": "HuggingFaceModelPredictor._predict_numpy (numpy batch -> DataFrame[generated_output])"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            # frac = the dominant kernel AS THE TIMED PATH RUNS IT: inside the step graph, one launch per row-chain and
            # layer, next to the other chain's kernels. Every launch stamps first-CTA-start / last-CTA-end
            # (%globaltimer; two extra untimed passes). The chains' launches of a layer may OVERLAP each other and then
            # share the HBM, so the rate is taken per layer: bytes all of the layer's launches read / time during
            # which at least one of them ran (union of the intervals). frac_per_launch_in_situ = one launch's bytes /
            # its own duration (equal to frac when the launches do not overlap). frac_isolated_*: the kernel alone.
            "roofline": {"bound": "hbm", "kernel": "cross-attention decode: " + ("attn_cross_stream_kernel (TMA ring + mma.sync)" if xattn_kernel else "attn_decode_kernel<false> (per-thread loads)")
                                   + "; chosen per call from the prompt fill (B200T5_XATTN=ldg|stream|auto)",
                         "achieved": ach_situ, "peak": hbm_peak, "unit": "GB/s",
                         "frac": (ach_situ / hbm_peak) if ach_situ else None, "traffic": traffic, "peak_source": peak_src,
                         "frac_per_launch_in_situ": (ach_launch / hbm_peak) if ach_launch else None,
                         "in_situ": {"rows_per_launch": rows_per_launch, "launches_timed": prof["launches"],
                                     "algo_bytes_per_launch": prof["bytes_per_launch"], "us_per_launch": prof["us_per_launch"],
                                     "algo_bytes_per_layer": prof["bytes_per_layer"], "busy_us_per_layer": prof["busy_us_per_layer"]},
                         "frac_isolated_chain_rows": ach_chain / hbm_peak, "frac_isolated_full_batch": ach_full / hbm_peak,
                         "isolated": {"chain_rows": {"rows": rows_per_launch, **ca_chain}, "full_batch": {"rows": B, **ca_full}},
                         "decode_loop_frac_of_hbm_peak": dec_frac, "encoder_frac_of_bf16_sustained": enc_frac,
                         "whole_batch_frac": roof_ms / (elapsed_ms / K), "whole_batch_roofline_ms": roof_ms},
            "decode_loop": {"algo_gbytes_per_step_batch": dec_bytes / K / 1e9, "ms": dec_ms / K,
                            "achieved_gbs": dec_bytes / (dec_ms / 1e3) / 1e9, "frac_of_hbm_peak": dec_frac},
            "encoder": {"tflop_per_batch": enc_flops / K / 1e12, "ms": enc_ms / K,
                        "achieved_tflops": enc_flops / (enc_ms / 1e3) / 1e12, "frac_of_bf16_sustained": enc_frac},
        }
        if world == 1 and (a.parity_rows > 0 or a.hf_gpu_batches > 0):
            try:
                line.update(hf_gpu_legs(a, ckpt, spec, host[W + K - 1], last_out, tdtype, model))
            except Exception as e:  # noqa: BLE001 - the headline number must still be printed
                line["parity"] = {"error": f"{type(e).__name__}: {e}"}
        if world == 1 and not a.no_cpu_baseline:
            log("timing the CPU baseline (bounded sample, own process)")
            cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                   "--model", a.model, "--batch", str(a.batch), "--seq", str(a.seq), "--new", str(a.new),
                   "--lengths", a.lengths, "--cpu-sample", str(a.cpu_sample)]
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
            env["CUDA_VISIBLE_DEVICES"] = ""
            try:
                sub = subprocess.run(cmd, capture_output=True, text=True, timeout=a.cpu_timeout, env=env)
                ref = json.loads(sub.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref["cpu_baseline"]
            except (subprocess.TimeoutExpired, IndexError, ValueError, KeyError) as e:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": effective_cores(), "kind": "port",
                                        "sample": f"not finished within {a.cpu_timeout}s ({type(e).__name__})"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    a = parse_args()
    return main_reference(a) if a.impl == "reference" else main_b200(a)


if __name__ == "__main__":
    sys.exit(main())
