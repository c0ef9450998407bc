#!/usr/bin/env python
"""Benchmark of the hot path: RTFx (audio-seconds / second) of reverb_asr_v1-shaped attention-rescoring
decode of 30 s chunks (BASELINE.json metric), one process per GPU.

    python bench.py --gpus N --steps K --warmup W             # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W      # the reference algorithm on the host cores
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR   # + the last timed step's hypotheses, DIR/*.npy

A "step" = one recording of N x `--chunks` (default 64) 30 s chunks, chunk-sharded over the N ranks (contiguous
blocks, reverb_b200/dist.py): every rank runs
    fbank -> Conformer encoder -> CTC head -> ctc_prefix_beam_search -> attention_rescoring
on its 64 chunks and the step ENDS with the path's single collective, the NCCL all-gather of the per-chunk result
records (tokens / times / confidences) — inside the timed region.  The K steps are software-pipelined on one stream by
one host thread (ASRModel.decode_stream), the all-gathers run on a side stream.
`value`: int16 PCM already resident in HBM when the timed region starts.  `e2e`: the same through the public host API
with pinned HOST PCM — H2D of the PCM and D2H of the hypotheses inside the timed region.  Per-GPU work is fixed as N
grows ("scaling": "weak").  `strong_scaling` (same JSON line): BASELINE configs[2] — ONE 3600 s recording = 121 chunks
(120 x 2998 frames + a 238-frame tail) sharded over the N ranks through dist.transcribe_sharded (fbank per rank on its
own sample range with the 240-sample overlap, all-gather at the end), the gathered CTM compared with a 1-GPU decode of
the same recording on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CHUNK_FRAMES = 2998                     # 30 s of 10 ms frames (snip_edges)
CHUNK_SAMPLES = 480000
METRIC = "rtfx_attention_rescoring_30s_chunks"
UNIT = "audio-seconds/second"


def algorithmic_flops_per_chunk(shape) -> float:
    """Encoder + CTC head FLOPs per 30 s chunk (BASELINE.md §3 formula)."""
    d, ff, L, K, V = shape["d"], shape["ff"], shape["blocks"], shape["kernel"], shape["vocab"]
    T = CHUNK_FRAMES
    T1, F1 = (T - 1) // 2, 39
    Tp, F2 = (T1 - 1) // 2, 19
    mac = T1 * F1 * 9 * d + Tp * F2 * 9 * d * d + Tp * F2 * d * d \
        + L * Tp * (4 * d * ff + 7 * d * d + 3 * Tp * d + K * d) + 2 * Tp * shape["emb_len"] * d * d + Tp * d * V
    return 2.0 * mac


def model_dir_for(shape_name: str) -> str:
    from reverb_b200 import synth
    shape = synth.BENCH_SHAPE if shape_name == "bench" else synth.TEST_SHAPE
    d = os.path.join(os.environ.get("RVB_BENCH_DIR", "/tmp"), f"rvb_bench_model_{shape_name}")
    if not (os.path.exists(os.path.join(d, "synth.pt")) and os.path.exists(os.path.join(d, ".complete"))):
        synth.write_model_dir(d, shape=shape, seed=0, causal=True, cnn_module_norm="layer_norm", reverse_weight=0.3)
        open(os.path.join(d, ".complete"), "w").close()
    return d


def make_pcm(n_chunks: int, seed: int) -> np.ndarray:
    """n_chunks x 30 s of speech-like int16 audio; the first 5 chunks are synthesised, the rest tiled with a
    per-chunk gain so that chunks differ."""
    from reverb_b200 import synth
    base = [synth.synth_audio(30.0, seed=seed + i) for i in range(min(n_chunks, 5))]
    out = np.empty((n_chunks, CHUNK_SAMPLES), dtype=np.int16)
    for i in range(n_chunks):
        g = 1.0 - 0.03 * (i // len(base) % 8)
        out[i] = (base[i % len(base)].astype(np.float32) * g).astype(np.int16)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class NvmlClockSampler:
    """Same record through NVML in-process (nvidia_ml_py): two light queries per sample instead of an nvidia-smi
    subprocess polling nine fields.  RVB_BENCH_CLOCKS=nvml selects it."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index: int, period: float = 0.2):
        self.gpu, self.period = gpu_index, period
        self.ok = False
        self.sm, self.bits = [], 0
        self.stop_flag = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.gpu]) if visible and visible.split(",")[self.gpu].isdigit() else self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception:
            self.ok = False

    def _loop(self):
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.bits |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag.set()
        self.t.join(timeout=1.0)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.smax,
                "reasons": sorted(n for b, n in self.REASONS if self.bits & b), "samples": len(self.sm), "via": "nvml"}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def pick_threads(orc) -> int:
    """torch CPU throughput is not monotone in the thread count (a 128-way split of a 748-row GEMM thrashes):
    probe the encoder on a 10 s chunk with a few counts and keep the fastest — 'all the threads it can USE'."""
    avail = host_threads()
    cands = sorted({c for c in (avail, 64, 32, 16, 8) if 1 <= c <= avail}, reverse=True)
    feats = torch.randn(1, 998, 80) * 3 + 10
    lens = torch.tensor([998], dtype=torch.int32)
    cat = torch.tensor([1.0, 0.0])
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        orc.forward_encoder(feats, lens, cat)
        t0 = time.perf_counter()
        orc.forward_encoder(feats, lens, cat)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def run_cpu_reference(model_dir: str, n_chunks: int, steps: int, warmup: int, threads: int, batch8: bool = False):
    """The reference algorithm (oracle port: same ATen CPU operators as the reference's torch.nn graph, same Python
    searches) on the host cores.  One step = `n_chunks` 30 s chunks, batch_size 1 like the reference default; the
    reported time is the MEDIAN over the timed steps, with a per-stage split (SURVEY.md §8d).  `batch8`: one extra
    pass with 8 chunks stacked in one batch (the reference's --batch_size 8).
    Returns a dict: rtfx, sec_per_step, threads, stages (seconds per step), results (chunk 0), batch8_rtfx."""
    from oracle import fbank_np, model_ref, pipeline_ref, search_ref
    orc = pipeline_ref.OracleASR(model_dir)
    threads = pick_threads(orc) if threads <= 0 else threads
    torch.set_num_threads(threads)
    pcm = make_pcm(max(n_chunks, 8 if batch8 else 1), seed=4321)
    cat = torch.tensor([1.0, 0.0])
    keep = {}

    def run(chunks, acc):
        t0 = time.perf_counter()
        feats = torch.from_numpy(np.stack([fbank_np.fbank(pcm[c].astype(np.float32)) for c in chunks]))
        lens = torch.full((len(chunks),), feats.shape[1], dtype=torch.int32)
        t1 = time.perf_counter()
        with torch.no_grad():
            enc, enc_lens, _ = orc.forward_encoder(feats, lens, cat)
            t2 = time.perf_counter()
            ctc = model_ref.ctc_logprobs(enc, orc.sd, 0.0, 0)
            t3 = time.perf_counter()
            prefix = search_ref.ctc_prefix_beam_search(ctc, enc_lens, 10, 0)
            t4 = time.perf_counter()
            resc = orc.attention_rescoring(prefix, enc, enc_lens, 0.1, 0.0, cat)
        t5 = time.perf_counter()
        for k, v in zip(("fbank", "encoder", "ctc_head", "prefix_beam", "rescoring"), (t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4)):
            acc[k] = acc.get(k, 0.0) + v
        if chunks[0] == 0:
            keep.update(feats=feats[:1], enc=enc[:1], ctc=ctc[:1], prefix=prefix[0], resc=resc[0], pcm=pcm[0])
        return t5 - t0

    def step(acc):
        return sum(run([c], acc) for c in range(n_chunks))

    for _ in range(warmup):
        step({})
    times, stages = [], []
    for _ in range(max(steps, 1)):
        acc = {}
        times.append(step(acc))
        stages.append(acc)
    med = statistics.median(times)
    mean = sum(times) / len(times)
    st = stages[times.index(sorted(times)[len(times) // 2])]
    out = {"rtfx": n_chunks * 30.0 / med, "sec_per_step": med, "threads": threads, "passes": len(times), "mean_sec_per_step": mean,
           "stages": {k: round(v, 4) for k, v in st.items()}, "results": keep, "batch8_rtfx": None}
    if batch8:
        out["batch8_rtfx"] = 8 * 30.0 / run(list(range(8)), {})
    return out


def parity_vs_cpu(asr, eng, model, cpu) -> dict:
    """The CUDA path against the oracle pass the CPU baseline just timed (chunk 0 of its sample): measured tolerances
    for the JSON line.  Tokens on IDENTICAL fbank features (the oracle's), fbank compared separately."""
    k = cpu["results"]
    if not k:
        return {}
    dev = asr.device
    cat = torch.tensor([1.0, 0.0])
    gf = eng.fbank_batch(torch.from_numpy(k["pcm"][None]).to(dev))
    feats = k["feats"].to(dev)
    lens = torch.full((1,), feats.shape[1], dtype=torch.int32)
    enc, enc_lens = model._forward_encoder(feats, lens, cat)
    logp = model.ctc_logprobs(enc).cpu()
    res = model.decode(["ctc_greedy_search", "ctc_prefix_beam_search", "attention_rescoring"], feats, lens, 10,
                       ctc_weight=0.1, reverse_weight=0.0, blank_id=asr.blank_id, cat_embs=cat)
    from oracle import search_ref
    want_greedy = search_ref.ctc_greedy_search(k["ctc"], torch.tensor([int(enc_lens[0])]), 0)[0].tokens
    a, b = enc[0].cpu().double(), k["enc"][0].double()
    sel = k["ctc"] > -12
    return {
        "against": "oracle port (pinned bit-identical to the live reference), 1 x 30 s chunk, identical fbank features",
        "fbank_max_abs": float((gf[0].cpu() - k["feats"][0]).abs().max()),
        "encoder_rel_rms": float(((a - b) ** 2).mean().sqrt() / (b ** 2).mean().sqrt()),
        "ctc_logp_max_abs": float((logp - k["ctc"])[sel].abs().max()),
        "ctc_argmax_agreement": float((logp.argmax(-1) == k["ctc"].argmax(-1)).float().mean()),
        "greedy_ids_equal": list(res["ctc_greedy_search"][0].tokens) == list(want_greedy),
        "prefix_best_equal": list(res["ctc_prefix_beam_search"][0].tokens) == list(k["prefix"].tokens),
        "rescoring_tokens_equal": list(res["attention_rescoring"][0].tokens) == list(k["resc"].tokens),
        "rescoring_score_abs_diff": abs(float(res["attention_rescoring"][0].score) - float(k["resc"].score)),
        "tokens": len(k["resc"].tokens),
    }


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, hyps, max_tok: int) -> None:
    """Writes the hypotheses of one step to out_dir/<name>.npy as float64, one row per chunk in chunk order
    (`chunk`), token-indexed arrays padded with -1 after `num_tokens` entries.  Above DUMP_LIMIT_BYTES a fixed,
    seeded sample of the chunks is written instead, so two builds given the same arguments dump the same rows."""
    rows = np.arange(len(hyps))
    row_bytes = 8 * (4 + 3 * max_tok)
    if len(rows) * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(len(rows), DUMP_LIMIT_BYTES // row_bytes, replace=False))
    out = {"chunk": rows.astype(np.float64), "num_tokens": np.empty(len(rows)), "score": np.empty(len(rows)),
           "confidence": np.empty(len(rows))}
    for name in ("tokens", "times", "tokens_confidence"):
        out[name] = np.full((len(rows), max_tok), -1.0)
    for i, c in enumerate(rows):
        h = hyps[c]
        n = len(h.tokens)
        out["num_tokens"][i], out["score"][i], out["confidence"][i] = n, float(h.score), float(h.confidence)
        out["tokens"][i, :n] = h.tokens
        if h.times is not None:
            out["times"][i, :len(h.times)] = h.times
        if h.tokens_confidence is not None:
            out["tokens_confidence"][i, :n] = h.tokens_confidence
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _claim_stdout():
    """Only the JSON line may reach stdout: libraries (NCCL prints its version there) are redirected to stderr."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def _emit(real_fd: int, line: dict):
    sys.stdout.flush()
    os.write(real_fd, (json.dumps(line) + "\n").encode())


def main():
    real_stdout = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="rvb", choices=["rvb", "reference"])
    ap.add_argument("--chunks", type=int, default=64, help="30 s chunks per GPU per step")
    ap.add_argument("--shape", default="bench", choices=["bench", "test"])
    ap.add_argument("--reverse_weight", type=float, default=0.0)
    ap.add_argument("--mode", default="attention_rescoring", choices=["attention_rescoring", "ctc_prefix_beam_search"],
                    help="decode mode of the step: the metric's attention_rescoring (default; a superset of BASELINE "
                         "configs[1]) or configs[1] exactly (encoder + ctc_prefix_beam_search)")
    ap.add_argument("--cpu-chunks", type=int, default=1, help="30 s chunks per step of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=1, help="concurrent decoding lanes (streams + host threads) per GPU")
    ap.add_argument("--profile-step", action="store_true",
                    help="after warm-up run ONE step between cudaProfilerStart/Stop and exit (for `ncu --profile-from-start off`)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling (configs[2]) record")
    ap.add_argument("--breakdown", action="store_true", help="print a per-stage wall-clock split (synchronised) to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the hypotheses of the last timed step (every rank's chunks) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "rvb":
        ap.error("--dump-outputs applies to the CUDA path (--impl rvb)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from reverb_b200 import synth
    shape = synth.BENCH_SHAPE if args.shape == "bench" else synth.TEST_SHAPE
    stages = "fbank+ConformerEncoder+ctc_prefix_beam_search" + ("+attention_rescoring" if args.mode == "attention_rescoring" else "")
    config = {"workload": f"BASELINE configs[1]: {args.chunks}x30s chunks per GPU, {stages}, synthetic reverb_asr_v1 shape "
                          f"(d={shape['d']}, L={shape['blocks']}, V={shape['vocab']})", "mode": args.mode,
              "chunk_frames": CHUNK_FRAMES, "chunks_per_gpu": args.chunks, "beam_size": 10, "ctc_weight": 0.1,
              "reverse_weight": args.reverse_weight, "parallelism": f"chunk-sharded x{world} + all-gather of the result records per step",
              "pipelining": "software-pipelined on one stream (decode_stream)" if args.lanes <= 1 else f"{args.lanes} lanes",
              "lanes_per_gpu": args.lanes,
              "l2_policy": "inputs larger than L2 (61 MB PCM, multi-GB activations per step); no explicit flush"}

    # ------------------------------------------------------------------ reference arm (host cores)
    if args.impl == "reference":
        if rank != 0:
            return
        mdir = model_dir_for(args.shape)
        cpu = run_cpu_reference(mdir, args.cpu_chunks, max(args.steps, 1), max(args.warmup, 0), 0)
        sec = cpu["mean_sec_per_step"]                      # exactly K timed steps: total / K
        val = args.cpu_chunks * 30.0 / sec
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cpu["threads"], "kind": "port",
                                 "sample": f"{args.cpu_chunks} x 30 s chunks per step, batch_size 1, torch "
                                           f"{torch.__version__} CPU fp32, {cpu['passes']} timed steps",
                                 "median_value": cpu["rtfx"], "stages_s_per_step": cpu["stages"]},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        _emit(real_stdout, line)
        return

    # ------------------------------------------------------------------ CUDA arm
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        mdir = model_dir_for(args.shape)
    if world > 1:
        dist.barrier()
    mdir = model_dir_for(args.shape)
    import reverb_b200
    from reverb_b200 import _lib
    from reverb_b200 import dist as rdist
    from reverb_b200.engine import launch_count
    asr = reverb_b200.ReverbASR(os.path.join(mdir, "config.yaml"), os.path.join(mdir, "synth.pt"), gpu=local_rank)
    lib = _lib.load()
    eng, model = asr.engine, asr.model
    pcm_host = torch.from_numpy(make_pcm(args.chunks, seed=1234 + 17 * rank)).pin_memory()
    pcm_dev = pcm_host.to(dev)
    cat = torch.tensor([1.0, 0.0])
    lens = torch.full((args.chunks,), CHUNK_FRAMES, dtype=torch.int32)
    max_tok = eng.encoder_out_frames(CHUNK_FRAMES)
    gatherer = rdist.RecordGatherer(dev, args.chunks, max_tok)
    dkw = dict(ctc_weight=0.1, reverse_weight=args.reverse_weight, blank_id=asr.blank_id, cat_embs=cat)

    def batches(n, e2e):
        # one batch per step: (this rank's 64 chunks of) one recording; fbank on the device
        for _ in range(n):
            pcm = pcm_host.to(dev, non_blocking=True) if e2e else pcm_dev
            yield eng.fbank_batch(pcm), lens

    def run_steps(n, e2e):
        """n steps, software-pipelined; every step's records are all-gathered (side stream); returns the last step's
        local hypotheses and the gathered records of every step."""
        hyps, handles = None, []
        for res in model.decode_stream(batches(n, e2e), [args.mode], 10, **dkw):
            hyps = res[args.mode]
            handles.append(gatherer.submit(hyps))
        recs = [gatherer.wait(h) for h in handles]
        return hyps, recs

    lanes = None
    if args.lanes > 1:
        from reverb_b200.pipeline import Lanes
        lanes = Lanes(asr, args.lanes)
        assert args.chunks % args.lanes == 0
        per = args.chunks // args.lanes
        lens_lane = lens[:per]

        def lane_job(mdl, pcm):     # pcm: (per, samples) int16, device or pinned host
            if not pcm.is_cuda:
                pcm = pcm.to(dev, non_blocking=True)
            feats = mdl.engine.fbank_batch(pcm)
            return mdl.decode([args.mode], feats, lens_lane, 10, **dkw)[args.mode]

        def run_steps(n, e2e):       # noqa: F811 — thread-per-lane variant (--lanes > 1)
            hyps, handles = None, []
            src = pcm_host if e2e else pcm_dev
            for _ in range(n):
                outs = lanes.run([src[i * per:(i + 1) * per] for i in range(args.lanes)], lane_job)
                hyps = [h for o in outs for h in o]
                handles.append(gatherer.submit(hyps))
            return hyps, [gatherer.wait(h) for h in handles]

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    run_steps(max(args.warmup, 3), False)

    if args.profile_step:
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        run_steps(1, False)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        print("profiled one step", file=sys.stderr)
        return

    if args.breakdown and rank == 0:
        from reverb_b200.search import rescoring_pick_batch

        def tick(label, fn, acc):
            fn()                                  # first call may allocate; time the second
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize(dev)
            acc.append((label, (time.perf_counter() - t0) * 1e3))
            return out
        acc = []
        feats = tick("fbank", lambda: eng.fbank_batch(pcm_dev), acc)
        enc, enc_lens = tick("encoder", lambda: eng.forward_encoder(feats, lens.numpy(), cat), acc)
        tv, ti, _ = tick("ctc_head+topk", lambda: eng.ctc_topk(enc, 10, 0.0, asr.blank_id), acc)
        tick("prefix_beam only (gpu+copy)", lambda: eng.prefix_beam_search_raw(tv, ti, enc_lens, 10, asr.blank_id), acc)
        raw = tick("prefix_beam+rescoring decoder (fused native call)",
                   lambda: eng.beam_search_rescoring(tv, ti, enc, enc_lens, 10, asr.blank_id, cat, args.reverse_weight), acc)
        hy = tick("host pick", lambda: rescoring_pick_batch(*raw[:5], raw[5], raw[6], 0.1, args.reverse_weight), acc)
        tick("pack records", lambda: rdist.pack_results(hy, args.chunks, max_tok), acc)
        tick("whole step, not pipelined", lambda: model.decode([args.mode], eng.fbank_batch(pcm_dev), lens, 10, **dkw), acc)
        print("BREAKDOWN " + json.dumps({k: round(v, 2) for k, v in acc}), file=sys.stderr)
    clocks = NvmlClockSampler(local_rank) if os.environ.get("RVB_BENCH_CLOCKS") == "nvml" else ClockSampler(local_rank)
    sample_clocks = rank == 0 and os.environ.get("RVB_BENCH_NO_CLOCKS") != "1"   # A/B switch: is the sampler itself felt?
    if sample_clocks:
        clocks.start()
    # one untimed step with the per-launch GEMM timing on: fills the library's event pool, so the timed region below does
    # not create events (host time that showed up at N = 2, where the device-resident run measured slower than e2e)
    lib.rvb_gemm_profile_begin()
    run_steps(1, False)
    lib.rvb_gemm_profile_end(None, None, None)
    l0 = launch_count()
    lib.rvb_gemm_profile_begin()
    ms, (hyps, recs) = timed(lambda: run_steps(args.steps, False))
    gms, gfl, gn = C.c_double(), C.c_double(), C.c_longlong()
    lib.rvb_gemm_profile_end(C.byref(gms), C.byref(gfl), C.byref(gn))
    launches = launch_count() - l0
    clk = clocks.stop() if sample_clocks else ({"sm_mhz": None, "sm_max_mhz": None, "reasons": ["not sampled"]} if rank == 0 else None)
    audio_s = args.chunks * 30.0 * args.steps * world
    value = audio_s / (ms / 1e3)
    # the gathered records of the last step must hold every rank's chunks, this rank's block at its place
    got = rdist.unpack_results(recs[-1], max_tok)
    assert len(recs) == args.steps and len(got) == args.chunks * world, (len(recs), len(got))
    mine = got[rank * args.chunks:(rank + 1) * args.chunks]
    assert all(list(a.tokens) == list(b.tokens) and a.times == b.times for a, b in zip(mine, hyps)), "all-gather corrupted the records"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, got, max_tok)

    # end-to-end through the host API (pinned host PCM in, host hypotheses out)
    run_steps(1, True)
    ms_e2e, (hyps, recs) = timed(lambda: run_steps(args.steps, True))
    e2e_val = audio_s / (ms_e2e / 1e3)
    n_tok = sum(len(h.tokens) for h in hyps)
    d2h = int(getattr(eng, "last_d2h_bytes", 0))     # counted by the engine from the arrays the native call fills
    gather_bytes = int(recs[-1].nbytes) if world > 1 else 0

    strong = None
    if not args.no_strong:
        strong = run_strong_scaling(asr, rdist, dev, rank, world, args, sync_all)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    achieved_tf = (gfl.value / (gms.value / 1e3)) / 1e12 if gms.value > 0 else 0.0
    # dram__bytes_read.sum + dram__bytes_write.sum per GEMM launch, from the committed ncu pass over one step of this
    # same command (profiles/gemm_traffic.json, written from the ncu csv by tools/summarize_dram.py); None if absent
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "gemm_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("shape") == args.shape and tj.get("chunks") == args.chunks:
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": config,
        "clocks": clk,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(pcm_host.numel() * 2),
                "d2h_bytes_per_step": int(d2h) + gather_bytes, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gemm_tc2_kernel (2-CTA tcgen05 + TMA, all dense layers incl. conv2 implicit GEMM)",
                     "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "peak_source": peak_src, "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu)",
                     "traffic_source": traffic_src,
                     "launches_timed": int(gn.value), "kernel_ms_per_step": gms.value / args.steps,
                     "kernel_share_of_step": gms.value / ms if ms > 0 else None,
                     "algorithmic_flops_per_step": gfl.value / args.steps,
                     "whole_step_tflops": (gfl.value / (ms / 1e3)) / 1e12 if ms > 0 else None,
                     "whole_step_frac_of_peak": (gfl.value / (ms / 1e3)) / 1e12 / peak_tf if ms > 0 else None},
        "collective": {"op": "all_gather_into_tensor of per-chunk records, one per step, inside the timed region",
                       "bytes_per_rank_per_step": int(args.chunks * rdist.record_words(max_tok) * 4), "ranks": world},
        "tokens_per_step": n_tok,
        "encoder_ctc_tflop_per_step": algorithmic_flops_per_chunk(shape) * args.chunks / 1e12,
    }
    if strong is not None:
        line["strong_scaling"] = strong
    if not args.no_cpu_baseline and world == 1:
        t0 = time.time()
        cpu = run_cpu_reference(mdir, args.cpu_chunks, 3, 1, 0, batch8=True)
        line["cpu_baseline"] = {"value": cpu["rtfx"], "unit": UNIT, "cores": cpu["threads"], "kind": "port",
                                "sample": f"{args.cpu_chunks} x 30 s chunks per pass, batch_size 1: median of 3 passes after 1 "
                                          f"warm-up and a thread-count probe; oracle port of the reference on torch "
                                          f"{torch.__version__} CPU fp32, {time.time() - t0:.0f} s wall",
                                "stages_s_per_pass": cpu["stages"],
                                "batch_size_8_value": cpu["batch8_rtfx"]}
        try:
            line["parity"] = parity_vs_cpu(asr, eng, model, cpu)
            line["parity"]["mode"] = "bf16 (the timed configuration)"
            # the same read-out in the fp32-accurate mode (precision="fp32": bf16x3 tcgen05 passes + fp32 attention)
            acc = reverb_b200.ReverbASR(os.path.join(mdir, "config.yaml"), os.path.join(mdir, "synth.pt"), gpu=local_rank,
                                        precision="fp32")
            line["parity_fp32_mode"] = parity_vs_cpu(acc, acc.engine, acc.model, cpu)
            del acc
        except Exception as e:      # the parity read-out must never cost the bench line
            line.setdefault("parity", {})["error"] = repr(e)
    _emit(real_stdout, line)
    if world > 1:
        dist.destroy_process_group()


STRONG_SECONDS = 3600.0


def run_strong_scaling(asr, rdist, dev, rank, world, args, sync_all):
    """BASELINE configs[2]: ONE 1 h recording, 121 chunks of 30 s (the last one 238 frames), sharded over the ranks
    (dist.transcribe_sharded: contiguous chunk blocks, fbank per rank on its own samples, ONE all-gather of the result
    records).  Timed with CUDA events, max over ranks, host PCM -> gathered DecodeResults on every rank."""
    import torch.distributed as dist
    n_samples = int(STRONG_SECONDS * 16000)
    base = make_pcm(5, seed=977)
    reps = -(-n_samples // base.size)
    pcm = np.tile(base.reshape(-1), reps)[:n_samples].copy()
    g = 1.0 - 0.04 * ((np.arange(n_samples) // CHUNK_SAMPLES // 5) % 8)          # chunks differ
    pcm = (pcm.astype(np.float32) * g.astype(np.float32)).astype(np.int16)
    total_frames, n_chunks = rdist.chunk_plan(n_samples, CHUNK_FRAMES)
    kw = dict(mode="attention_rescoring", chunk_size=CHUNK_FRAMES, batch_size=args.chunks, beam_size=10, ctc_weight=0.1,
              reverse_weight=args.reverse_weight)

    def once():
        return rdist.transcribe_sharded(asr, pcm, **kw)

    once()
    times = []
    for _ in range(3):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        hyps = once()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        times.append(float(ms.item()))
    ms = statistics.median(times)
    assert len(hyps) == n_chunks
    out = {"workload": f"BASELINE configs[2]: one {STRONG_SECONDS:.0f} s recording = {n_chunks} chunks of 30 s (last: "
                       f"{total_frames - (n_chunks - 1) * CHUNK_FRAMES} frames), attention_rescoring, chunk-sharded x{world}, "
                       f"batches of <= {args.chunks}",
           "scaling": "strong", "value": STRONG_SECONDS / (ms / 1e3), "unit": UNIT, "ms": ms, "runs_ms": times,
           "n_gpus": world, "chunks": n_chunks, "chunks_per_rank": -(-n_chunks // world),
           "collective": "one all_gather_into_tensor of the per-chunk records, inside the timed region",
           "timed": "host int16 PCM -> fbank per rank -> decode -> all-gather -> DecodeResults on every rank"}
    if world > 1 and rank == 0:
        # the same recording decoded by rank 0 alone (no process group involved) must give the same CTM
        from reverb_b200.reverb import get_output
        total, nch = rdist.chunk_plan(n_samples, CHUNK_FRAMES)
        wave = torch.from_numpy(pcm).pin_memory().to(dev, non_blocking=True)
        feats = asr.engine.fbank(wave)[:total].unsqueeze(0)
        cat = torch.tensor([1.0, 0.0])
        solo = []
        for res in asr.model.decode_stream(asr.feats_batcher(feats, CHUNK_FRAMES, args.chunks), ["attention_rescoring"], 10,
                                           ctc_weight=0.1, reverse_weight=args.reverse_weight, blank_id=asr.blank_id,
                                           cat_embs=cat):
            solo.extend(res["attention_rescoring"])
        fmt = lambda hs: get_output("ctm", asr.tokenizer, "strong.wav", hs, 230, CHUNK_FRAMES, asr.input_frame_length,
                                    asr.output_frame_length)
        a, b = fmt(hyps), fmt(solo)
        words = lambda t: [ln.split(" ")[:5] for ln in t.split("\n")]
        out["ctm_equal_to_1gpu"] = (a == b)
        out["ctm_words_times_equal_to_1gpu"] = (words(a) == words(b))
        out["ctm_lines"] = a.count("\n") + 1
        assert words(a) == words(b), "sharded decode changed the transcript"
    return out


if __name__ == "__main__":
    main()
