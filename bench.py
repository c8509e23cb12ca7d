#!/usr/bin/env python
"""bench.py -- utterances/sec of the alignment hot path (get_attentions + force_align).

    python bench.py --gpus N --steps K --warmup W            # this repo, one rank per GPU
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write what the last timed step returned

Headline workload (BASELINE.json configs[1]): TIMIT-shaped synthetic utterances (2-4 s, ~40 chars),
Whisper-medium dimensions with seeded random-init weights, char units, aggr=topk k=10, medfilt_width=3,
fp32 like the reference (`whisper.load_model` default, allow_tf32 off).  A step is one batch of `--batch`
utterances through get_attentions_batch + force_align_batch; with N ranks every rank aligns its own batch
(utterances are independent: weak scaling) and the job ends with the single all_gather of alignments and
metric counters.

Timed regions (CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks):
    value : mel and tokens already resident in HBM; ends with start/end times on the host
    e2e   : mel and tokens start in pinned host memory; H2D copies inside the timed region

The same run also measures, at the same N, the other configurations BASELINE.json names (key `configs`):
    librispeech : configs[2] -- the FIXED list of 2620 LibriSpeech-shaped utterances (2-30 s) is drained once by the
                  N ranks (strong scaling: LPT shards by cost, length-bucketed batches); utt/s = 2620 / slowest rank
    ami         : configs[3] -- AMI-shaped short segments (1-6 s, 5-25 subword tokens), Whisper-large-v3 dims (128 mels,
                  32 x 20 heads), subword units, aggr=mean, the reference's default medfilt_width 7; weak scaling
    probe_sweep : configs[4] -- filter_attention over all 384 heads, then every head DTW'd on its own
                  (reference probe_oracle.py:82-90) through timing.probe_heads_batch; DTWs/s
One JSON line on rank 0; see the task contract for the keys.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def _preload_cublas_emulation():
    """fp32 GEMMs of the upstream Whisper linears stay on cuBLAS (north_star); cuBLAS 12.9 can run
    them as BF16x9-emulated fp32 on the tensor cores (CUBLAS_EMULATE_SINGLE_PRECISION) at fp32
    accuracy.  torch 2.11+cu128 bundles cuBLAS 12.8, which predates that switch, so the CUDA
    toolkit's 12.9 libraries of this image are mapped first (same SONAME: torch then binds to
    them).  Must run before `import torch`.  Off with --fp32-gemm native / WCA_FP32_GEMM=native.
    There is NO silent fallback: if the libraries cannot be mapped the run ends with a non-zero status."""
    mode = os.environ.get("WCA_FP32_GEMM", "")
    for i, a in enumerate(sys.argv):
        if a == "--fp32-gemm" and i + 1 < len(sys.argv):
            mode = sys.argv[i + 1]
        elif a.startswith("--fp32-gemm="):
            mode = a.split("=", 1)[1]
    if "--impl" in sys.argv and "reference" in sys.argv:
        return "native"
    if mode == "native":
        return "native"
    import ctypes

    libdir = os.environ.get("WCA_CUBLAS_DIR", "/usr/local/cuda/lib64")
    os.environ.setdefault("CUBLAS_EMULATE_SINGLE_PRECISION", "1")
    try:
        for name in ("libcublasLt.so.12", "libcublas.so.12"):
            ctypes.CDLL(os.path.join(libdir, name), mode=ctypes.RTLD_GLOBAL)
    except OSError as e:
        sys.stderr.write(f"bench.py: cannot map the CUDA 12.9 cuBLAS from {libdir} ({e}); the benchmarked fp32-GEMM mode "
                         "is BF16x9 emulation and there is no silent fallback -- pass --fp32-gemm native to measure SIMT SGEMM\n")
        raise SystemExit(3)
    return "bf16x9"


FP32_GEMM = _preload_cublas_emulation()

import numpy as np  # noqa: E402
import torch  # noqa: E402

# stdout carries exactly ONE line (the JSON result); library banners (NCCL version, ...) go to stderr
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


METRIC = "utterances/sec (Whisper-medium char align)"
UNIT = "utt/s"
N_LIBRISPEECH = 2620  # BASELINE.json configs[2]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="medium")
    ap.add_argument("--workload", default="timit", choices=["timit", "librispeech", "ami", "probe"])
    ap.add_argument("--batch", type=int, default=32, help="utterances per step per GPU")
    ap.add_argument("--topk", type=int, default=10)
    ap.add_argument("--aggr", default=None, choices=["topk", "mean"], help="default: topk (mean for the ami workload)")
    ap.add_argument("--medfilt_width", type=int, default=3)
    ap.add_argument("--fp32-gemm", default="bf16x9", choices=["bf16x9", "native"],
                    help="cuBLAS fp32 GEMMs of the upstream linears: BF16x9-emulated fp32 (cuBLAS 12.9) or SIMT SGEMM")
    ap.add_argument("--profile-range", action="store_true",
                    help="cudaProfilerStart/Stop around the timed `value` region (for `ncu --profile-from-start off`)")
    ap.add_argument("--cpu-sample", type=int, default=10, help="utterances timed for cpu_baseline (0 = skip)")
    ap.add_argument("--configs", default="librispeech,ami,probe_sweep",
                    help="extra BASELINE.json configurations measured in the same run ('' = none)")
    ap.add_argument("--libri-utts", type=int, default=N_LIBRISPEECH, help="length of the fixed LibriSpeech-shaped list")
    ap.add_argument("--libri-batch", type=int, default=32, help="largest length-bucketed batch of the LibriSpeech drain")
    ap.add_argument("--probe-batch", type=int, default=32, help="utterances per probe-sweep step per GPU")
    ap.add_argument("--probe-heads", type=int, default=384, help="heads aligned individually per utterance")
    ap.add_argument("--probe-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step of the headline workload returned "
                         "as DIR/<name>.npy (rank 0, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.aggr is None:
        args.aggr = "mean" if args.workload == "ami" else "topk"
    if args.workload != "timit" or args.model != "medium":
        args.configs = ""
    return args


def workload_config(args, world):
    return {
        "workload": f"{args.workload}-shaped synthetic, Whisper-{args.model} dims (random-init, seeded), "
                    f"{'subword' if args.workload == 'ami' else 'char'} units, "
                    f"aggr={args.aggr}" + (f" k={args.topk}" if args.aggr == "topk" else "") + f", medfilt_width={args.medfilt_width}",
        "utterances_per_step_per_gpu": args.batch,
        "global_batch": args.batch * world,
        "parallelism": f"utterance sharding x{world}, no data-path collective; one final all_gather",
        "cache": "inputs larger than L2: each step streams the 3 GB fp32 weights and >2 GB of activations",
        "fp32_gemm": ("cuBLAS 12.9 BF16x9-emulated fp32 (CUBLAS_EMULATE_SINGLE_PRECISION=1) for the upstream linears"
                      if FP32_GEMM == "bf16x9" else "cuBLAS SIMT SGEMM (allow_tf32 off)"),
    }


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        return False

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's CPU path on the box's host cores
# ------------------------------------------------------------------------------------------
def _reference_hot_path():
    """(module with get_attentions / force_align, kind).  `oracle/_ref/` holds the reference's OWN, unmodified
    timing.py / retokenize.py / metrics.py when __graft_entry__.build() ran where /root/reference exists (the
    directory is git-ignored and travels to the GPU box with the snapshot): kind "reference".  Otherwise the oracle
    port of the same lines (oracle/ref_path.py, pinned to fixtures the reference's files produced): kind "port".
    Either way the third-party `whisper` package they import is the restated shim (oracle/whisper_shim) -- the
    real one is not installable offline."""
    from oracle import use_shim

    use_shim()
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if all(os.path.exists(os.path.join(ref_dir, f)) for f in ("timing.py", "retokenize.py", "metrics.py")):
        import importlib

        sys.path.insert(0, ref_dir)
        try:
            for name in ("timing", "retokenize", "metrics"):
                sys.modules.pop(name, None)
            return importlib.import_module("timing"), "reference"
        finally:
            sys.path.remove(ref_dir)
    from oracle import ref_path

    return ref_path, "port"


def cpu_reference_run(args, n_utts, warm):
    """Times the reference's own CPU implementation of the path (fp32 torch on CPU with SDPA off,
    unfold().sort() median, .item() scoring loop, numba / C dtw_cpu) on `n_utts` utterances of the same
    workload, all host threads.  Returns (utt/s, seconds, cores, kind)."""
    from dataclasses import asdict

    ref, kind = _reference_hot_path()
    from whisper.model import ModelDimensions as ODims, Whisper as OWhisper

    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every host core
    try:
        n_cpu = len(os.sched_getaffinity(0))
    except AttributeError:
        n_cpu = os.cpu_count() or 1
    torch.set_num_threads(max(n_cpu, 1))

    from whisper_char_alignment_b200 import synthetic, whisper_model
    from whisper_char_alignment_b200.tokenizer import get_tokenizer

    tk = get_tokenizer(True, language="English")
    pm = whisper_model.load_model(f"random:{args.model}", None, seed=0, qk_gain=4.0)
    om = OWhisper(ODims(**asdict(pm.dims)))
    om.load_state_dict(pm.state_dict())
    om.eval()
    del pm
    utts = synthetic.WORKLOADS[args.workload](n_utts + warm, tk, n_mels=om.dims.n_mels, seed=1234)

    def one(u):
        w, _ = ref.get_attentions(u.mel, u.tokens, om, tk, u.max_frames, args.medfilt_width, 1.0)
        return ref.force_align(w, u.text_tokens, tk, "char" if args.workload != "ami" else "subword",
                               args.aggr, args.topk)

    for u in utts[:warm]:
        one(u)
    t0 = time.perf_counter()
    for u in utts[warm:]:
        one(u)
    dt = time.perf_counter() - t0
    return n_utts / dt, dt, torch.get_num_threads(), kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # a step of the reference arm is ONE utterance of the workload (bounded sample)
    per_step = 1
    ups, dt, cores, kind = cpu_reference_run(args, args.steps * per_step, max(args.warmup, 1) * per_step)
    line = {
        "impl": "reference", "metric": METRIC, "value": ups, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": workload_config(args, 1) | {"utterances_per_step_per_gpu": per_step, "global_batch": per_step},
        "cpu_baseline": {"value": ups, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{args.steps} utterances of the workload, one per step, host CPU only"},
        "e2e": {"value": ups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------
def matmul_tflops(dev, tf32: bool, n: int = 8192, reps: int = 6):
    """Sustained fp32-input matmul rate of cuBLAS on this box: with tf32=True the tf32 tensor-core peak that
    `roofline_attention` is measured against; with tf32=False the rate of the fp32 GEMM mode in use."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    try:
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(6):
            a @ b
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            a @ b
        e1.record()
        torch.cuda.synchronize()
        return reps * 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def capture_bytes(utts, L, H, d):
    """Algorithmic bytes of the capture launch(es) for a list of utterances (SURVEY.md section 8(d)):
    the maps written once, Q and K[:F] read once -- plus the head-score partials the fused epilogue leaves behind
    (one row term and F column sums of squares per head and group of 32 token rows: ~3 % of the maps), which replace
    the second full read of the maps that scoring the heads used to cost."""
    maps = sum(4 * L * H * len(u.tokens) * u.max_frames + 4 * L * (len(u.tokens) + u.max_frames) * d for u in utts)
    partials = sum(4 * L * H * -(-len(u.tokens) // 32) * (1 + u.max_frames) for u in utts)
    return float(maps + partials)


def pair_roofline(kernel_ms, step_batches, L, H, d, peak):
    ms = sum(kernel_ms.get(k, (0, 0.0))[1] for k in ("wca_capture_attention", "wca_head_scores", "wca_head_scores_from_partials"))
    by = float(sum(8 * L * H * len(u.tokens) * u.max_frames + 4 * L * (len(u.tokens) + u.max_frames) * d
                   for b in step_batches for u in b))
    gbs = by / (ms / 1000.0) / 1e9 if ms > 0 else 0.0
    return {"kernels": "wca_capture_attention + wca_head_scores[_from_partials]", "bound": "hbm", "achieved": gbs, "peak": peak,
            "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes_per_step": by / max(len(step_batches), 1),
            "ms_per_step": ms / max(len(step_batches), 1),
            "basis": "8*L*H*T*F + 4*L*(T+F)*d per utterance (SURVEY.md 8(d): maps written once and read once for scoring)"}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, results):
    """Writes what one step of force_align_batch returned, so that two builds can be compared output for output:
    per utterance the word start / end times, the DTW cost matrix and, for aggr=topk, the kept heads (layer, head)
    with their scores, each concatenated over the batch in utterance order.  Utterances that came back as the
    reference's empty sentinel add nothing.  When the matrices would take the dump past DUMP_BYTES, a fixed, seeded
    sample of their elements is written instead (`matrix_sample`, with the flat positions in `matrix_sample_index`)."""
    aligned = [r for r in results if not isinstance(r, list)]

    def cat(parts, dtype):
        return np.concatenate([np.asarray(p, dtype=dtype).ravel() for p in parts]) if parts else np.zeros(0, dtype)

    out = {"start_times": cat([r[1] for r in aligned], np.float64),
           "end_times": cat([r[2] for r in aligned], np.float64)}
    if aligned and aligned[0][4] is not None:
        out["head_scores"] = cat([[s for s, _, _ in r[4]] for r in aligned], np.float32)
        out["head_layer_head"] = cat([[lh for _, lh, _ in r[4]] for r in aligned], np.float64).reshape(-1, 2)
    matrix = cat([r[3].numpy() for r in aligned], np.float32)
    room = DUMP_BYTES - sum(a.nbytes for a in out.values()) - 4096  # 4 KB for the .npy headers
    if matrix.nbytes <= room:
        out["matrix"] = matrix
    else:  # a float32 value and its float64 position per sampled element
        idx = np.sort(np.random.default_rng(0).choice(matrix.size, room // 12, replace=False))
        out["matrix_sample"], out["matrix_sample_index"] = matrix[idx], idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist

    from whisper_char_alignment_b200 import _cabi, batching, sharding, synthetic, timing, whisper_model
    from whisper_char_alignment_b200.tokenizer import get_tokenizer

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    torch.backends.cuda.matmul.allow_tf32 = False  # fp32 like the reference's default model
    torch.backends.cudnn.allow_tf32 = False
    # the fp32 GEMM mode must be the one the config line claims: CUDA cores cannot exceed ~74 TFLOP/s
    fp32_tflops = matmul_tflops(dev, tf32=False)
    if FP32_GEMM == "bf16x9" and fp32_tflops < 85.0:  # clocks still ramping up? measure once more, longer
        fp32_tflops = matmul_tflops(dev, tf32=False, reps=20)
    if FP32_GEMM == "bf16x9" and fp32_tflops < 85.0:
        sys.stderr.write(f"bench.py: fp32 matmul runs at {fp32_tflops:.1f} TFLOP/s -- BF16x9 emulation is not active\n")
        return 3
    tf32_tflops = matmul_tflops(dev, tf32=True)

    tk = get_tokenizer(True, language="English")
    model = whisper_model.load_model(f"random:{args.model}", dev, seed=0, qk_gain=4.0)
    dims = model.dims
    L, H, d = dims.n_text_layer, dims.n_text_head, dims.n_text_state
    unit = "subword" if args.workload == "ami" else "char"
    sot = len(tk.sot_sequence)
    # one committed figure, so that the roofline fractions of runs on different boxes compare
    peak, peak_src = 6548.5, "HBM copy bandwidth measured on a B200 (BASELINE.md section 2)"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return float(x)
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x: float):
        if world == 1:
            return [float(x)]
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        return [float(p.item()) for p in parts]

    # ---------------------------------------------------------------- headline: configs[1]
    # a pool of distinct batches per rank, cycled through the steps
    n_batches = max(2, min(4, args.steps))
    pool = synthetic.WORKLOADS[args.workload](args.batch * n_batches, tk, n_mels=dims.n_mels, seed=1000 + rank)
    batches = [pool[i * args.batch: (i + 1) * args.batch] for i in range(n_batches)]
    host = [(torch.stack([u.mel for u in b]).pin_memory(), [u.tokens.pin_memory() for u in b]) for b in batches]
    resident = [(m.to(dev), [t.to(dev) for t in toks]) for m, toks in host]

    def align(mels, toks, batch):
        ws, _ = timing.get_attentions_batch(mels, toks, model, tk, [u.max_frames for u in batch],
                                            args.medfilt_width, 1.0)
        return timing.force_align_batch(ws, [u.text_tokens for u in batch], tk, unit, args.aggr, args.topk)

    def step_resident(i):
        mels, toks = resident[i % n_batches]
        return align(mels, toks, batches[i % n_batches])

    def step_e2e(i):
        mels_h, toks_h = host[i % n_batches]
        mels = mels_h.to(dev, non_blocking=True)
        toks = [t.to(dev, non_blocking=True) for t in toks_h]
        return align(mels, toks, batches[i % n_batches])

    def timed(step_fn, steps, collect=None):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        last = None
        for i in range(steps):
            last = step_fn(i)
            if collect is not None:
                collect(i, last)
        if world > 1 and collect is not None:  # the job's single collective
            collect(-1, None)
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b)), last

    for i in range(args.warmup):
        step_resident(i)
    for i in range(min(args.warmup, 2)):
        step_e2e(i)

    local_alignments = {}

    def collect(i, res):
        if i < 0:
            sharding.gather_alignments(local_alignments)
            sharding.gather_counters(len(local_alignments), 0, 0)
            return
        for j, r in enumerate(res):
            if not isinstance(r, list):
                local_alignments[(i * args.batch + j) * world + rank] = (r[1], r[2])

    launches0 = _cabi.launch_count()
    if args.profile_range:
        torch.cuda.profiler.start()
    with ClockSampler(local_rank) as clocks, _cabi.KernelTimer() as kt:
        ms_value, last = timed(step_resident, args.steps, collect)
    if args.profile_range:
        torch.cuda.profiler.stop()
    launches = _cabi.launch_count() - launches0
    kernel_ms = kt.summary()
    with ClockSampler(local_rank) as clocks_e2e:
        ms_e2e, _ = timed(step_e2e, args.steps)

    total_utts = args.batch * args.steps * world
    value = total_utts / (ms_value / 1000.0)
    e2e = total_utts / (ms_e2e / 1000.0)

    # ---- bytes moved per step (counted from the tensors that are copied) -----------------
    b0 = batches[0]
    h2d = int(host[0][0].numel() * 4 + sum(t.numel() * 8 for t in host[0][1]))
    d2h = 0
    for u in b0:
        n_rows = len(u.tokens) - sot - 1
        d2h += n_rows * u.max_frames * 4 + 2 * 8 * (len(u.text.split()) + 1) + (2 * 4 * args.topk if args.aggr == "topk" else 0)

    # ---- roofline of the dominant kernel of OUR path: the capture launches of a step -------
    # PER STEP: sum of the algorithmic bytes of the steps timed / sum of the capture time of those steps (a step makes
    # one launch per frame-cluster bucket, so per-launch time x per-batch bytes would overstate multi-bucket workloads)
    used = [i % n_batches for i in range(args.steps)]
    cap_calls, cap_ms = kernel_ms.get("wca_capture_attention", (0, 0.0))
    cap_bytes_total = float(sum(capture_bytes(batches[i], L, H, d) for i in used))
    achieved = cap_bytes_total / (cap_ms / 1000.0) / 1e9 if cap_ms > 0 else 0.0
    # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this launch
    # (profiles/traffic.json, written from the .ncu-rep by tools/ncu_traffic.py); null for other shapes
    traffic = None
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["wca_capture_attention"]
        if rec["workload"] == args.workload and rec["batch"] == args.batch and rec["model"] == args.model:
            traffic = float(rec["dram_bytes_per_launch"])
    except (OSError, KeyError, ValueError):
        pass
    # ---- the tensor-bound kernel of the forward: unmasked attention (encoder self-attention + decoder cross-attention
    # output), fp32-grade = three tf32 products per contraction.  Algorithmic FLOPs = 4 * n_q * n_kv * 64 per (batch, head).
    att_calls, att_ms = kernel_ms.get("wca_full_attention", (0, 0.0))
    att_flops = []
    for b in batches:
        t_max = max(len(u.tokens) for u in b)
        att_flops.append(dims.n_audio_layer * 4.0 * len(b) * dims.n_audio_head * dims.n_audio_ctx ** 2 * 64
                         + L * 4.0 * len(b) * H * t_max * dims.n_audio_ctx * 64)
    att_step_flops = float(np.mean([att_flops[i] for i in used]))
    att_useful = att_step_flops * args.steps / (att_ms / 1000.0) / 1e12 if att_ms > 0 else 0.0
    dtw_calls, dtw_ms = kernel_ms.get("wca_dtw_align", (0, 0.0))
    cells = float(sum(sum((len(u.tokens) - sot - 1) * u.max_frames for u in batches[i]) for i in used))

    # ---------------------------------------------------------------- the other BASELINE.json configurations
    extra = {}
    wanted = [c for c in args.configs.split(",") if c]
    if "librispeech" in wanted:
        extra["librispeech"] = run_librispeech_drain(args, model, tk, dev, rank, world, peak, barrier, all_ranks)
    if "probe_sweep" in wanted:
        extra["probe_sweep"] = run_probe_sweep(args, model, tk, dev, rank, world, barrier, max_over_ranks)
    if "ami" in wanted:
        del model, resident
        torch.cuda.empty_cache()
        extra["ami"] = run_ami(args, dev, rank, world, peak, barrier, max_over_ranks)

    if rank == 0:
        cpu = None
        if world == 1 and args.cpu_sample > 0:
            ups, dt, cores, kind = cpu_reference_run(args, args.cpu_sample, 1)
            cpu = {"value": ups, "unit": UNIT, "cores": cores, "kind": kind,
                   "sample": f"{args.cpu_sample} utterances of the same workload after 1 warm-up utterance, {dt:.1f} s"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_value / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic",
            "config": workload_config(args, world) | {"fp32_matmul_tflops_measured": fp32_tflops},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(), "clocks_e2e": clocks_e2e.summary(),
            "roofline": {"kernel": "wca_capture_attention (QK^T capture + median filter + softmax [+ head-score partials])",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": cap_bytes_total / max(args.steps, 1),
                         "launches_per_step": cap_calls / max(args.steps, 1),
                         "ms_per_step": cap_ms / max(args.steps, 1),
                         "basis": "per step: sum of algorithmic bytes / sum of capture launch time (CUDA events)",
                         "fused": "head-score partials (timing.py:17-34) are produced in the capture epilogue; scoring no longer "
                                  "reads the maps (see stages_ms_per_step: wca_head_scores_from_partials vs round 1's wca_head_scores)"},
            # the pair capture + head scoring on SURVEY.md section 8(d)'s figure for it (maps written once by get_attentions
            # and read once by force_align's scoring, Q / K read once): round 1 ran it as two kernels (0.327 + 0.135 ms for
            # 1 293 MB = 0.43 of the copy peak), the fused epilogue no longer performs the read at all
            "roofline_capture_plus_scoring": pair_roofline(kernel_ms, [batches[i] for i in used], L, H, d, peak),
            "roofline_attention": {"kernel": "wca_full_attention (tcgen05, 3 x tf32 split for both contractions)", "bound": "tensor",
                                   "achieved": att_useful, "unit": "TFLOP/s", "executed_tf32": 3.0 * att_useful,
                                   "peak": tf32_tflops, "frac": 3.0 * att_useful / tf32_tflops if tf32_tflops else None,
                                   "peak_source": "measured in this run: cuBLAS tf32 matmul 8192^3, sustained (allow_tf32)",
                                   "calls_per_step": att_calls / max(args.steps, 1), "ms_per_step": att_ms / max(args.steps, 1),
                                   "algorithmic_flops_per_step": att_step_flops},
            "cpu_baseline": cpu,
            "stages_ms_per_step": {k: v[1] / args.steps for k, v in sorted(kernel_ms.items())},
            "dtw_cells_per_s": cells / (dtw_ms / 1000.0) if dtw_ms > 0 else None,
            "utterances_aligned": len(local_alignments),
            "configs": extra,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def device_mels(utts, n_mels, dev, seed):
    """Synthetic mels created directly in HBM (the drain list is 2620 x 0.96 MB): N(0, 0.3^2) over the speech part,
    zero beyond it, like synthetic.make_utterance."""
    g = torch.Generator(device=dev).manual_seed(seed)
    mels = torch.randn(len(utts), n_mels, 3000, device=dev, generator=g) * 0.3
    speech = torch.tensor([min(2 * u.max_frames, 3000) for u in utts], device=dev)
    mels *= (torch.arange(3000, device=dev)[None, None, :] < speech[:, None, None])
    return mels


def run_librispeech_drain(args, model, tk, dev, rank, world, peak, barrier, all_ranks):
    """BASELINE.json configs[2]: the fixed list of LibriSpeech-shaped utterances (2-30 s, T up to 448, F up to 1500),
    the same on every rank, drained ONCE by all ranks together -- strong scaling.  Shards are cost-balanced (LPT over
    sharding.shard_by_cost), batches are length-bucketed (batching.plan_batches).  Each rank times its own shard with
    CUDA events; the job's time is the slowest rank's."""
    from whisper_char_alignment_b200 import _cabi, batching, sharding, synthetic, timing

    dims = model.dims
    L, H, d = dims.n_text_layer, dims.n_text_head, dims.n_text_state
    sot = len(tk.sot_sequence)
    descr = synthetic.librispeech_shaped(args.libri_utts, tk, n_mels=dims.n_mels, seed=2620, with_mel=False)
    n_tok = [len(u.tokens) for u in descr]
    n_frm = [u.max_frames for u in descr]
    costs = [batching.utterance_cost(t, f, L, d, dims.n_audio_layer) for t, f in zip(n_tok, n_frm)]
    mine = sharding.shard_by_cost(costs, rank, world)
    plan, skipped = batching.plan_batches([n_tok[i] for i in mine], [n_frm[i] for i in mine], args.libri_batch,
                                          n_maps=L * H)
    plan = [[mine[j] for j in b] for b in plan]
    # longest batches first: the tail of the drain is then made of short batches
    plan.sort(key=lambda b: -sum(costs[i] for i in b))
    utts_by_batch = [[descr[i] for i in b] for b in plan]
    mels = [device_mels(ub, dims.n_mels, dev, 7000 + 131 * rank + k) for k, ub in enumerate(utts_by_batch)]
    toks = [[u.tokens.to(dev) for u in ub] for ub in utts_by_batch]

    def one(k):
        ub = utts_by_batch[k]
        ws, _ = timing.get_attentions_batch(mels[k], toks[k], model, tk, [u.max_frames for u in ub], args.medfilt_width, 1.0)
        return timing.force_align_batch(ws, [u.text_tokens for u in ub], tk, "char", "topk", args.topk)

    if plan:  # warm-up on the two extreme shapes: allocator growth, cuBLAS heuristics, cluster occupancy queries
        one(0)
        one(len(plan) - 1)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    aligned = 0
    with _cabi.KernelTimer() as kt:
        e0.record()
        for k in range(len(plan)):
            aligned += sum(1 for r in one(k) if not isinstance(r, list))
        e1.record()
    barrier()
    my_ms = e0.elapsed_time(e1)
    km = kt.summary()
    per_rank = all_ranks(my_ms)
    n_aligned = int(sum(all_ranks(float(aligned))))
    cap_calls, cap_ms = km.get("wca_capture_attention", (0, 0.0))
    dtw_calls, dtw_ms = km.get("wca_dtw_align", (0, 0.0))
    my_bytes = float(sum(capture_bytes(ub, L, H, d) for ub in utts_by_batch))
    my_cells = float(sum((len(u.tokens) - sot - 1) * u.max_frames for ub in utts_by_batch for u in ub))
    cap_gbs = my_bytes / (cap_ms / 1000.0) / 1e9 if cap_ms > 0 else 0.0
    slow = max(per_rank)
    return {
        "workload": f"LibriSpeech-shaped synthetic, fixed list of {args.libri_utts} utterances (2-30 s, T <= 448, F <= 1500), "
                    f"Whisper-medium dims, char units, aggr=topk k={args.topk}, medfilt_width={args.medfilt_width}",
        "scaling": "strong", "n_gpus": world, "utterances": args.libri_utts, "aligned": n_aligned,
        "value": args.libri_utts / (slow / 1000.0), "unit": UNIT,
        "rank_ms_max": slow, "rank_ms_mean": float(np.mean(per_rank)), "rank_ms": per_rank,
        "imbalance_measured": slow / float(np.mean(per_rank)),
        "imbalance_cost_model": {"lpt": sharding.shard_imbalance(costs, world, "lpt"),
                                 "round_robin": sharding.shard_imbalance(costs, world, "round_robin")},
        "batches_rank0": len(plan), "largest_batch": args.libri_batch,
        "decoder_padding_waste_rank0": batching.padding_waste(n_tok, plan),
        "capture_rank0": {"bound": "hbm", "achieved": cap_gbs, "peak": peak, "unit": "GB/s", "frac": cap_gbs / peak,
                          "launches": cap_calls, "ms": cap_ms, "algorithmic_bytes": my_bytes,
                          "basis": "whole shard: sum of algorithmic bytes / sum of capture launch time"},
        "dtw_cells_per_s_rank0": my_cells / (dtw_ms / 1000.0) if dtw_ms > 0 else None,
        "stages_ms_rank0": {k: v[1] for k, v in sorted(km.items())},
    }


def run_ami(args, dev, rank, world, peak, barrier, max_over_ranks, batch=32, n_steps=3):
    """BASELINE.json configs[3]: AMI-shaped short segments, Whisper-large-v3 dimensions (random init created on the device),
    subword units, aggr=mean (upper half of the layers, timing.py:84-89), medfilt_width 7 (the reference CLI's default).
    Every rank aligns its own batches (weak scaling); a step is one batch of 32 segments."""
    from whisper_char_alignment_b200 import _cabi, synthetic, timing, whisper_model
    from whisper_char_alignment_b200.tokenizer import get_tokenizer

    dims = whisper_model.dims_for("large-v3")
    model = whisper_model.random_init(dims, seed=0, qk_gain=4.0, device=dev)
    tk = get_tokenizer(True, language="English", num_languages=model.num_languages)
    L, H, d = dims.n_text_layer, dims.n_text_head, dims.n_text_state
    pool = synthetic.ami_shaped(batch * 2, tk, n_mels=dims.n_mels, seed=4000 + rank)
    groups = [pool[:batch], pool[batch:]]
    res_in = [(torch.stack([u.mel for u in g]).to(dev), [u.tokens.to(dev) for u in g]) for g in groups]

    def step(i):
        g = groups[i % 2]
        mels, toks = res_in[i % 2]
        ws, _ = timing.get_attentions_batch(mels, toks, model, tk, [u.max_frames for u in g], 7, 1.0)
        return timing.force_align_batch(ws, [u.text_tokens for u in g], tk, "subword", "mean")

    step(0)
    step(1)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with _cabi.KernelTimer() as kt:
        e0.record()
        for i in range(n_steps):
            step(i)
        e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    km = kt.summary()
    cap_calls, cap_ms = km.get("wca_capture_attention", (0, 0.0))
    by = float(sum(capture_bytes(groups[i % 2], L, H, d) for i in range(n_steps)))
    gbs = by / (cap_ms / 1000.0) / 1e9 if cap_ms > 0 else 0.0
    del model
    torch.cuda.empty_cache()
    return {
        "workload": "AMI-shaped synthetic short segments (1-6 s, 5-25 subword tokens), Whisper-large-v3 dims (128 mels, 32 x 20 "
                    "heads, random-init on the device), subword units, aggr=mean, medfilt_width=7",
        "scaling": "weak", "n_gpus": world, "steps": n_steps, "utterances_per_step_per_gpu": batch,
        "value": batch * n_steps * world / (ms / 1000.0), "unit": UNIT, "ms_per_step": ms / n_steps,
        "capture_rank0": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                          "ms_per_step": cap_ms / n_steps, "launches_per_step": cap_calls / n_steps},
        "stages_ms_per_step_rank0": {k: v[1] / n_steps for k, v in sorted(km.items())},
    }


def run_probe_sweep(args, model, tk, dev, rank, world, barrier, max_over_ranks):
    """BASELINE.json configs[4] (reference probe_oracle.py:82-90): get_attentions, filter_attention over the heads,
    then `force_align(w.unsqueeze(0), ..., aggregation="mean", topk=1)` for EVERY kept head -- 384 DTWs per
    utterance (the reference keeps 360, `:83`; BASELINE.json names all 24 x 16).  Every rank sweeps its own
    utterances (weak scaling); a step is one batch of `--probe-batch` utterances."""
    from whisper_char_alignment_b200 import _cabi, synthetic, timing

    dims = model.dims
    sot = len(tk.sot_sequence)
    n_steps = max(1, args.probe_steps)
    pool = synthetic.probe_shaped(args.probe_batch * 2, tk, n_mels=dims.n_mels, seed=5000 + rank)
    groups = [pool[: args.probe_batch], pool[args.probe_batch:]]
    res_in = [(torch.stack([u.mel for u in g]).to(dev), [u.tokens.to(dev) for u in g]) for g in groups]

    def step(i):
        g = groups[i % 2]
        mels, toks = res_in[i % 2]
        ws, _ = timing.get_attentions_batch(mels, toks, model, tk, [u.max_frames for u in g], args.medfilt_width, 1.0)
        return timing.probe_heads_batch(ws, [u.text_tokens for u in g], tk, "char", args.probe_heads)

    step(0)
    step(1)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_dtw = 0
    with _cabi.KernelTimer() as kt:
        e0.record()
        for i in range(n_steps):
            for outs, _ in step(i):
                n_dtw += sum(1 for o in outs if not isinstance(o, list))
        e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    km = kt.summary()
    dtw_calls, dtw_ms = km.get("wca_dtw_align", (0, 0.0))
    heads = min(args.probe_heads, dims.n_text_layer * dims.n_text_head)
    cells = float(sum(heads * (len(u.tokens) - sot - 1) * u.max_frames for i in range(n_steps) for u in groups[i % 2]))
    utts = args.probe_batch * n_steps * world
    return {
        "workload": f"probe_oracle head sweep: {heads} single-head alignments per utterance, probe-shaped synthetic "
                    f"(>= 18 words, 4-8 s), Whisper-medium dims, char units, medfilt_width={args.medfilt_width}",
        "scaling": "weak", "n_gpus": world, "steps": n_steps, "utterances_per_step_per_gpu": args.probe_batch,
        "value": utts / (ms / 1000.0), "unit": UNIT, "ms_per_step": ms / n_steps,
        "dtw_per_s": utts * heads / (ms / 1000.0), "dtw_aligned_rank0": n_dtw,
        "dtw_kernel_cells_per_s_rank0": cells / (dtw_ms / 1000.0) if dtw_ms > 0 else None,
        "stages_ms_per_step_rank0": {k: v[1] / n_steps for k, v in sorted(km.items())},
    }


if __name__ == "__main__":
    sys.exit(main())
