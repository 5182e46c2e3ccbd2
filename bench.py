#!/usr/bin/env python
"""bench.py -- the reference's headline metric (real-time factor + aligned words/s, Whisper large-v3, 30 s windows) on
N B200s of one node.

    python bench.py [--gpus N --steps K --warmup W]              # this repo's B200 path (N>1: launched by torchrun)
    python bench.py --impl reference [...]                       # the reference's CPU path on the host cores: the UNMODIFIED
                                                                 # transcribe_stable (baseline/_ref) over the oracle's whisper
                                                                 # restatement, else the oracle port
    python bench.py --model small --workload align --windows 64  # BASELINE config 3;  --model base --windows 1: config 2;
    python bench.py --workload refine                            # config 5

One "step" (default workload, BASELINE configs 2/4 shape) = one pass of the hot path over one batch of synthetic 30 s
windows per GPU:
    log-mel -> encoder -> cross K/V -> 224 KV-cached decode steps (filters + pick, fixed token script) -> segment slicing ->
    teacher-forced decoder with cross-attention capture -> token probabilities -> QK post-processing -> DTW -> word timings
`value` times the device pipeline with inputs resident in HBM (CUDA events); `e2e` times the public API call
(`stable_ts_b200.transcribe.transcribe_windows` through `sharding.run_sharded`) from pinned HOST audio to host word lists,
including the final all-gather of word records when N > 1.  Weights are seeded random init at the true shapes (no
checkpoints offline); token scripts are seeded synthetic ids (SURVEY.md section 8d).  stdout carries exactly the one JSON
line; everything else goes to stderr.
"""
import argparse
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

# one 30 s window keeps ~0.9 GB of fp32-grade cross K/V + KV cache resident: at 100+ windows per GPU the caching allocator must
# not fragment (the cross-K/V block alone is > 80 GB)
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

import numpy as np  # noqa: E402
import torch  # noqa: E402

AUDIO_S = 30.0
N_SAMPLES = 480000


# stdout carries exactly ONE line, the JSON result: the process's real stdout is kept aside and file descriptor 1 is pointed at
# stderr for everything else (NCCL prints its version banner on stdout, libraries and warnings may print too)
_REAL_STDOUT = None


def claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit_json(obj):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=8)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--model", default="large-v3")
    p.add_argument("--workload", default="transcribe", choices=["transcribe", "align", "refine"],
                   help="transcribe: 224 forced KV-cached decode steps + word timestamps (BASELINE configs 2/4 shape); "
                        "align: forced alignment of a 100-token script (configs 1/3 shape); refine: the Refiner's inference "
                        "call (config 5): per group a [2, 480000] audio pair + token script -> probabilities and ranks, group "
                        "lengths cycling 442 / 442 / 116 tokens (a 1000-token script = 3 groups); --windows = groups per step")
    p.add_argument("--windows", type=int, default=120,
                   help="30 s windows per GPU per step (120 = one rank's share of BASELINE config 4: 8 h of audio over 8 GPUs)")
    p.add_argument("--tokens", type=int, default=None, help="text tokens per window (default: 224 transcribe / 100 align)")
    p.add_argument("--precision", default="fp16x3", choices=["fp16x3", "fp16"])
    p.add_argument("--cpu-windows", type=int, default=1, help="windows in the bounded CPU-baseline sample")
    p.add_argument("--alignment-heads", type=int, default=10,
                   help="number of cross-attention alignment heads (released large-v3 checkpoints mark 10; without a "
                        "checkpoint whisper would fall back to all heads of the upper half of the decoder)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--ncu", action="store_true", help="profiling run: warm up, then ONE step inside cudaProfilerStart/Stop")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 / float64), "
                        "so that two builds can be compared output for output on the same seeded inputs")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.tokens is None:
        a.tokens = 224 if a.workload == "transcribe" else 100
    if a.workload == "refine" and a.windows == 120:
        a.windows = 3                                       # config 5: one 1000-token script = 3 refine groups
    return a


REFINE_LENS = (442, 442, 116)


def make_refine_groups(n, eot, seed0):
    """n refine groups: (audio pair fp32 [2, 480000] -- the second row with a muted span, as the Refiner produces --, tokens)"""
    groups = []
    for i in range(n):
        a = synth_audio(N_SAMPLES, seed0 + i)
        pair = torch.stack([a, a.clone()])
        g = torch.Generator().manual_seed(977 + seed0 + i)
        lo = int(torch.randint(0, N_SAMPLES - 40000, (1,), generator=g))
        pair[1, lo:lo + 40000] = 0
        toks = torch.randint(256, eot, (REFINE_LENS[i % 3],), generator=g).tolist()
        groups.append((pair, toks))
    return groups


# ------------------------------------------------------------------------------------------------- synthetic workload
def synth_audio(n_samples: int, seed: int) -> torch.Tensor:
    """AM-modulated sinusoids + noise, peak 0.3 (SURVEY.md section 8d); same recipe as the oracle's generator."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n_samples, dtype=torch.float64) / 16000
    k = int(torch.randint(3, 6, (1,), generator=g))
    x = torch.zeros(n_samples, dtype=torch.float64)
    for _ in range(k):
        f = 100 + 3900 * float(torch.rand(1, generator=g))
        fm = 2 + 6 * float(torch.rand(1, generator=g))
        ph = 2 * np.pi * float(torch.rand(1, generator=g))
        x += torch.sin(2 * np.pi * f * t + ph) * (0.5 + 0.5 * torch.sin(2 * np.pi * fm * t))
    x += 0.01 * torch.randn(n_samples, generator=g, dtype=torch.float64)
    return (0.3 * x / x.abs().max()).float()


def make_windows(n, n_tokens, eot, seed0):
    audios, word_tokens = [], []
    for i in range(n):
        audios.append(synth_audio(N_SAMPLES, seed0 + i))
        g = torch.Generator().manual_seed(4321 + seed0 + i)
        script = torch.randint(256, eot, (n_tokens,), generator=g).tolist()
        wts, j = [], 0
        while j < n_tokens:                               # synthetic "words" of 1-3 tokens
            k = int(torch.randint(1, 4, (1,), generator=g))
            wts.append(script[j:j + k])
            j += k
        word_tokens.append(wts)
    return audios, word_tokens


def alignment_head_pairs(dims_tuple, n):
    """Deterministic stand-in for a checkpoint's alignment-head table: n (layer, head) pairs spread over the upper half
    of the decoder layers (where the released tables live)."""
    n_layer, n_head = dims_tuple[9], dims_tuple[8]
    lo = n_layer // 2
    pairs = []
    for i in range(n):
        l = lo + (i * (n_layer - lo)) // n
        pairs.append((l, (7 * i + 3) % n_head))
    return pairs


def algorithmic_flops_per_window(d, n_tokens, S):
    """SURVEY.md section 8(d): encoder + teacher-forced decoder FLOPs of one 30 s window."""
    T, M = 1500, S + n_tokens + 2
    dm, L, V, C = d.n_audio_state, d.n_audio_layer, d.n_vocab, d.n_mels
    enc = 2 * 3000 * 3 * C * dm + 2 * 1500 * 3 * dm * dm + L * (24 * T * dm * dm + 4 * T * T * dm)
    dt, Ld = d.n_text_state, d.n_text_layer
    dec = Ld * (28 * M * dt * dt + 4 * M * M * dt + 4 * T * dt * dt + 4 * M * T * dt) + 2 * M * dt * V
    return float(enc + dec)


# ------------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------- CPU arm
_CPU = {}


def host_cores() -> int:
    """Cores this process may actually use: min(affinity mask, cgroup CPU quota).  os.cpu_count() reports the whole
    host and oversubscribes badly inside a quota-limited container."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def cpu_model(args, dims_tuple):
    """The fp32 CPU model of the oracle with the bench's seeded weights and alignment heads (built once, outside any timed
    region) + its tokenizer."""
    import oracle.whisper_ref as W
    from stable_ts_b200.api import random_state_dict
    from stable_ts_b200.model import ModelDimensions
    if "model" not in _CPU:
        model = W.Whisper(W.ModelDimensions(*dims_tuple)).eval()
        model.load_state_dict(random_state_dict(ModelDimensions(*dims_tuple), seed=0))
        mask = np.zeros((dims_tuple[9], dims_tuple[8]), dtype=bool)
        for l, h in alignment_head_pairs(dims_tuple, args.alignment_heads):
            mask[l, h] = True
        model.set_alignment_heads(mask)
        tk = W.tokenizer.get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en",
                                       task="transcribe")
        _CPU.update(model=model, tk=tk)
    return _CPU["model"], _CPU["tk"]


def cpu_arm(args, dims_tuple, n_windows, threads=None):
    """The reference's CPU path for the same workload: oracle port (oracle/ = restated openai-whisper + stable-ts
    orchestration, fp32, PyTorch CPU with all host threads).  Returns (audio_s_per_s, words_per_s, seconds, cores).
    Model construction is outside the timed region (as for the GPU arm)."""
    import oracle.whisper_ref as W
    from oracle import stable_path as SP
    from stable_ts_b200.api import random_state_dict
    from stable_ts_b200.model import ModelDimensions
    cores = threads or host_cores()
    torch.set_num_threads(cores)
    model, tk = cpu_model(args, dims_tuple)
    if "data" not in _CPU:
        _CPU["data"] = (make_windows(n_windows, args.tokens, tk.eot, seed0=1000) if args.workload != "refine"
                        else make_refine_groups(n_windows, tk.eot, seed0=1000))
    if args.workload == "refine":
        t0 = time.perf_counter()
        detail, n_tok = [], 0
        for pair, toks in _CPU["data"]:
            p, r = SP.prob_and_rank(SP.refine_token_probs(model, tk, pair, toks), toks)
            detail.append(dict(p=p, rank=r))
            n_tok += len(toks)
        dt = time.perf_counter() - t0
        _CPU["detail"] = detail
        return n_windows * AUDIO_S / dt, n_tok / dt, dt, cores
    audios, wts = _CPU["data"]
    t0 = time.perf_counter()
    n_words = 0
    detail = []
    for a, wt in zip(audios, wts):
        if args.workload == "align":
            words = SP.align_audio_window(model, tk, wt, a)
            detail.append(dict(words=words, step_argmax=None))
        else:       # the per-window body of transcribe_stable: decode.py main loop (forced script) -> segment slicing ->
            # gap-padded word timestamps (timing.py:411-500), restated in oracle/stable_path.py:transcribe_window
            script = [t for w in wt for t in w]
            segs, ex = SP.transcribe_window(model, tk, a, forced_tokens=script, sample_len=len(script), language="en")
            words = [w for s_ in segs for w in s_["words"]]
            detail.append(dict(words=words, step_argmax=ex["step_argmax"]))
        n_words += len(words)
    dt = time.perf_counter() - t0
    _CPU["detail"] = detail
    return n_windows * AUDIO_S / dt, n_words / dt, dt, cores


def parity_vs_cpu(gpu_words, gpu_step_argmax, cpu_detail):
    """Window 0 of the GPU batch against the CPU oracle's result for the SAME window (same audio seed, script and weights):
    the gates of BASELINE.json north_star, evaluated at the benchmarked model depth."""
    cw = cpu_detail["words"]
    out = {"window": 0, "words_gpu": len(gpu_words), "words_cpu": len(cw), "tokens_equal": None, "worst_dt_s": None,
           "prob_rel": None, "ok": False}
    if cpu_detail["step_argmax"] is not None and gpu_step_argmax is not None:
        out["tokens_equal"] = bool(list(gpu_step_argmax) == list(cpu_detail["step_argmax"]))
        out["decode_steps_compared"] = len(cpu_detail["step_argmax"])
    if len(gpu_words) != len(cw) or any(list(a["tokens"]) != list(b["tokens"]) for a, b in zip(gpu_words, cw)):
        out["detail"] = "word lists differ"
        return out
    wt = max([0.0] + [max(abs(a["start"] - b["start"]), abs(a["end"] - b["end"])) for a, b in zip(gpu_words, cw)])
    wp = max([0.0] + [abs(a["probability"] - b["probability"]) / max(abs(b["probability"]), 1e-30) for a, b in zip(gpu_words, cw)])
    out.update(worst_dt_s=round(wt, 4), prob_rel=float(f"{wp:.3e}"),
               ok=bool(wt <= 0.0201 and wp <= 2e-3 and out["tokens_equal"] is not False))
    return out


def reference_arm(args, dims_tuple, n_windows):
    """The UNMODIFIED reference (`baseline/_ref`, the pip --target install of /root/reference) on the host cores:
    `stable_whisper.transcribe_stable` over the CPU model of `oracle.whisper_ref` -- the reference's arithmetic lives in the
    un-vendored dependency openai-whisper, absent offline, so that one module is the oracle's restatement; everything
    else (decode_stable, timestamp slicing, add_word_timestamps_stable, seek) is the reference's own code.  Greedy at
    temperature 0, `sample_len` = the bench's step count, free-running (the reference has no forced-script hook; a random-init
    model practically never emits EOT, so every window runs all steps, as the B200 arm's fixed script does).
    -> (audio_s_per_s, words_per_s, seconds, cores) or None when the install is absent."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if args.workload != "transcribe" or not os.path.isdir(os.path.join(ref_dir, "stable_whisper")):
        return None
    import oracle.whisper_ref as W
    W.install_as_whisper()
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import stable_whisper.whisper_word_level.original_whisper as ow
    model, _ = cpu_model(args, dims_tuple)
    cores = host_cores()
    torch.set_num_threads(cores)
    audio = torch.cat([synth_audio(N_SAMPLES, 1000 + i) for i in range(n_windows)])
    t0 = time.perf_counter()
    res = ow.transcribe_stable(model, audio, language="en", temperature=0.0, condition_on_previous_text=False,
                               word_timestamps=True, vad=False, suppress_silence=False, suppress_ts_tokens=False, regroup=False,
                               verbose=None, fp16=False, ignore_compatibility=True, sample_len=args.tokens)
    dt = time.perf_counter() - t0
    n_words = sum(len(s.words) for s in res.segments)
    return n_windows * AUDIO_S / dt, n_words / dt, dt, cores


def run_reference(args, dims_tuple):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                     # only rank 0 runs the CPU arm
    per_step = []
    words = 0.0
    kind, why_port = "reference", None
    for i in range(args.warmup + args.steps):
        r = None
        if kind == "reference":
            try:
                r = reference_arm(args, dims_tuple, args.cpu_windows)
                if r is None:
                    kind, why_port = "port", "baseline/_ref absent or workload without a reference driver hook"
            except Exception as e:                 # the port always exists
                kind, why_port = "port", f"unmodified reference failed: {type(e).__name__}: {e}"
        v, w, dt, cores = r if r is not None else cpu_arm(args, dims_tuple, args.cpu_windows)
        if i >= args.warmup:
            per_step.append(dt)
            words = w
        if sum(per_step) > 240:                    # bounded: stop early, report the steps that ran
            break
    dt = statistics.mean(per_step)
    value = args.cpu_windows * AUDIO_S / dt
    out = {
        "impl": "reference", "metric": f"rtfx_{args.model}_{args.workload}", "value": value, "unit": "audio_s/s", "n_gpus": args.gpus,
        "steps": len(per_step), "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload} {args.model}, {args.cpu_windows} window(s) of 30 s per step, {args.tokens} tokens/window",
                   "weights": "seeded random init"},
        "aligned_words_per_s": words, "rtf": 1.0 / value,
        "cpu_baseline": {"value": value, "unit": "audio_s/s", "cores": cores, "kind": kind,
                         "sample": (f"{args.cpu_windows} window(s) x {len(per_step)} step(s), "
                                    + ("unmodified stable_whisper.transcribe_stable (baseline/_ref) over the CPU model of "
                                       "oracle.whisper_ref (openai-whisper restated), free-running greedy"
                                       if kind == "reference" else f"oracle port of the reference CPU path ({why_port})"))},
        "e2e": {"value": value, "unit": "audio_s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_json(out)


def parity_refine(p, r, cpu):
    """Group 0 of the refine workload: probabilities within 2e-3 of the CPU oracle's; ranks equal except where the oracle
    itself has classes within that tolerance of the target (counted, not hidden)."""
    rel = float(((p - cpu["p"]).abs() / cpu["p"].clamp_min(1e-30)).max())
    eq = int((r.long() == cpu["rank"]).sum())
    return {"group": 0, "tokens": int(p.numel()), "prob_rel": float(f"{rel:.3e}"), "ranks_equal": eq,
            "rank_max_delta": int((r.long() - cpu["rank"]).abs().max()), "ok": bool(rel <= 2e-3)}


def ncu_traffic(kernel: str, algorithmic_bytes_per_launch: float):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` export of this workload (profiles/r2_ncu_*.csv:
    dram__bytes_read.sum + dram__bytes_write.sum, raw page).  Only used when the capture's launch moved the same
    algorithmic bytes as this run's launches (same windows / heads); otherwise None -- never a constant."""
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r2_ncu_*.csv")), reverse=True):
        try:
            rows = list(csv.DictReader(line for line in open(path) if not line.startswith("==")))
        except Exception:
            continue
        for r in rows:
            if kernel not in (r.get("Kernel Name") or ""):
                continue
            try:
                def val(key):
                    v = float(str(r[key]).replace(",", ""))
                    unit = (rows[0].get(key) or "").lower() if rows and rows[0] is not r else ""
                    return v * {"kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1.0)
                t = val("dram__bytes_read.sum") + val("dram__bytes_write.sum")
            except Exception:
                continue
            if 0.9 * algorithmic_bytes_per_launch <= t <= 3.0 * algorithmic_bytes_per_launch:
                return t, os.path.relpath(path, ROOT)
    return None, None


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, workload, step_out):
    """What one device step returned, as flat arrays in window order (every output of these workloads is far below
    DUMP_LIMIT_BYTES, so nothing is sampled):
      transcribe: per word its window, start, end, probability and tokens (padded with -1 to the longest word), and the
                  token argmax of every decode step [steps, windows];
      align:      per window the DTW jump indices and the text-token probabilities, concatenated, with per-window lengths;
      refine:     per group the probabilities and ranks [2, N] of its script, concatenated along N, with per-group lengths."""
    arrays = {}
    if workload == "transcribe":
        segs, info = step_out
        words = [(b, w) for b, ws in enumerate(segs) for s_ in ws for w in s_["words"]]
        width = max([len(w["tokens"]) for _, w in words] + [1])
        arrays["word_window"] = np.array([b for b, _ in words], dtype=np.float64)
        for k in ("start", "end", "probability"):
            arrays[f"word_{k}"] = np.array([w[k] for _, w in words], dtype=np.float64)
        arrays["word_tokens"] = np.array([list(w["tokens"]) + [-1] * (width - len(w["tokens"])) for _, w in words],
                                         dtype=np.float64).reshape(len(words), width)
        sa = info["step_argmax"]
        arrays["step_argmax"] = (sa.cpu().numpy() if torch.is_tensor(sa) else np.asarray(sa)).astype(np.float64)
    elif workload == "align":
        arrays["jumps"] = np.concatenate([np.asarray(j) for j, _ in step_out]).astype(np.float64)
        arrays["jumps_len"] = np.array([len(j) for j, _ in step_out], dtype=np.float64)
        arrays["token_probs"] = np.concatenate([np.asarray(p, dtype=np.float64) for _, p in step_out])
        arrays["token_probs_len"] = np.array([len(p) for _, p in step_out], dtype=np.float64)
    else:
        arrays["probs"] = torch.cat([p.float().cpu() for p, _ in step_out], dim=1).numpy()
        arrays["ranks"] = torch.cat([r.cpu() for _, r in step_out], dim=1).numpy().astype(np.float64)
        arrays["group_len"] = np.array([p.shape[1] for p, _ in step_out], dtype=np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py --dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print(f"[bench] dumped {len(arrays)} arrays ({total} bytes) to {out_dir}", file=sys.stderr)


# ------------------------------------------------------------------------------------------------- B200 arm
def run_b200(args, dims_tuple):
    import torch.distributed as dist
    from stable_ts_b200 import _lib as L
    from stable_ts_b200.alignment import align_words_batch
    from stable_ts_b200.api import load_model
    from stable_ts_b200.timing import WindowJob, align_windows
    from stable_ts_b200.tokenizer import get_tokenizer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # NCCL_DEBUG is left as the launcher set it (the rank / transport evidence must stay observable); its log goes to stderr
    # so that stdout carries only the one JSON line
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    lib = L.lib()

    model = load_model(args.model, device=dev, precision=args.precision, seed=0)
    model.alignment_head_pairs = alignment_head_pairs(dims_tuple, args.alignment_heads)
    tk = get_tokenizer(model, language="en", task="transcribe", synthetic=True)
    S = len(tk.sot_sequence)
    Wn = args.windows
    pools = 2                                           # rotate distinct inputs between steps
    refine = args.workload == "refine"
    if refine:
        from stable_ts_b200.alignment import refine_probs
        groups = [make_refine_groups(Wn, tk.eot, seed0=1000 + 100000 * rank + 1000 * p) for p in range(pools)]
        host_pairs = [[g[0].pin_memory() for g in gp] for gp in groups]
        dev_pairs = [[h.to(dev) for h in hp] for hp in host_pairs]
        batches = [([], [[g[1]] for g in gp]) for gp in groups]          # token scripts in the (audios, word_tokens) shape used below
        host_audio = dev_audio = jobs = None
    else:
        batches = [make_windows(Wn, args.tokens, tk.eot, seed0=1000 + 100000 * rank + 1000 * p) for p in range(pools)]
        host_audio = [torch.stack(b[0]).pin_memory() for b in batches]
        dev_audio = [h.to(dev) for h in host_audio]
        jobs = [[WindowJob([t for w in wt for t in w], N_SAMPLES, None) for wt in b[1]] for b in batches]

    from stable_ts_b200.decode import DecodingOptions
    from stable_ts_b200.sharding import run_sharded
    from stable_ts_b200.transcribe import transcribe_windows
    scripts = None if refine else [torch.tensor([[t for w in wt for t in w] for wt in b[1]], dtype=torch.int32).T.contiguous()
                                   for b in batches]
    dopt = DecodingOptions(language="en", sample_len=args.tokens, max_initial_timestamp=None)

    def device_step(p, use_graph=True):
        """hot path with inputs resident in HBM; only the tiny jumps/probs/token tables are read back"""
        if refine:                                   # refinement.py:291: one inference call per group, [2, n] audio + script
            return [refine_probs(model, tk, pair, g[1]) for pair, g in zip(dev_pairs[p], groups[p])]
        enc = model.encode(model.log_mel(dev_audio[p]))
        if args.workload == "align":
            return align_windows(model, tk, jobs[p], enc=enc)
        return transcribe_windows(model, tk, None, enc=enc, options=dopt, forced_tokens=scripts[p], use_graph=use_graph)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    device_step(0)                                      # first touch of every kernel / buffer (not one of the W warm-up steps)
    barrier()

    # ---- full-size self-check (size-independent property): the first, middle and last window of the full batch, processed
    # again as a batch of 3 (different kernels: mma.sync GEMV decode linears instead of the split-K GEMMs, other grid sizes,
    # other buffer offsets), must give the same words -- catches index overflow / layout faults that only show at 100+ windows
    selfcheck = None
    gpu_w0 = None                                       # window 0 of pool 0 (rank 0): compared with the CPU oracle below
    if refine and rank == 0 and not args.ncu:
        gpu_w0 = refine_probs(model, tk, host_pairs[0][0], groups[0][0][1])
    if args.workload == "align" and rank == 0 and not args.ncu:
        gpu_w0 = (align_words_batch(model, tk, [host_audio[0][0]], [batches[0][1][0]])[0], None)
    if args.workload == "transcribe" and rank == 0 and not args.ncu:
        try:
            idx = sorted({0, Wn // 2, Wn - 1})
            full, finfo = transcribe_windows(model, tk, host_audio[0], options=dopt, forced_tokens=scripts[0])
            gpu_w0 = ([w for s_ in full[0] for w in s_["words"]], finfo["step_argmax"][:, 0].tolist())
            small, _ = transcribe_windows(model, tk, host_audio[0][idx].contiguous(), options=dopt,
                                          forced_tokens=scripts[0][:, idx].contiguous())
            worst_t, worst_p, n_cmp, bad = 0.0, 0.0, 0, None
            for k, i in enumerate(idx):
                wa = [w for s_ in full[i] for w in s_["words"]]
                wb = [w for s_ in small[k] for w in s_["words"]]
                if len(wa) != len(wb) or any(x["tokens"] != y["tokens"] for x, y in zip(wa, wb)):
                    bad = f"window {i}: word lists differ ({len(wa)} vs {len(wb)} words)"
                    break
                for x, y in zip(wa, wb):
                    worst_t = max(worst_t, abs(x["start"] - y["start"]), abs(x["end"] - y["end"]))
                    worst_p = max(worst_p, abs(x["probability"] - y["probability"]) / max(abs(y["probability"]), 1e-30))
                    n_cmp += 1
            ok = bad is None and worst_t <= 0.0201 and worst_p <= 2e-3
            selfcheck = {"ok": bool(ok), "windows": idx, "words_compared": n_cmp, "worst_word_dt_s": round(worst_t, 4),
                         "worst_prob_rel": float(f"{worst_p:.3e}"), "detail": bad}
            del full, small
        except Exception as e:                              # a diagnostic: never costs the bench line
            selfcheck = {"ok": None, "detail": f"self-check did not run: {type(e).__name__}: {e}"}
        print(f"[bench] self-check: {selfcheck}", file=sys.stderr)
    # ---- value: device-timed.  The W warm-up steps run immediately before the timed region (the self-check above changes
    # batch shapes, so it must not sit between them)
    for i in range(args.warmup):
        device_step(i % pools)
    barrier()
    if args.ncu:                                        # `ncu --profile-from-start off ... bench.py --ncu`
        torch.cuda.profiler.start()
        device_step(0)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local)
    sampler.start()
    l0 = lib.stb_launch_count() + model.graph_kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    e0.record()
    for i in range(args.steps):
        last = device_step(i % pools)
        marks[i].record()
    e1.record()
    barrier()
    launches = (lib.stb_launch_count() + model.graph_kernel_launches - l0) // max(args.steps, 1)   # eager + graph replays
    ms = e0.elapsed_time(e1)
    step_ms = [round(a.elapsed_time(b), 1) for a, b in zip([e0] + marks[:-1], marks)]    # per-step spread (rank 0)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, args.workload, last)
    del last
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = world * Wn * AUDIO_S / (ms_step / 1e3)

    # ---- e2e: public API with host buffers (+ the one gather of word records when N > 1)
    def e2e_step(p):
        if refine:                                # pinned host pairs in, host probabilities + ranks out (+ one gather when N > 1)
            out = [refine_probs(model, tk, pair, g[1]) for pair, g in zip(host_pairs[p], groups[p])]
            flat = torch.cat([torch.cat([pr.flatten(), rk.flatten().float()]) for pr, rk in out])
            if world > 1:
                parts = [torch.empty_like(flat) for _ in range(world)]
                dist.all_gather(parts, flat)
                flat = torch.cat(parts)
            res = flat.cpu()
            res.n_words = world * sum(len(g[1]) for g in groups[p])
            return res

        def process(lo, hi):                      # this rank's windows (weak scaling: Wn per rank)
            if args.workload == "align":
                return align_words_batch(model, tk, list(host_audio[p]), batches[p][1])
            segs, _ = transcribe_windows(model, tk, host_audio[p], options=dopt, forced_tokens=scripts[p])   # pinned [W, 480000]
            return [[w for s_ in ws for w in s_["words"]] for ws in segs]
        return run_sharded(process, world * Wn, device=dev, lazy=True)   # gathered records; dicts built on access

    merged = None
    for i in range(max(1, min(args.warmup, 2))):
        merged = e2e_step(i % pools)
    n_words_total = getattr(merged, "n_words", None)     # words actually aligned per step over all ranks
    if n_words_total is None:
        n_words_total = sum(len(w) for w in merged)
    barrier()
    t0 = time.perf_counter()
    e2e_step_ms = []
    for i in range(args.steps):
        t1 = time.perf_counter()
        e2e_step(i % pools)
        e2e_step_ms.append(round((time.perf_counter() - t1) * 1e3, 1))
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    t = torch.tensor([e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = world * Wn * AUDIO_S / e2e_s

    # ---- roofline of the dominant kernel (tcgen05 GEMM core): per-launch CUDA events on the launching stream
    lib.stb_prof_enable(1)
    device_step(0, use_graph=False)                    # eager: every launch bracketed by events on its stream
    prof = L.prof_report()
    lib.stb_prof_enable(0)

    class _V:                                           # keep the field names used below
        def __init__(self, v): self.value = v
    gp = prof.get("gemm_tc", {"n": 0, "ms": 0.0, "flops": 0.0})
    g_ms, g_fl, g_n = _V(gp["ms"]), _V(gp["flops"]), _V(gp["n"])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    achieved_tf = g_fl.value / (g_ms.value * 1e-3) / 1e12 if g_ms.value > 0 else 0.0
    passes = 3 if args.precision == "fp16x3" else 1
    roof = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05.mma kind::f16, TMA-fed)", "achieved": achieved_tf,
            "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s (of fallback)",
            "traffic": None,
            "note": f"achieved = algorithmic fp32-grade GEMM FLOPs / event-timed GEMM time; each is executed as {passes} fp16 "
                    f"tensor-core pass(es), i.e. tensor-pipe rate = {achieved_tf * passes:.1f} TFLOP/s",
            "gemm_launches_per_step": int(g_n.value), "gemm_ms_per_step": g_ms.value,
            "gemm_share_of_step": g_ms.value / ms_step if ms_step > 0 else None,
            "algorithmic_gflop_per_window": algorithmic_flops_per_window(model.dims, args.tokens, S) / 1e9}
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    # The decode-step cross-attention is the other heavy kernel (HBM-bound: it streams every window's cross K/V once per
    # step).  Whichever of the two takes more of the step is reported as "roofline", the other as "roofline_other".
    roof_x = None
    try:
        xp = prof.get("decode_cross_attn")
        if xp and xp["ms"] > 0 and xp["n"] > 0:
            x_gbs = xp["bytes"] / (xp["ms"] * 1e-3) / 1e9
            H = model.dims.n_text_head
            variant = {0: "decode_cross_attn_kernel (scalar lanes)", 1: "decode_cross_attn_tc_kernel (ldmatrix + mma.sync)"}.get(
                L.get_option("xattn_tc"), "decode_cross_attn")
            traffic, traffic_src = ncu_traffic(variant.split(" ")[0], xp["bytes"] / xp["n"])
            roof_x = {"bound": "hbm", "kernel": variant + ": flash-decoding over the per-window cross K/V, TMA-fed",
                      "achieved": x_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": x_gbs / hbm_peak,
                      "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                      "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": xp["bytes"] / xp["n"],
                      "avg_launch_us": xp["ms"] * 1e3 / xp["n"], "launches_per_step": int(xp["n"]), "ms_per_step": xp["ms"],
                      "share_of_step": xp["ms"] / ms_step if ms_step > 0 else None,
                      "note": "achieved = algorithmic bytes per launch (B x H x 2 x 1500 x 64 x 2 B: fp16 K and V planes) / "
                              "event-timed average launch duration"}
    except Exception as e:                                  # diagnostics must never cost the bench line
        print(f"[bench] cross-attention roofline skipped: {e}", file=sys.stderr)
        roof_x = None
    # third candidate: the decode-step linears (one cluster split-K launch per Linear; HBM-bound on the weight stream)
    roof_l = None
    try:
        lp = prof.get("decode_linear")
        if lp and lp["ms"] > 0 and lp["n"] > 0:
            l_gbs = lp["bytes"] / (lp["ms"] * 1e-3) / 1e9
            traffic, traffic_src = ncu_traffic("decode_linear_kernel", lp["bytes"] / lp["n"])
            roof_l = {"bound": "hbm", "kernel": "decode_linear_kernel (swapped tcgen05 GEMM, cluster split-K over DSMEM)",
                      "achieved": l_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": l_gbs / hbm_peak,
                      "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                      "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": lp["bytes"] / lp["n"],
                      "avg_launch_us": lp["ms"] * 1e3 / lp["n"], "launches_per_step": int(lp["n"]), "ms_per_step": lp["ms"],
                      "share_of_step": lp["ms"] / ms_step if ms_step > 0 else None,
                      "note": "achieved = (weight planes + activation planes + output) bytes per launch, averaged over the step's "
                              "launches / event-timed average launch duration"}
    except Exception as e:
        print(f"[bench] decode-linear roofline skipped: {e}", file=sys.stderr)
    roof["ms_per_step"] = g_ms.value
    cands = sorted([r for r in (roof, roof_x, roof_l) if r is not None], key=lambda r: -r["ms_per_step"])
    roof, roof_other = cands[0], (cands[1:] or None)
    kernels = {k: {"launches": v["n"], "ms": round(v["ms"], 3),
                   "GBps": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["ms"] > 0 and v["bytes"] > 0 else None,
                   "hbm_frac": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / hbm_peak, 3) if v["ms"] > 0 and v["bytes"] > 0 else None}
               for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}

    if world > 1:                                       # every GPU number is final: the CPU arm below is rank 0 alone
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    cpu, parity = None, None
    if not args.no_cpu_baseline:
        v, w, dt, cores = cpu_arm(args, dims_tuple, args.cpu_windows)
        cpu = {"value": v, "unit": "audio_s/s", "cores": cores, "kind": "port", "aligned_words_per_s": w,
               "sample": f"{args.cpu_windows} window(s) of the same workload ({dt:.1f} s of CPU work), oracle port of the "
                         f"reference CPU path, fp32, torch threads = {cores}"}
        if gpu_w0 is not None:                          # same window (audio seed 1000, script, weights) through both paths
            try:
                parity = (parity_refine(gpu_w0[0].cpu(), gpu_w0[1].cpu(), _CPU["detail"][0]) if refine else
                          parity_vs_cpu(gpu_w0[0], gpu_w0[1], _CPU["detail"][0]))
            except Exception as e:
                parity = {"ok": None, "detail": f"parity check did not run: {type(e).__name__}: {e}"}
            print(f"[bench] parity_vs_cpu: {parity}", file=sys.stderr)
    out = {
        "metric": f"rtfx_{args.model}_{args.workload}", "value": value, "unit": "audio_s/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 x3 split (fp32-grade), fp32 accumulate" if args.precision == "fp16x3" else "f16, fp32 accumulate",
        "data": "synthetic", "peak_hbm_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1),
        "step_ms": step_ms, "e2e_step_ms": e2e_step_ms, "selfcheck": selfcheck,
        "allocator": {k: int(torch.cuda.memory_stats().get(k, 0)) for k in ("num_alloc_retries", "num_ooms", "num_device_alloc",
                                                                               "num_device_free")},
        "config": {"workload": (f"transcribe+word_timestamps {args.model}: {Wn} windows of 30 s per GPU per step, {args.tokens} forced "
                                "KV-cached decode steps then word alignment (BASELINE configs 2/4 shape)") if args.workload == "transcribe"
                   else (f"align {args.model}: {Wn} windows of 30 s per GPU per step, {args.tokens} text tokens/window "
                         "(BASELINE configs 1/3 shape)") if args.workload == "align"
                   else (f"refine {args.model}: {Wn} refine groups per GPU per step, each one inference call of the Refiner: audio "
                         "[2, 480000] + script of 442 / 442 / 116 tokens -> probabilities and ranks (BASELINE config 5 shape)"),
                   "weights": "seeded random init at true shapes", "precision": args.precision,
                   "alignment_heads": args.alignment_heads,
                   "kernel_options": {k: L.get_option(k) for k in ("decode_splitk_legacy", "xattn_tc", "decode_fused_ln")},
                   "l2": "per-step working set (weights 6.2 GB + activations) >> 126 MB L2; inputs rotate between 2 pools"},
        "rtf": 1.0 / value, "aligned_words_per_s": n_words_total / (ms_step / 1e3),
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_other": roof_other, "kernels": kernels,
        "cpu_baseline": cpu, "parity_vs_cpu": parity,
        "e2e": {"value": e2e_value, "unit": "audio_s/s", "h2d_bytes_per_step": Wn * N_SAMPLES * 4 * (2 if refine else 1),
                # jumps int32 [N+1] + token probs fp32 [N] per window (+ token/argmax tables and sampler state for decode);
                # refine: probabilities + ranks [2, N] per group
                "d2h_bytes_per_step": int(sum(2 * 2 * 4 * len(g[1]) for g in groups[0])) if refine else
                                      int(Wn * ((args.tokens + 3) * 4 + (args.tokens + 2) * 4)
                                          + (Wn * (2 * args.tokens * 4 + 24 + 4) if args.workload == "transcribe" else 0)),
                "ms_per_step": e2e_s * 1e3, "aligned_words_per_s": n_words_total / e2e_s},
    }
    emit_json(out)


def main():
    args = parse()
    claim_stdout()
    from stable_ts_b200.api import MODEL_DIMS
    dims_tuple = MODEL_DIMS[args.model]
    if args.impl == "reference":
        run_reference(args, dims_tuple)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback); use --impl reference for the CPU arm")
        run_b200(args, dims_tuple)


if __name__ == "__main__":
    main()
