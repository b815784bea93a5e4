"""bench.py -- throughput of the CTC beam-search hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4] [--regime peaky|diffuse]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...        # CPU arm: the unmodified Python reference over a fork pool
                                                # (oracle/_ref; LM workloads: the oracle C++ port)
    python bench.py --dump-outputs DIR ...      # also write the last timed step's results to DIR/*.npy

A "step" is one decode_batch() pass over one batch of synthetic logits.  `value` is frames/s
with the batch already resident in HBM (device pointers handed to the C ABI); `e2e` is the same
call with PINNED HOST buffers, host->device copies and result copies inside the timed region.
Between timed steps L2 is flushed by writing a 512 MiB buffer (inputs of the headline config are
smaller than L2).  Multi-GPU: one rank per GPU, utterances sharded with no data-path
collective (the only collective is the broadcast of the LM blob before timing) -> "weak".
Prints ONE JSON line on rank 0.  Besides the headline (C2) the line carries
  secondary        (1 GPU) the other BASELINE.json configurations -- C3, C4 shape in f32 and f16, the diffuse regime,
                   the beam sweep {10, 50, 500, 2000}, decode_beams_batch -- each with value, e2e, kernel times, a CPU
                   figure and transcript identity against the oracle;
  strong_scaling   (N > 1) ONE 2048-utterance C3 list decoded through sharding.decode_batch_sharded after the NCCL
                   broadcast of the LM blob, checked against rank 0's single-GPU decode of the same list.
"""
import argparse
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "logit frames/sec decoded (batch, beam=100)"

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the headline metric is quoted on
    "c2": dict(kind="char", vocab="B", n_words=20000, lm_order=0, T=1000, batch=256, beam=100, lm={}, hot=0,
               name="Wav2Vec2-base char vocab V=32, T=1000, beam=100, no LM, batch=256 per GPU"),
    "c3": dict(kind="char", vocab="B", n_words=20000, lm_order=3, T=1000, batch=1024, beam=100,
               lm=dict(alpha=0.5, beta=1.0), hot=0,
               name="Wav2Vec2-base V=32, T=1000, beam=100 + synthetic 3-gram (alpha=0.5,beta=1.0), batch=1024 per GPU"),
    # opt-in (--secondary c3_biglm): the C3 shape with a ~10^7 n-gram model, i.e. tables several times the 126 MB L2
    "c3_biglm": dict(kind="char", vocab="B", n_words=420000, lm_order=3, T=1000, batch=1024, beam=100,
                     lm=dict(alpha=0.5, beta=1.0), hot=0,
                     name="C3 shape + synthetic 3-gram over 420k words (~10^7 n-grams: tables several times the L2), batch=1024 per GPU"),
    "c4": dict(kind="bpe", n_words=50000, lm_order=4, T=500, batch=512, beam=100, lm=dict(alpha=0.5, beta=1.0), hot=16,
               name="Conformer-CTC BPE V=1024, T=500, beam=100 + synthetic 4-gram + 16 hotwords, batch=512 per GPU"),
}


def make_workload(spec):
    from tests import synth
    if spec["kind"] == "char":
        return synth.CharWorkload(spec["vocab"], n_words=spec["n_words"], lm_order=spec["lm_order"])
    return synth.BpeWorkload(n_words=spec["n_words"], lm_order=spec["lm_order"])


class ClockSampler:
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md's clocks line), read through NVML
    in this process every 20 ms.  (A polling `nvidia-smi -lms` child process was used first: its driver queries
    delayed the decode calls of the timed loop by up to 2 ms per step.)  Falls back to nvidia-smi without pynvml."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index):
        self.index = index
        self.sm, self.mx, self.reasons = [], [], set()
        self.proc = None
        self.nvml = None
        self._stop = threading.Event()
        self._thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except (ValueError, IndexError):
                    pass
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
            self.nvml = pynvml
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for name, bit in self.BITS:
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def _read(self):
        for line in self.proc.stdout:
            p = [q.strip() for q in line.split(",")]
            if len(p) < 7:
                continue
            try:
                self.sm.append(float(p[0]))
                self.mx.append(float(p[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if val.lower().startswith("active"):
                    self.reasons.add(name)

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self._thread.join(timeout=1.0)
            how = "nvml, 20 ms"
        elif self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            how = "nvidia-smi -lms 100"
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"]}
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "how": how}


def host_cores():
    """CPU threads this process can really use: os.cpu_count() capped by the scheduler affinity and by the
    cgroup CPU quota (the GPU boxes report 128 logical CPUs under a 16-CPU quota; 128 runnable threads on
    16 CPUs' worth of time only thrash -- measured 56 k frames/s against 83 k with 16-32 threads)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as fh:
                parts = fh.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, -(-int(parts[0]) // int(parts[1]))))
            else:
                quota = int(parts[0])
                if quota > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fh:
                        n = min(n, max(1, -(-quota // int(fh.read().split()[0]))))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def workload_objects(spec):
    """-> (workload, build_ctcdecoder keyword arguments, hotword list or None)"""
    wl = make_workload(spec)
    kw = dict(spec["lm"])
    if wl.arpa:
        kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
    hot = wl.hotwords(spec["hot"]) if spec["hot"] else None
    return wl, kw, hot


def config_of(spec, regime, beam, B, V, logits_dtype, world):
    """the `config` object of a JSON line -- the SAME dict for the B200 arm and the reference arm"""
    return {"workload": spec["name"], "regime": regime, "beam_width": beam, "batch_per_gpu": B, "T": spec["T"], "V": V,
            "logits_dtype": logits_dtype, "l2": "flushed between timed steps (512 MiB write)",
            "parallelism": "utterance-sharded x%d" % world}


def port_arm(wl, spec, kw, xs, beam, hot, target_cpu_seconds=20.0, min_utts=0, wall_seconds=0.0, call="decode_batch"):
    """The reference's CPU path restated (oracle/ctc_oracle.cpp, a C++ port -- the reference itself is
    pure Python) on all host cores, over a bounded sample of the same workload: about `target_cpu_seconds` of CPU work,
    or (wall_seconds > 0) about that much wall time on all cores; the list is cycled if the sample needs more
    utterances than were generated."""
    from oracle import oracle as orc
    cores = host_cores()
    ora = orc.OracleDecoder(wl.labels, **kw)
    t0 = time.perf_counter()
    ora.decode_batch(xs[:2], n_threads=2, beam_width=beam, hotwords=hot)
    per_utt = max((time.perf_counter() - t0), 1e-3)  # two utterances on two threads ~ one utterance-time
    if wall_seconds > 0:
        n = int(max(wall_seconds * cores / per_utt, min_utts, cores))
        sample = [xs[i % len(xs)] for i in range(n)]
    else:
        n = int(max(min(len(xs), target_cpu_seconds / per_utt), min(len(xs), max(cores, min_utts))))
        sample = xs[:n]
    t0 = time.perf_counter()
    if call == "decode_beams_batch":        # all beams, prune_history off (decoder.py:801-857); top-1 text for the comparison
        texts = [(b[0][0] if b else "") for b in ora.decode_beams_batch(sample, n_threads=cores, beam_width=beam, hotwords=hot)]
    else:
        texts = ora.decode_batch(sample, n_threads=cores, beam_width=beam, hotwords=hot)
    dt = time.perf_counter() - t0
    frames = sum(x.shape[0] for x in sample)
    return {"value": frames / dt, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": "%d utterances x T=%d of the same workload, oracle C++ port of the reference's Python loop, "
                      "%d threads, %.1f s" % (n, spec["T"], cores, dt)}, texts, n


REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def pyref_available(spec):
    """The unmodified reference (pip-installed into oracle/_ref by build(), see oracle.install_reference)
    can be timed for workloads without a language model: its only missing hard dependency is then pygtrie's import,
    served by the stand-in under oracle/refshim.  LM workloads would run on the pure-Python kenlm stand-in, which
    would handicap the reference -- they are timed on the C++ port instead."""
    return spec["lm_order"] == 0 and os.path.isdir(os.path.join(REF_DIR, "pyctcdecode"))


class PyRef:
    """`with multiprocessing.get_context('fork').Pool(n) as pool: decoder.decode_batch(pool, logits_list, ...)`
    (reference README.md:82-85, decoder.py:895-945); pool start-up and decoder construction outside the timing."""

    def __init__(self, labels, cores):
        import logging
        import multiprocessing as mp
        for p in (os.path.join(ROOT, "oracle", "refshim"), REF_DIR):
            if p not in sys.path:
                sys.path.insert(0, p)
        logging.disable(logging.CRITICAL)
        from pyctcdecode import build_ctcdecoder as ref_build
        import pyctcdecode as ref_pkg
        assert os.path.realpath(ref_pkg.__file__).startswith(os.path.realpath(REF_DIR)), ref_pkg.__file__
        self.dec = ref_build(labels)
        self.cores = cores
        self.pool = mp.get_context("fork").Pool(cores)

    def run(self, sample, beam, hot):
        t0 = time.perf_counter()
        texts = self.dec.decode_batch(self.pool, sample, beam_width=beam, hotwords=hot)
        return time.perf_counter() - t0, texts

    def close(self):
        self.pool.close()
        self.pool.join()


def reference_main(args, spec, B, beam):
    """--impl reference: CPU only.  Each step is a bounded sample (>= 4 utterances per thread, >= ~2 s) of the
    configured workload; the whole run is sized to about two minutes."""
    wl, kw, hot = workload_objects(spec)
    cores = host_cores()
    T = spec["T"]
    use_py = pyref_available(spec) and not args.ref_port
    n_steps = max(1, args.warmup + args.steps)
    per_step = args.ref_seconds if args.ref_seconds > 0 else min(8.0, max(2.2, 120.0 / n_steps))
    n0 = 4 * cores
    xs = wl.batch(1, n0, T, args.regime)
    if args.logits_dtype == "f16":
        xs = [x.astype(np.float16).astype(np.float32) for x in xs]
    texts = None
    if use_py:
        ref = PyRef(wl.labels, cores)
        dt0, _ = ref.run(xs[:cores], beam, hot)                     # pool warm-up + calibration: one utterance per process
        n = int(max(n0, min(64 * cores, per_step / max(dt0, 1e-3) * cores)))
        if n > len(xs):
            xs = wl.batch(1, n, T, args.regime)
        sample = xs[:n]
        vals = []
        for i in range(n_steps):
            dt, texts = ref.run(sample, beam, hot)
            if i >= args.warmup:
                vals.append(n * T / dt)
        ref.close()
        kind = "reference"
        what = ("%d utterances x T=%d of the same workload, the UNMODIFIED Python reference (oracle/_ref, pyctcdecode 0.6.0) "
                "through decode_batch over a fork Pool(%d), %.1f s per step" % (n, T, cores, n * T / vals[-1]))
    else:
        vals, info = [], None
        if len(xs) < min(B, 16 * cores):
            xs = wl.batch(1, min(B, 16 * cores), T, args.regime)
            if args.logits_dtype == "f16":
                xs = [x.astype(np.float16).astype(np.float32) for x in xs]
        for i in range(n_steps):
            info, texts, n = port_arm(wl, spec, kw, xs, beam, hot, min_utts=n0, wall_seconds=per_step)
            if i >= args.warmup:
                vals.append(info["value"])
        kind = "port"
        what = info["sample"] + ("" if pyref_available(spec) else
                                 "; the Python reference is not timed for LM workloads (kenlm is not installed: its stand-in is pure Python)")
    v = statistics.mean(vals)
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": config_of(spec, args.regime, beam, B, wl.V, args.logits_dtype, max(1, args.gpus)),
           "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": kind, "sample": what},
           "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.emit_texts:
        out["texts"] = list(texts)
    _emit(out)
    return 0


def pyref_subprocess(args_workload, regime, beam, seconds):
    """cpu_baseline of the B200 arm, `kind: reference`: the reference arm in a child process (the fork pool must not
    be forked from a process that holds a CUDA context and helper threads)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0", "--workload",
           args_workload, "--regime", regime, "--beam", str(beam), "--emit-texts", "--ref-seconds", str(seconds)]
    try:
        run = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=300)
        line = [ln for ln in run.stdout.splitlines() if ln.startswith("{")][-1]
        obj = json.loads(line)
        return obj["cpu_baseline"], obj.get("texts", [])
    except Exception as exc:  # the figure is a reported baseline, not a gate: say why it is missing
        return {"value": None, "unit": "frames/s", "cores": host_cores(), "kind": "reference", "sample": "failed: %r" % (exc,)}, []


class Stepper:
    """one decoder + one batch resident in pinned host memory and in HBM; times the public call"""

    def __init__(self, torch, dist, dec, xs, beam, hot, logits_dtype, call="decode_batch"):
        self.torch, self.dist, self.dec, self.beam, self.hot, self.call = torch, dist, dec, beam, hot, call
        if logits_dtype == "f16":                             # the model emitted half precision: both arms see those values
            xs16 = [x.astype(np.float16) for x in xs]
            self.xs = [x.astype(np.float32) for x in xs16]
            self.host = torch.from_numpy(np.stack(xs16)).pin_memory()
        else:
            self.xs = xs
            self.host = torch.from_numpy(np.stack(xs)).pin_memory()
        self.dev = self.host.cuda(non_blocking=False)

    def step_dev(self):
        return getattr(self.dec, self.call)(None, self.dev, beam_width=self.beam, hotwords=self.hot)

    def step_host(self):
        return getattr(self.dec, self.call)(None, self.host, beam_width=self.beam, hotwords=self.hot)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, flush):
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        total, tms, out = 0.0, [], None
        for _ in range(steps):
            flush.fill_(1)                       # L2 flush, outside the timed bracket
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            total += time.perf_counter() - t0
            tms.append(self.dec.last_timings())
        self.barrier()
        if self.dist is not None:
            t = torch.tensor([total], dtype=torch.float64, device="cuda")
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            total = float(t.item())
        return total, tms, out


DUMP_LIMIT = 64_000_000      # bytes of .npy files (64 MB)


def _codepoints(texts):
    """strings -> [N, longest] float32 Unicode code points (exact: every code point is below 2^24), padded with -1"""
    arr = np.full((len(texts), max([len(t) for t in texts], default=0)), -1.0, np.float32)
    for i, t in enumerate(texts):
        arr[i, :len(t)] = [ord(c) for c in t]
    return arr


def output_arrays(call, out, keep):
    """What `call` returned for the utterances `keep`, one row per transcript: decode_batch -> `text`;
    decode_beams_batch -> every beam's `text`, `logit_score`, `lm_score` and `word_frames` (start and end frame of each
    word, padded with -1).  `utterance` is the batch index of each row."""
    if call == "decode_batch":
        return {"utterance": keep.astype(np.float64), "text": _codepoints([out[i] for i in keep])}
    beams = [(i, b) for i in keep for b in out[i]]
    frames = np.full((len(beams), max([len(b.text_frames) for _, b in beams], default=0), 2), -1.0, np.float32)
    for r, (_, b) in enumerate(beams):
        for w, (_, span) in enumerate(b.text_frames):
            frames[r, w] = span
    return {"utterance": np.array([i for i, _ in beams], np.float64), "text": _codepoints([b.text for _, b in beams]),
            "logit_score": np.array([b.logit_score for _, b in beams], np.float64),
            "lm_score": np.array([b.lm_score for _, b in beams], np.float64), "word_frames": frames}


def _npy_files(arrays):
    """{name: the bytes of name.npy, header included}"""
    files = {}
    for name, arr in arrays.items():
        buf = io.BytesIO()
        np.save(buf, arr)
        files[name] = buf.getvalue()
    return files


def dump_outputs(path, call, out):
    """DIR/<name>.npy of output_arrays() for the whole batch or, above DUMP_LIMIT bytes of files, for a fixed sample
    of it: a prefix of a seeded permutation, halved until the files fit"""
    keep = np.arange(len(out))
    perm = np.random.default_rng(0).permutation(len(out))
    files = _npy_files(output_arrays(call, out, keep))
    while sum(len(b) for b in files.values()) > DUMP_LIMIT and len(keep) > 1:
        keep = np.sort(perm[:len(keep) // 2])
        files = _npy_files(output_arrays(call, out, keep))
    os.makedirs(path, exist_ok=True)
    for name, data in files.items():
        with open(os.path.join(path, name + ".npy"), "wb") as fh:
            fh.write(data)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh)
    except OSError:
        return {}


def secondary_entry(torch, pkg, flush, name, spec, regime, beam, logits_dtype, call, steps, warmup, batch=0, cpu_seconds=4.0):
    """one more BASELINE.json configuration on one GPU: value / e2e / kernel times / CPU figure / transcript identity"""
    t_start = time.perf_counter()
    wl, kw, hot = workload_objects(spec)
    t_gen = time.perf_counter() - t_start
    B, T = batch or spec["batch"], spec["T"]
    t_b = time.perf_counter()
    dec = pkg.build_ctcdecoder(wl.labels, device=torch.cuda.current_device(), **kw)
    t_build = time.perf_counter() - t_b
    st = Stepper(torch, None, dec, wl.batch(1, B, T, regime), beam, hot, logits_dtype, call)
    total, tms, out = st.timed(st.step_dev, steps, warmup, flush)
    e2e_total, e2e_tms, out_e2e = st.timed(st.step_host, steps, warmup, flush)
    same = out == out_e2e
    frames = B * T
    peak = float(load_peaks().get("hbm_gbs", 6650.0))
    esz = 2 if logits_dtype == "f16" else 4
    ms_beam = statistics.mean(t["ms_beam"] for t in tms)
    ms_prep = statistics.mean(t["ms_prepare"] for t in tms)
    texts = out if call == "decode_batch" else [beams[0].text if beams else "" for beams in out]
    info, cpu_texts, n = port_arm(wl, spec, kw, st.xs, beam, hot, target_cpu_seconds=cpu_seconds, call=call)
    ent = {"name": name, "config": config_of(spec, regime, beam, B, wl.V, logits_dtype, 1), "call": call,
           "value": frames * steps / total, "unit": "frames/s", "ms_per_step": 1e3 * total / steps, "steps": steps, "warmup": warmup,
           "e2e": {"value": frames * steps / e2e_total, "unit": "frames/s", "ms_per_step": 1e3 * e2e_total / steps,
                   "h2d_bytes_per_step": int(e2e_tms[-1]["h2d_bytes"]), "d2h_bytes_per_step": int(e2e_tms[-1]["d2h_bytes"])},
           "beam_kernel_ms": ms_beam, "prepare_ms": ms_prep,
           "roofline_frac": frames * wl.V * esz / (ms_beam * 1e-3) / 1e9 / peak if ms_beam > 0 else None,
           "roofline_prepare_frac": frames * wl.V * esz / (ms_prep * 1e-3) / 1e9 / peak if ms_prep > 0 else None,
           "kernel_variant": tms[-1]["kernel_variant"], "resident_ctas": tms[-1]["cta_slots"], "cap_candidates": tms[-1]["cap_candidates"],
           "inplace_frames_per_step": tms[-1]["inplace_frames"], "sorted_frames_per_step": tms[-1]["sorted_frames"],
           "oversize_frames_per_step": tms[-1]["oversize_frames"],
           "gpu_launches": int(sum(t["launches"] for t in tms)),
           "host_equals_device_input": bool(same),
           "cpu_baseline": info,
           "transcripts_identical_to_oracle": "%d/%d" % (sum(a == b for a, b in zip(cpu_texts, texts[:n])), n),
           "wall_s": None}
    if spec["lm_order"]:
        try:        # how big the flattened model is (what one NCCL broadcast ships) and how long building it took
            with open(wl.arpa, encoding="utf-8") as fh:
                counts = [int(ln.split("=")[1]) for ln in (fh.readline() for _ in range(12)) if ln.startswith("ngram ")]
            ent["lm"] = {"ngrams": counts, "arpa_mb": round(os.path.getsize(wl.arpa) / 1e6, 1),
                         "blob_mb": round(dec._language_model._kenlm_model.blob()[1] / 1e6, 1),
                         "build_decoder_s": round(t_build, 2), "generate_arpa_s": round(t_gen, 1)}
        except Exception as exc:
            ent["lm"] = {"error": repr(exc)}
    del st, dec
    torch.cuda.empty_cache()
    ent["wall_s"] = round(time.perf_counter() - t_start, 1)
    return ent


def _stream_run(dec, xs, chunk, beam):
    """get_starting_state / partial_decode_beams(_batch) over `xs` in chunks of `chunk` frames (reference decoder.py:669-728,
    the streaming form of the same frame loop) -> (seconds per call, final top-1 texts)"""
    n, T = len(xs), len(xs[0])
    starts = [dec.get_starting_state() for _ in range(n)]
    beams, caches, pcaches = [s[0] for s in starts], [s[1] for s in starts], [s[2] for s in starts]
    lat = []
    for t0 in range(0, T, chunk):
        t1 = min(T, t0 + chunk)
        t = time.perf_counter()
        if n == 1 or not hasattr(dec, "partial_decode_beams_batch"):
            beams = [dec.partial_decode_beams(xs[i][t0:t1], caches[i], pcaches[i], beams[i], t0, beam_width=beam, is_end=t1 >= T)
                     for i in range(n)]
        else:
            beams = dec.partial_decode_beams_batch([x[t0:t1] for x in xs], caches, beams, [t0] * n, beam_width=beam, is_end=t1 >= T)
        lat.append(time.perf_counter() - t)
    return lat, [b[0].text if b else "" for b in beams]


def streaming_entry(torch, pkg, name, spec, n_streams, chunk=50, beam=100):
    """Per-call latency of the streaming form of the path: `n_streams` independent streams advance by `chunk` frames per
    call (host logits, beams carried as LMBeam lists exactly like in the reference).  `final_text_equals_one_shot` is
    informational: every chunk ends with _finalize_beams (sort, trim, prune), so the reference's own streaming result
    differs from its one-shot decode on a few percent of the utterances too; parity of the streaming path is what the
    22 reference-generated streaming goldens and `cpu_baseline.final_text_equals_b200` check.  CPU figure: the unmodified Python reference's own partial_decode_beams on
    one stream (workloads without a language model, when oracle/_ref is present)."""
    t_start = time.perf_counter()
    wl, kw, _ = workload_objects(spec)
    T = spec["T"]
    dec = pkg.build_ctcdecoder(wl.labels, device=torch.cuda.current_device(), **kw)
    xs = wl.batch(1, n_streams, T, "peaky")
    one_shot = dec.decode_batch(None, xs, beam_width=beam)
    _stream_run(dec, xs, chunk, beam)                                    # warm-up pass
    lat, texts = _stream_run(dec, xs, chunk, beam)
    ent = {"name": name, "call": "partial_decode_beams" + ("_batch" if n_streams > 1 else ""), "streams": n_streams,
           "chunk_frames": chunk, "beam": beam, "config": config_of(spec, "peaky", beam, n_streams, wl.V, "f32", 1),
           "ms_per_call": {"median": 1e3 * statistics.median(lat), "first": 1e3 * lat[0], "last": 1e3 * lat[-1], "max": 1e3 * max(lat)},
           "value": n_streams * T / sum(lat), "unit": "frames/s", "calls": len(lat),
           "final_text_equals_one_shot": "%d/%d" % (sum(a == b for a, b in zip(texts, one_shot)), n_streams),
           "cpu_baseline": None}
    if pyref_available(spec):
        try:
            ref = PyRef(wl.labels, 1)
            rlat, rtexts = _stream_run(ref.dec, xs[:1], chunk, beam)
            ref.close()
            ent["cpu_baseline"] = {"kind": "reference", "cores": 1, "streams": 1, "ms_per_call_median": 1e3 * statistics.median(rlat),
                                   "value": T / sum(rlat), "unit": "frames/s",
                                   "final_text_equals_b200": bool(rtexts[0] == texts[0]),
                                   "sample": "the unmodified Python reference's partial_decode_beams, one stream, same chunks"}
        except Exception as exc:
            ent["cpu_baseline"] = {"kind": "reference", "value": None, "sample": "failed: %r" % (exc,)}
    del dec
    ent["wall_s"] = round(time.perf_counter() - t_start, 1)
    return ent


def strong_scaling(torch, dist, pkg, sharding, flush, rank, world, local_rank, steps, n_utts=2048):
    """The north_star multi-GPU path: every rank holds the SAME list of utterances (C3: 3-gram LM), the decoder is
    built with ONE NCCL broadcast of the flattened LM, decode_batch_sharded splits the list over the ranks (no
    data-path collective), the transcripts are gathered, and rank 0 checks them against its own single-GPU decode."""
    spec = dict(WORKLOADS["c3"])
    wl, kw, hot = workload_objects(spec)
    T, beam = spec["T"], spec["beam"]
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    dec = sharding.build_ctcdecoder_broadcast(wl.labels, device=local_rank, **kw)
    torch.cuda.synchronize()
    dist.barrier()
    build_s = time.perf_counter() - t0
    bc = dict(sharding.last_broadcast)
    big = np.stack(wl.batch(1, n_utts, T, "peaky"))          # one allocation: a rank's utterances are adjacent where possible
    xs = [big[i] for i in range(n_utts)]

    def sharded():
        return sharding.decode_batch_sharded(dec, xs, beam_width=beam, hotwords=hot)

    def timed(fn, n):
        tot, out = 0.0, None
        for _ in range(n):
            flush.fill_(1)
            torch.cuda.synchronize()
            dist.barrier()
            t1 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            tot += time.perf_counter() - t1
        t = torch.tensor([tot], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out

    sharded()
    sharded()                                               # warm-up: buffers, kernel variant hint
    t_sh, texts = timed(sharded, steps)
    # the same list on ONE GPU through the same public call (rank 0 decodes, the others wait at the barrier)
    single_texts, t_single = None, None
    if rank == 0:
        dec.decode_batch(None, xs, beam_width=beam, hotwords=hot)
        dec.decode_batch(None, xs, beam_width=beam, hotwords=hot)
    tot = 0.0
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        dist.barrier()
        if rank == 0:
            t1 = time.perf_counter()
            single_texts = dec.decode_batch(None, xs, beam_width=beam, hotwords=hot)
            torch.cuda.synchronize()
            tot += time.perf_counter() - t1
    dist.barrier()
    if rank != 0:
        return None
    t_single = tot
    frames = n_utts * T
    return {"workload": spec["name"].replace("batch=1024 per GPU", "ONE list of %d utterances" % n_utts), "n_utts": n_utts, "T": T,
            "beam_width": beam, "path": "sharding.build_ctcdecoder_broadcast -> sharding.decode_batch_sharded (host numpy in, texts out, all_gather_object of the transcripts inside the timed region)",
            "lm_broadcast": {"bytes": bc.get("bytes"), "ms": bc.get("ms"), "gb_per_s": bc.get("gb_per_s"), "backend": bc.get("backend"),
                             "build_decoder_s_incl_arpa_parse_on_rank0": build_s},
            "sharded": {"value": frames * steps / t_sh, "unit": "frames/s", "ms_per_step": 1e3 * t_sh / steps, "n_gpus": world},
            "single_gpu_same_list": {"value": frames * steps / t_single, "unit": "frames/s", "ms_per_step": 1e3 * t_single / steps},
            "speedup_vs_one_gpu": t_single / t_sh,
            "sharded_equals_single": bool(texts == single_texts), "steps": steps,
            "limit": "per-rank host work (Python list handling, per-utterance H2D copies) and the latency of one resident wave: "
                     "%d utterances per GPU are %s the resident set" % (n_utts // world, "within" if n_utts // world <= 592 else "above")}


_REAL_STDOUT = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line: everything else a library writes to fd 1 (NCCL's version banner,
    nvcc output of a rebuild, ...) is sent to stderr for the lifetime of the process."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(obj) + "\n").encode())


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--regime", default="peaky", choices=["peaky", "diffuse"])
    ap.add_argument("--batch", type=int, default=0, help="utterances per GPU (default: the workload's)")
    ap.add_argument("--beam", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary configurations (1 GPU) / the strong-scaling section (N > 1)")
    ap.add_argument("--secondary", default="", help="comma separated subset of: c3,c4,c4_f16,diffuse,beam10,beam50,beam500,beam2000,beams_batch,stream1,stream64,stream64_lm; opt-in: c3_biglm")
    ap.add_argument("--secondary-steps", type=int, default=5)
    ap.add_argument("--call", default="decode_batch", choices=["decode_batch", "decode_beams_batch"])
    ap.add_argument("--logits-dtype", default="f32", choices=["f32", "f16"],
                    help="dtype of the model output handed to decode_batch (f16: 2-byte elements over PCIe, widened on the device)")
    ap.add_argument("--ref-port", action="store_true", help="reference arm: time the oracle C++ port even where the Python reference can run")
    ap.add_argument("--ref-seconds", type=float, default=0.0, help="reference arm: target seconds of one step (default: sized from --steps)")
    ap.add_argument("--emit-texts", action="store_true", help="reference arm: add the transcripts of the last step to the JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step of the headline call returned (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    spec = dict(WORKLOADS[args.workload])
    B = args.batch or spec["batch"]
    beam = args.beam or spec["beam"]
    T = spec["T"]

    # ------------------------------------------------------------------------------------
    # reference arm: CPU only, rank 0 only
    # ------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_main(args, spec, B, beam)

    # ------------------------------------------------------------------------------------
    # B200 arm
    # ------------------------------------------------------------------------------------
    import torch

    import __graft_entry__ as graft
    if not os.path.exists(os.path.join(ROOT, "pyctcdecode_b200", "libb200ctc.so")) or rank == 0:
        graft.build()
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    else:
        dist = None
        torch.cuda.set_device(local_rank)
    import pyctcdecode_b200 as pkg
    from pyctcdecode_b200 import sharding
    if os.environ.get("B200CTC_PROFILING_LIB"):   # opt-in phase-clock build (profiles/README.md), never the default
        from pyctcdecode_b200 import _lib
        _lib.use_library(os.environ["B200CTC_PROFILING_LIB"])

    wl, kw, hot = workload_objects(spec)
    lm_broadcast = None
    if world > 1 and wl.arpa:
        # rank 0 parses the ARPA file; every other rank receives the flattened LM over NCCL
        dec = sharding.build_ctcdecoder_broadcast(wl.labels, device=local_rank, **kw)
        lm_broadcast = dict(sharding.last_broadcast)
    else:
        dec = pkg.build_ctcdecoder(wl.labels, device=local_rank, **kw)

    xs = wl.batch(1 + rank * 100_000, B, T, args.regime)   # every rank its own utterances (weak scaling)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    st = Stepper(torch, dist, dec, xs, beam, hot, args.logits_dtype, args.call)
    xs = st.xs
    frames_per_step = B * T

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total, tms, texts = st.timed(st.step_dev, args.steps, args.warmup, flush)
    clocks = sampler.stop() if rank == 0 else None
    e2e_total, e2e_tms, texts_e2e = st.timed(st.step_host, args.steps, args.warmup, flush)   # the same W warm-up steps as the device-resident arm
    assert texts == texts_e2e
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, args.call, texts)
    if args.call != "decode_batch":
        texts = [beams[0].text if beams else "" for beams in texts]

    strong = None
    if world > 1 and not args.no_secondary:
        del st
        torch.cuda.empty_cache()
        strong = strong_scaling(torch, dist, pkg, sharding, flush, rank, world, local_rank, steps=max(2, min(5, args.steps)))

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    value = world * frames_per_step * args.steps / total
    ms_beam = statistics.mean(t["ms_beam"] for t in tms)
    ms_prep = statistics.mean(t["ms_prepare"] for t in tms)
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    esz = 2 if args.logits_dtype == "f16" else 4      # algorithmic bytes per logit: the dtype the rows arrive in
    alg_bytes = frames_per_step * wl.V * esz
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            traffic = json.load(fh).get(args.workload, {}).get("beam_kernel_dram_bytes")
    except OSError:
        pass
    ach = alg_bytes / (ms_beam * 1e-3) / 1e9
    ach_prep = alg_bytes / (ms_prep * 1e-3) / 1e9 if ms_prep > 0 else None
    out = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": config_of(spec, args.regime, beam, B, wl.V, args.logits_dtype, world),
        "roofline": {"bound": "hbm", "kernel": "b2c_beam_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": traffic, "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)",
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": ms_beam,
                     "note": "the beam kernel is a T-step serial chain per utterance (latency bound); the streaming stage is reported under roofline_prepare"},
        "roofline_prepare": {"bound": "hbm", "kernel": "b2c_prepare_kernel", "achieved": ach_prep, "peak": peak, "unit": "GB/s",
                             "frac": (ach_prep / peak) if ach_prep else None, "kernel_ms": ms_prep},
        "e2e": {"value": world * frames_per_step * args.steps / e2e_total, "unit": "frames/s",
                "h2d_bytes_per_step": int(e2e_tms[-1]["h2d_bytes"]), "d2h_bytes_per_step": int(e2e_tms[-1]["d2h_bytes"]),
                "ms_per_step": 1e3 * e2e_total / args.steps},
        "gpu_launches": int(sum(t["launches"] for t in tms)),
        "device_ms_per_step": statistics.mean(t["ms_total"] for t in tms),
        "beam_kernel_config": {"cap_candidates": tms[-1]["cap_candidates"], "cta_threads": tms[-1]["cta_threads"],
                               "resident_ctas": tms[-1]["cta_slots"], "oversize_frames_per_step": tms[-1]["oversize_frames"],
                               "kernel_variant": tms[-1]["kernel_variant"],
                               "planned_from_previous_call_statistics": int(tms[-1].get("hinted", 0)),
                               "inplace_single_token_frames_per_step": tms[-1]["inplace_frames"],
                               "sorted_no_merge_frames_per_step": tms[-1]["sorted_frames"],
                               "frames_over_128_256_512_1024_2048_4096_total": tms[-1]["cand_hist"]},
        "clocks": clocks,
    }
    if lm_broadcast:
        out["lm_broadcast"] = lm_broadcast
    if strong is not None:
        out["strong_scaling"] = strong
    if world == 1 and not args.no_cpu_baseline:
        # the reference's own CPU path: the unmodified Python package over a fork pool where it can run (no LM), in a
        # child process; next to it the C++ port of the same loop, which also provides the transcripts to compare with
        port, cpu_texts, n = port_arm(wl, spec, kw, xs, beam, hot, target_cpu_seconds=10.0 if pyref_available(spec) else 20.0)
        if pyref_available(spec) and args.logits_dtype == "f32":
            ref_info, ref_texts = pyref_subprocess(args.workload, args.regime, beam, 6.0)
            out["cpu_baseline"] = dict(ref_info, port=port)
            m = min(len(ref_texts), len(texts))
            out["transcripts_identical_to_reference"] = "%d/%d" % (sum(a == b for a, b in zip(ref_texts[:m], texts[:m])), m)
        else:
            out["cpu_baseline"] = port
        out["transcripts_identical_to_oracle"] = "%d/%d" % (sum(a == b for a, b in zip(cpu_texts, texts[:n])), n)
        # "WER parity" of the metric: both systems against the word sequence the synthetic alignment spells
        from tests import synth
        err = {"b200": [0, 0], "cpu_port": [0, 0]}
        for i in range(n):
            truth = wl.truth(1 + i, T)
            for key, hyp in (("b200", texts[i]), ("cpu_port", cpu_texts[i])):
                e, m = synth.word_errors(truth, hyp)
                err[key][0] += e
                err[key][1] += m
        out["wer"] = {k: (v[0] / v[1] if v[1] else None) for k, v in err.items()}
        out["wer"].update(utterances=n, against="ground-truth word sequence of the synthetic alignment (noisy logits, so not 0)")
    if world == 1 and not args.no_secondary and args.workload == "c2" and args.regime == "peaky" and not args.batch and not args.beam:
        del st, dec
        torch.cuda.empty_cache()
        S, W = max(1, args.secondary_steps), 3
        plan = [("c3", WORKLOADS["c3"], "peaky", 100, "f32", "decode_batch", 0),
                ("c4", WORKLOADS["c4"], "peaky", 100, "f32", "decode_batch", 0),
                ("c4_f16", WORKLOADS["c4"], "peaky", 100, "f16", "decode_batch", 0),
                ("diffuse", WORKLOADS["c2"], "diffuse", 100, "f32", "decode_batch", 0),
                ("beam10", WORKLOADS["c2"], "peaky", 10, "f32", "decode_batch", 0),
                ("beam50", WORKLOADS["c2"], "peaky", 50, "f32", "decode_batch", 0),
                ("beam500", WORKLOADS["c2"], "peaky", 500, "f32", "decode_batch", 0),
                ("beam2000", WORKLOADS["c2"], "peaky", 2000, "f32", "decode_batch", 0),
                ("beams_batch", WORKLOADS["c2"], "peaky", 100, "f32", "decode_beams_batch", 0)]
        want = [w for w in args.secondary.split(",") if w]
        if "c3_biglm" in want:     # opt-in only: generating and loading the 10^7 n-gram model takes minutes
            plan.append(("c3_biglm", WORKLOADS["c3_biglm"], "peaky", 100, "f32", "decode_batch", 0))
        out["secondary"] = []
        for name, sp, regime, bm, dt, call, bsz in plan:
            if want and name not in want:
                continue
            try:
                out["secondary"].append(secondary_entry(torch, pkg, flush, name, dict(sp), regime, bm, dt, call, S, W, bsz))
            except Exception as exc:  # one configuration must not take the headline down with it
                out["secondary"].append({"name": name, "error": repr(exc)})
        for name, sp, n_streams in (("stream1", WORKLOADS["c2"], 1), ("stream64", WORKLOADS["c2"], 64), ("stream64_lm", WORKLOADS["c3"], 64)):
            if want and name not in want:
                continue
            try:
                out["secondary"].append(streaming_entry(torch, pkg, name, dict(sp), n_streams))
            except Exception as exc:
                out["secondary"].append({"name": name, "error": repr(exc)})
    _emit(out)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
