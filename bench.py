#!/usr/bin/env python
"""bench.py -- benchmarks of the native GridLLM worker on B200 (BASELINE.json configs 2-5; config 2 is the headline default).

  --workload config2 (default)  Llama-3-8B q4_K_M, greedy, 512-in / 128-out, batch 1 per GPU           generated tokens/s
  --workload config3            the same model, 32 concurrent streamed chat requests per GPU (256 on 8)   generated tokens/s
                                through NativeWorker x scheduler rules, decoded together (continuous batching)
  --workload config4            Llama-3-8B bf16, batched prefill, 32 sequences x 2048 tokens              prompt tokens/s
  --workload config5            Mistral-7B q8_0 embeddings, 256-token documents (10 000 docs = 8 x 1 250)   documents/s

A "step" is one pass of the workload over one batch of synthetic input on one GPU (config2: one request; config3: 32 requests;
config4: 32 x 2048 prompt tokens; config5: 1 250 documents / 8 = the share of one of 8 workers scaled to --docs).
  value        whole-job throughput, DEVICE-timed (cudaEvent inside the library), inputs resident, max over ranks
  e2e          the same metric through the reference-facing call with HOST buffers (C ABI / NativeWorker), wall clock
  roofline     dominant kernel: algorithmic bytes (or flops) / measured device time vs the measured peak (MEASURED_PEAKS.json)
  cpu_baseline the C restatement of the reference's CPU path (oracle/c/llama_cpu.c: ggml-style int8-activation integer dots,
               batched prompt pass) on the host cores, a bounded sample of the same workload (rank 0, N = 1 only; the 8B-shape
               parity pre-flight of config2 likewise runs on the N = 1 line)
`--impl reference` times only that CPU restatement, really -- model loaded once, thread count chosen once, every step a
measured bounded sample -- and prints the same metric / unit / config as the native arm.  (The reference's own engine, an
un-vendored Ollama/llama.cpp behind HTTP, cannot be installed here: no node / ollama / network -- DESIGN.md section 2.)

Launch: python bench.py [--gpus N --steps K --warmup W]; N>1 via torchrun (one rank per GPU, no data-path collective: requests
are independent, SURVEY.md section 8e) -- weak scaling.  `--workload config3 --gpus N` WITHOUT torchrun runs N engines in ONE
process behind one scheduler (the north_star's in-process shape).
`--dump-outputs DIR` writes what the last timed step returned (config2 / config4: token ids and logprobs; config5: the embeddings)
as DIR/<name>.npy: the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import asyncio
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: nothing is written beside the sources

N_PROMPT, N_GEN = 512, 128
MODEL_DIR = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
MODELS = {
    "llama3_8b_q4km": ("gridllm_llama3_8b_q4km_synth_seed1234.gguf", "LLAMA3_8B", "q4_k_m", 4912898048),
    "llama3_8b_bf16": ("gridllm_llama3_8b_bf16_synth_seed1234.gguf", "LLAMA3_8B", "bf16", 16060000000),
    "mistral7b_q8": ("gridllm_mistral7b_q8_0_synth_seed1234.gguf", "MISTRAL_7B", "q8_0", 7600000000),
}
# one metric string per workload, shared by BOTH arms (the driver divides the two lines only when they agree)
METRICS = {
    "config2": ("generated tokens/sec (aggregate, device-timed), Llama-3-8B q4_K_M, 512-in/128-out, greedy, batch 1 per GPU", "tokens/s"),
    "config3": ("generated tokens/sec (aggregate, device-timed), Llama-3-8B q4_K_M, 512-in/128-out, greedy, 32 concurrent streamed chat "
                "requests per GPU through the scheduler rules", "tokens/s"),
    "config4": ("prompt tokens/sec (aggregate, device-timed), Llama-3-8B bf16 batched prefill, 32 sequences x 2048 tokens per GPU", "tokens/s"),
    "config5": ("documents/sec (aggregate, device-timed), Mistral-7B q8_0 embeddings, 256-token documents", "docs/s"),
}
WORKLOAD_MODEL = {"config2": "llama3_8b_q4km", "config3": "llama3_8b_q4km", "config4": "llama3_8b_bf16", "config5": "mistral7b_q8"}
DOC_TOKENS = 256


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def model_path(key: str) -> str:
    return os.path.join(MODEL_DIR, MODELS[key][0])


def build_model_once(key: str, rank: int, barrier) -> str:
    """Synthetic GGUF (random well-formed blocks, SURVEY.md section 8d).  Rank 0 writes it once per box."""
    from oracle import gguf_synth as S
    fname, shape, recipe, expect = MODELS[key]
    path = os.path.join(MODEL_DIR, fname)
    if rank == 0:
        ok = os.path.exists(path) and os.path.getsize(path) > expect
        if not ok:
            t0 = time.time()
            tmp = path + f".tmp{os.getpid()}"
            S.build_model(tmp, getattr(S, shape), recipe, seed=1234, mode="random", with_vocab=False)
            os.replace(tmp, path)
            log(f"[bench] built {path} in {time.time() - t0:.1f}s")
    barrier()
    return path


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, device: int):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# =====================================================================================================================
# CPU restatement (reference arm and cpu_baseline): loaded once, threads chosen once, every call really timed
# =====================================================================================================================
def physical_cores() -> int:
    """distinct (socket, core) pairs among the CPUs this process may run on"""
    try:
        allowed = os.sched_getaffinity(0)
        cores, cpu, phys = set(), None, None
        for line in open("/proc/cpuinfo"):
            if line.startswith("processor"):
                cpu = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = int(line.split(":")[1])
            elif line.startswith("core id") and cpu in allowed:
                cores.add((phys, int(line.split(":")[1])))
        return max(1, len(cores)) if cores else max(1, len(allowed))
    except Exception:
        return max(1, os.cpu_count() or 1)


class CpuRestatement:
    """oracle/c/llama_cpu.c on this machine's host cores.  Prefers a -march=native build made at run time in a temporary
    directory; falls back to the portable library build() made (oracle/_ref/liboracle_cpu.so)."""

    def __init__(self, path: str, n_ctx: int):
        src = os.path.join(ROOT, "oracle", "c", "llama_cpu.c")
        so = os.path.join(ROOT, "oracle", "_ref", "liboracle_cpu.so")
        lib = None
        try:
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            with tempfile.TemporaryDirectory(prefix="gridllm_bench_") as d:
                native = os.path.join(d, "liboracle_cpu_native.so")
                subprocess.check_call([cc, "-O3", "-march=native", "-fopenmp", "-fPIC", "-shared", "-o", native, src, "-lm"],
                                      stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=180)
                lib = C.CDLL(native)            # stays mapped after the directory is removed
            so = native
        except Exception:
            lib = None
        if lib is None:
            lib = C.CDLL(so)
        lib.oc_load.restype = C.c_void_p
        lib.oc_load.argtypes = [C.c_char_p, C.c_int]
        lib.oc_step.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        lib.oc_prefill.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        lib.oc_fill_kv.argtypes = [C.c_void_p, C.c_int, C.c_uint]
        lib.oc_reset.argtypes = [C.c_void_p]
        lib.oc_set_threads.argtypes = [C.c_int]
        lib.oc_free.argtypes = [C.c_void_p]
        self.lib, self.so = lib, os.path.basename(so)
        t0 = time.time()
        self.h = lib.oc_load(path.encode(), n_ctx)
        if not self.h:
            raise RuntimeError("C restatement could not load the model")
        info = (C.c_int * 16)()
        lib.oc_info.argtypes = [C.c_void_p, C.c_void_p]
        lib.oc_info(self.h, info)
        self.n_vocab = int(info[6]) if int(info[6]) > 0 else 128256
        self.logits = np.zeros(max(self.n_vocab, 200000), np.float32)
        self.lp = self.logits.ctypes.data_as(C.c_void_p)
        lib.oc_step(self.h, 1, 1, self.lp, None)                   # page the weights in (untimed)
        self.load_s = time.time() - t0
        # thread count: chosen ONCE -- the fastest of {physical cores, half of them, all logical CPUs} on a one-token probe
        # (an oversubscribed run is orders of magnitude slower and would flatter the GPU)
        phys = physical_cores()
        best = None
        for n in sorted({phys, max(1, phys // 2), len(os.sched_getaffinity(0))}):
            lib.oc_set_threads(n)
            lib.oc_reset(self.h)
            t0 = time.time()
            lib.oc_step(self.h, 1, 1, self.lp, None)
            dt = time.time() - t0
            if best is None or dt < best[0]:
                best = (dt, n)
            if dt > 5.0:
                break
        self.threads = best[1]
        lib.oc_set_threads(self.threads)

    def request_sample(self, seed: int, n_prompt: int = 64, n_gen: int = 16, ctx0: int = N_PROMPT - 64):
        """A 1/8-scale request with the real request's 4:1 prompt:generation ratio, AT the real request's context: a synthetic
        KV prefix of ctx0 positions, then n_prompt prompt tokens in one batched pass, then n_gen greedy tokens one by one
        (context ctx0 + n_prompt ... ).  Returns (generated tokens, seconds, prefill seconds, decode seconds) -- all measured."""
        lib, h = self.lib, self.h
        lib.oc_fill_kv(h, ctx0, seed & 0xFFFFFFFF)
        ids = np.random.Generator(np.random.PCG64(1000 + seed)).integers(0, min(self.n_vocab, 128000), size=n_prompt).astype(np.int32)
        t0 = time.perf_counter()
        if lib.oc_prefill(h, ids.ctypes.data_as(C.c_void_p), n_prompt, 1, self.lp) != 0:
            raise RuntimeError("oc_prefill failed")
        t1 = time.perf_counter()
        tok = int(np.argmax(self.logits[: self.n_vocab]))
        for _ in range(n_gen):
            lib.oc_step(h, tok, 1, self.lp, None)
            tok = int(np.argmax(self.logits[: self.n_vocab]))
        t2 = time.perf_counter()
        return n_gen, t2 - t0, t1 - t0, t2 - t1

    def prefill_sample(self, seed: int, n_tokens: int):
        """n_tokens prompt tokens in one batched pass from an empty context; returns seconds (measured)"""
        lib, h = self.lib, self.h
        lib.oc_reset(h)
        ids = np.random.Generator(np.random.PCG64(2000 + seed)).integers(0, min(self.n_vocab, 128000) - 1, size=n_tokens).astype(np.int32)
        t0 = time.perf_counter()
        if lib.oc_prefill(h, ids.ctypes.data_as(C.c_void_p), n_tokens, 1, None) != 0:
            raise RuntimeError("oc_prefill failed")
        return time.perf_counter() - t0

    def close(self):
        self.lib.oc_free(self.h)


def cpu_step(cpu: CpuRestatement, workload: str, seed: int):
    """one bounded CPU sample of `workload` -> (units produced, seconds, description)"""
    if workload in ("config2", "config3"):
        n, dt, tp, td = cpu.request_sample(seed)
        return n, dt, (f"1/8-scale request at the real context: synthetic KV prefix of {N_PROMPT - 64} positions, 64 prompt tokens in one batched pass "
                       f"({tp * 1e3:.0f} ms), 16 greedy tokens ({td / 16 * 1e3:.0f} ms each); tokens/s = 16 / measured seconds")
    if workload == "config4":
        dt = cpu.prefill_sample(seed, 32)
        return 32, dt, "32 prompt tokens of the bf16 model in one batched pass; tokens/s = 32 / measured seconds"
    dt = cpu.prefill_sample(seed, DOC_TOKENS)
    return 1, dt, f"one {DOC_TOKENS}-token document: one batched pass over the q8_0 model (pooling is negligible); docs/s = 1 / measured seconds"


# =====================================================================================================================
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(METRICS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-preflight", action="store_true", help="skip the 8B-shape parity pre-flight (config2)")
    ap.add_argument("--batch", type=int, default=32, help="config3: concurrent requests per GPU")
    ap.add_argument("--docs", type=int, default=1250, help="config5: documents per GPU per step (10 000 / 8 workers)")
    ap.add_argument("--batch-weights", type=int, default=0, help="config3: 0 auto, 1 resident 16-bit weights, 2 quantised weights")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned to its caller as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    wl = args.workload
    if args.dump_outputs and (args.impl != "native" or wl == "config3"):
        # config3's callers receive streamed text, which the vocabulary-less synthetic model leaves empty
        ap.error("--dump-outputs: native arm, workloads config2 / config4 / config5")
    # a stall must leave evidence: every thread's stack goes to stderr if the run makes no visible progress for a while
    import faulthandler
    faulthandler.enable()
    if os.environ.get("GL_BENCH_WATCHDOG", "1") != "0":
        faulthandler.dump_traceback_later(int(os.environ.get("GL_BENCH_WATCHDOG_S", "240")), repeat=True, file=sys.stderr)
    if args.steps is None:
        args.steps = {"config2": 4, "config3": 2, "config4": 2, "config5": 1}[wl]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n_gpus = max(args.gpus, world) if world > 1 else args.gpus

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if args.impl == "native":
            torch.cuda.set_device(local_rank)
            dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        else:
            dist_mod.init_process_group("gloo")
        dist = dist_mod

    def barrier():
        if dist is not None:
            dist.barrier()

    metric, unit = METRICS[wl]
    mkey = WORKLOAD_MODEL[wl]
    config = {
        "config2": {"workload": f"Llama-3-8B q4_K_M synthetic GGUF, greedy decode, {N_PROMPT}-in/{N_GEN}-out, batch=1 per GPU (BASELINE.json configs[1])",
                    "requests_per_gpu_per_step": 1, "prompt_tokens": N_PROMPT, "generated_tokens": N_GEN},
        "config3": {"workload": f"Llama-3-8B q4_K_M synthetic GGUF, {args.batch} concurrent streamed chat requests per GPU ({args.batch * 8} on 8: BASELINE.json "
                                f"configs[2]), {N_PROMPT}-in/{N_GEN}-out, greedy, NativeWorker behind the scheduler rules (least-loaded, priority), continuous batching",
                    "requests_per_gpu_per_step": args.batch, "prompt_tokens": N_PROMPT, "generated_tokens": N_GEN,
                    "prompt": "chat messages flattened as the gateway does ('role: content\\n...assistant:', ollama.ts:367-370); token ids supplied (synthetic vocabulary)"},
        "config4": {"workload": "Llama-3-8B bf16 synthetic GGUF, batched prefill, 32 sequences x 2048 tokens per GPU per step (BASELINE.json configs[3])",
                    "sequences_per_step": 32, "prompt_tokens": 2048},
        "config5": {"workload": f"Mistral-7B q8_0 synthetic GGUF, embeddings of {DOC_TOKENS}-token documents, {args.docs} documents per GPU per step "
                                "(10 000 over 8 workers: BASELINE.json configs[4])", "docs_per_gpu_per_step": args.docs, "doc_tokens": DOC_TOKENS},
    }[wl]
    config["l2_policy"] = "weights (4.9-16 GB per pass) >> 126 MB L2: inputs larger than L2"
    config["parallelism"] = f"replicas x{n_gpus} (request sharding, no collective)"

    # ---------------------------------------------------------------- reference arm (CPU restatement, really timed)
    if args.impl == "reference":
        if rank != 0:
            barrier()
            return
        path = build_model_once(mkey, 0, lambda: None)
        cpu = CpuRestatement(path, 640 if wl in ("config2", "config3") else 512)
        units, secs, desc = 0, 0.0, ""
        for i in range(args.warmup + args.steps):
            n, dt, desc = cpu_step(cpu, wl, i)
            if i >= args.warmup:
                units += n
                secs += dt
        v = units / secs
        out = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "int8 activations x quantised weights (int32 accumulate), CPU", "data": "synthetic", "config": config,
               "cpu_baseline": {"value": v, "unit": unit, "cores": cpu.threads, "kind": "port", "sample": desc, "lib": cpu.so,
                                "note": "CPU restatement of the reference's Ollama-CPU path (ggml-style integer dots, batched prompt pass), not Ollama; "
                                        "model loaded once, thread count chosen once, every step measured"},
               "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        cpu.close()
        print(json.dumps(out), flush=True)
        barrier()
        return

    # ---------------------------------------------------------------- native arm
    from gridllm_b200 import multirank, native as N
    import torch
    if N.device_count() <= local_rank:
        raise SystemExit("bench.py: no CUDA device for this rank -- the native worker has no CPU fallback")
    torch.cuda.set_device(local_rank)
    path = build_model_once(mkey, rank, barrier)
    peaks = {"hbm_gbs": 6650.0, "tf": 1464.2, "src": "fallback (B200_PROFILING.md)"}
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peaks = {"hbm_gbs": float(pk["hbm_gbs"]), "tf": float(pk.get("bf16_tflops_sustained", 1464.2)), "src": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        pass
    sampler = ClockSampler(local_rank)

    def timed(fn):
        """barrier + synchronize, run, synchronize + barrier; clocks sampled on rank 0 during the region"""
        if rank == 0:
            sampler.start()
        try:
            barrier()
            torch.cuda.synchronize()
            r = fn()
            torch.cuda.synchronize()
            barrier()
        finally:                                     # the polling nvidia-smi must not outlive a region that raised
            clocks = sampler.stop() if rank == 0 else None
        return r, clocks

    extra = {}
    if wl == "config2":
        out = run_config2(args, N, path, rank, local_rank, world, dist, timed, peaks, extra)
    elif wl == "config3":
        out = run_config3(args, N, path, rank, local_rank, world, dist, timed, peaks, extra)
    elif wl == "config4":
        out = run_config4(args, N, path, rank, local_rank, world, dist, timed, peaks, extra)
    else:
        out = run_config5(args, N, path, rank, local_rank, world, dist, timed, peaks, extra)
    if rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs, out["outputs"])
    if rank == 0:
        line = {"metric": metric, "value": out["value"], "unit": unit, "n_gpus": out.get("n_gpus", world), "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": out["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": out["dtype"],
                "data": "synthetic", "config": config, "e2e": out["e2e"], "gpu_launches": out["gpu_launches"], "roofline": out["roofline"],
                "clocks": out["clocks"]}
        line.update(out.get("extra", {}))
        if not args.no_cpu and world == 1:                # the contract: the cpu_baseline leg on rank 0 at N = 1 only
            # the CPU leg runs in its own process (the reference arm of this same file, two measured samples after a warm one): the
            # engines are gone by now, and an OpenMP runtime started inside a process that has run CUDA, asyncio and a batch-runner
            # thread has been seen to stall for minutes -- a separate process cannot
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", wl, "--steps", "2", "--warmup", "1"],
                                   capture_output=True, text=True, timeout=420,
                                   env={k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")})
                ref = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
                line["cpu_baseline"] = dict(ref["cpu_baseline"], sample=ref["cpu_baseline"]["sample"] + " (2 measured samples after a warm one)")
            except Exception as ex:  # the baseline is a report, never a gate
                line["cpu_baseline"] = {"value": None, "unit": unit, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
        print(json.dumps(line), flush=True)
    barrier()
    if dist is not None:
        dist.destroy_process_group()


def prompt_for(i: int, n: int = N_PROMPT, vocab: int = 128000) -> np.ndarray:
    return np.random.Generator(np.random.PCG64(1000 + i)).integers(0, vocab, size=n).astype(np.int32)


DUMP_BYTES = 60 << 20                   # array data: with the .npy headers the files stay below 64 MB (10^6 or 2^20 bytes)


def write_outputs(out_dir: str, outputs: dict) -> None:
    """--dump-outputs: one out_dir/<name>.npy per array, token ids as float64 (exact), everything else as float32.  Inputs are
    seeded, so two builds run with the same arguments can be compared file by file.  Above DUMP_BYTES in all, each array keeps
    a fixed, seeded sample of its rows, whose indices are written beside it as <name>_rows.npy."""
    arrays = {k: np.asarray(v, np.float64 if np.issubdtype(np.asarray(v).dtype, np.integer) else np.float32) for k, v in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        for k, a in list(arrays.items()):
            keep = int(DUMP_BYTES * a.nbytes / total) // (a.nbytes // len(a) + 8)
            rows = np.sort(np.random.Generator(np.random.PCG64(0)).choice(len(a), keep, replace=False))
            arrays[k], arrays[f"{k}_rows"] = a[rows], rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)
    log(f"[bench] outputs of the last timed step: {', '.join(f'{k} {a.shape}' for k, a in arrays.items())} -> {out_dir}")


# ---------------------------------------------------------------------------------------------------------------------
def preflight_8b_parity(eng, path: str) -> dict:
    """The benchmarked model itself, GPU vs the C restatement in EXACT mode (dequantised fp32 weights x fp32 activations): 4 prompt
    tokens + 4 greedy tokens through the decode kernels at the full Llama-3-8B shape (32 layers, 128 256-entry vocabulary, K = 14336
    in 4 K-segments, GQA 4:1).  Tolerances of tests/test_gpu_decode.py: logits within 1e-2 * max|logit| of exact arithmetic, logprob
    within 2e-2, ids equal wherever the oracle's top-1/top-2 margin exceeds 5e-2.  Raises on a mismatch: a fast wrong kernel is not a result."""
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "liboracle_cpu.so"))
    lib.oc_load.restype = C.c_void_p
    lib.oc_load.argtypes = [C.c_char_p, C.c_int]
    lib.oc_step.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.oc_free.argtypes = [C.c_void_p]
    h = lib.oc_load(path.encode(), 64)
    nv = eng.info.n_vocab
    ref = np.zeros(nv, np.float32)
    prompt = prompt_for(424242, 4)
    eng.kv_reset()
    worst, margins, n_cmp = 0.0, [], 0
    tok = None
    for i in range(8):
        t = int(prompt[i]) if i < 4 else tok
        lg, am, lp = eng.decode_step(t)
        lib.oc_step(h, t, 0, ref.ctypes.data_as(C.c_void_p), None)
        scale = float(np.abs(ref).max())
        err = float(np.abs(lg - ref).max())
        worst = max(worst, err / scale)
        if not (err <= 1e-2 * scale):
            raise SystemExit(f"bench.py pre-flight: GPU logits differ from the oracle at token {i}: max|d| {err:.4g} vs scale {scale:.4g}")
        srt = np.sort(ref)
        margin = float(srt[-1] - srt[-2])
        margins.append(margin)
        ref_id = int(np.argmax(ref))
        lse = float(ref.max() + np.log(np.exp(ref - ref.max()).sum()))
        if abs(lp - (float(ref[am]) - lse)) > 2e-2:
            raise SystemExit(f"bench.py pre-flight: logprob differs at token {i}")
        if margin > 5e-2 and am != ref_id:
            raise SystemExit(f"bench.py pre-flight: greedy id differs from the oracle at token {i} with margin {margin:.3g}")
        n_cmp += 1
        tok = ref_id                                                 # follow the oracle's trajectory
    lib.oc_free(h)
    eng.kv_reset()
    return {"tokens_compared": n_cmp, "worst_logit_err_over_scale": worst, "min_top1_top2_margin": min(margins), "oracle": "oracle/c/llama_cpu.c exact mode",
            "tolerance": "1e-2 * max|logit|; ids equal where margin > 5e-2"}


def run_config2(args, N, path, rank, local_rank, world, dist, timed, peaks, extra):
    from gridllm_b200 import multirank
    eng = N.Engine(path, device=local_rank, max_ctx=1024)
    info = eng.info
    pre = None
    # At N > 1 every rank runs the same kernels on the same model as the N = 1 line of the same tree, which carries the check; the
    # C restatement also competes with the other ranks for the host cores there (66 s at N = 2 against 9 s at N = 1, run Y), so the
    # multi-rank lines skip it unless GL_BENCH_PREFLIGHT_MULTI=1.
    if world > 1 and os.environ.get("GL_BENCH_PREFLIGHT_MULTI", "0") != "1":
        pre = {"skipped": "world > 1: the N = 1 line of the same tree carries the 8B-shape parity check (GL_BENCH_PREFLIGHT_MULTI=1 runs it here too)"}
    elif rank == 0 and not args.no_preflight:
        t0 = time.time()
        pre = preflight_8b_parity(eng, path)
        pre["seconds"] = round(time.time() - t0, 1)
        log(f"[bench] pre-flight parity at the benchmarked shape: {pre}")
    for w in range(args.warmup):
        eng.generate(prompt_for(10_000 + w), num_predict=N_GEN, ignore_eos=True)

    def region():
        dev_ns = wall = launches = gen_tokens = prefill_ns = 0
        last = None
        for i in range(args.steps):
            p = prompt_for(multirank.request_seeds(rank, i, 1)[0])
            t0 = time.perf_counter()
            g = eng.generate(p, num_predict=N_GEN, ignore_eos=True)
            wall += time.perf_counter() - t0
            dev_ns += g.stats.prompt_eval_duration_ns + g.stats.eval_duration_ns
            prefill_ns += g.stats.prompt_eval_duration_ns
            launches += g.stats.kernel_launches
            gen_tokens += int(g.stats.eval_count)
            last = g
        return dev_ns, wall, launches, gen_tokens, prefill_ns, last
    (dev_ns, wall_s, launches, gen_tokens, prefill_ns, last), clocks = timed(region)
    assert gen_tokens == args.steps * N_GEN and np.isfinite(last.logprobs).all()
    ms_tok, nl_tok = eng.time_decode(N_PROMPT + N_GEN // 2, 32)      # decode-step roofline (CUDA events inside the library, its own stream)
    agg = multirank.aggregate_throughput(float(gen_tokens), dev_ns * 1e-9, wall_s, dist)
    bpt = int(info.decode_bytes_per_token)
    eng.close()
    achieved = bpt / (ms_tok * 1e-3) / 1e9
    return {"value": agg["value"], "ms_per_step": agg["device_s"] / args.steps * 1e3,
            "dtype": "q4_K/q6_K weights x int16 fixed-point activations (int32 dot, fp32 accumulate)",
            "e2e": {"value": agg["e2e"], "unit": "tokens/s", "h2d_bytes_per_step": N_PROMPT * 4 + 64, "d2h_bytes_per_step": N_GEN * 8 + 4 * 64,
                    "api": "gl_generate (C ABI, host buffers)"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "gemv_kernel (all weight GEMVs of one decode step, ctx 576)", "achieved": achieved, "peak": peaks["hbm_gbs"],
                         "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "peak_source": peaks["src"], "algorithmic_bytes_per_token": bpt,
                         "ms_per_decode_step": ms_tok, "launches_per_decode_step": nl_tok,
                         "traffic": None, "traffic_note": "DRAM bytes == algorithmic bytes to 0.02 % in the committed ncu --set full capture "
                                                          "(profiles/r01_run59_ncu_summary.md); not re-measured by this run"},
            "clocks": clocks,
            "extra": {"breakdown": {"prefill_ms_per_request": prefill_ns / args.steps * 1e-6, "decode_ms_per_request": (dev_ns - prefill_ns) / args.steps * 1e-6,
                                    "decode_tok_s_per_gpu": N_GEN / ((dev_ns - prefill_ns) / args.steps * 1e-9)},
                      "parity_preflight": pre},
            "outputs": {"ids": last.ids, "logprobs": last.logprobs}}


# ---------------------------------------------------------------------------------------------------------------------
def flatten_chat(messages) -> str:
    """the gateway's /api/chat prompt (server/src/routes/ollama.ts:367-370): 'role: content' lines, then 'assistant:'"""
    return "\n".join(f"{m['role']}: {m['content']}" for m in messages) + "\nassistant:"


def run_config3(args, N, path, rank, local_rank, world, dist, timed, peaks, extra):
    """B concurrent streamed chat requests per GPU through NativeWorker(s) behind the scheduler rules.  Under torchrun every rank
    is one worker; without torchrun and --gpus N, N workers (one engine per GPU) live in THIS process behind one scheduler."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from sched_standin import SchedulerStandIn
    from gridllm_b200 import multirank, service as SV
    from gridllm_b200.worker import LocalBus, NativeWorker
    B = args.batch
    n_local = args.gpus if (world == 1 and args.gpus > 1) else 1
    if n_local > N.device_count():
        raise SystemExit(f"bench.py: --gpus {n_local} in one process needs {n_local} visible devices")
    devices = [local_rank] if n_local == 1 else list(range(n_local))
    name = "llama3-8b-q4km:synth"
    svcs = [SV.NativeInferenceService({name: path}, device=d, max_ctx=1024, max_batch=B, batch_weights=args.batch_weights) for d in devices]
    for s in svcs:
        s.preload()
    engines = [s._engine(name) for s in svcs]
    log(f"[bench] config3: {n_local} engine(s) loaded, batch {B}")

    def make_jobs(step_tag, n_req):
        jobs = []
        for i in range(n_req):
            seed = multirank.request_seeds(rank, 0, 1)[0] * 64 + step_tag * 4096 + i
            msgs = [{"role": "system", "content": "You are a helpful assistant."}, {"role": "user", "content": f"synthetic request {seed}"}]
            jobs.append({"id": f"chat-{rank}-{step_tag}-{i}", "model": name, "prompt": flatten_chat(msgs), "stream": True,
                         "priority": ("high", "medium", "low")[i % 3], "timeout": 300000,
                         "options": {"num_predict": N_GEN, "temperature": 0, "ignore_eos": True},
                         "metadata": {"ollamaEndpoint": "/api/chat", "prompt_token_ids": prompt_for(seed).tolist()}})
        return jobs

    async def run_step(step_tag, tick_s):
        bus = LocalBus()
        sched = SchedulerStandIn(bus, max_jobs_per_worker=B, tick_s=tick_s)
        workers = [NativeWorker(f"b200-{rank * max(1, n_local) + k}", s, bus, max_concurrent=B) for k, s in enumerate(svcs)]
        await sched.start()
        for w in workers:
            await w.start()
        jobs = make_jobs(step_tag, B * n_local)
        for j in jobs:
            await sched.watch_stream(j["id"])
        t0 = time.perf_counter()
        for j in jobs:
            sched.add_job(j)
        await sched.run_until_empty()
        wall = time.perf_counter() - t0
        for w in workers:
            await w.stop()
        ok = sum(1 for j in jobs if "result" in sched.results.get(j["id"], {}))
        errs = [str(sched.results.get(j["id"], {}).get("error")) for j in jobs if "result" not in sched.results.get(j["id"], {})]
        chunks = sum(sched.stream_chunks.get(j["id"], 0) for j in jobs)
        used = sorted(set(sched.assigned.values()))
        ttft = [sched.first_chunk_at[j["id"]] - sched.submitted_at[j["id"]] for j in jobs if j["id"] in sched.first_chunk_at]
        return {"wall": wall, "ok": ok, "chunks": chunks, "workers_used": used, "ticks": sched.ticks, "n": len(jobs),
                "ttft_median_s": statistics.median(ttft) if ttft else None, "first_error": errs[0] if errs else None}

    loop = asyncio.new_event_loop()
    for w in range(min(args.warmup, 1) + 0):                          # one warm pass captures the graphs of every bucket it meets
        r = loop.run_until_complete(run_step(1000 + w, 0.0))
        log(f"[bench] config3 warm pass: {r['ok']}/{r['n']} requests in {r['wall']:.2f} s, counters {engines[0].batch_counters()}")
        if r["ok"] != r["n"]:            # fail NOW and loudly: a worker that answers every job with an error is not a slow worker
            raise SystemExit(f"[bench] config3: {r['n'] - r['ok']} of {r['n']} warm-up requests failed: {r.get('first_error')}")
    for e in engines:
        e.batch_counters(reset=True)

    def region():
        res = []
        for i in range(args.steps):
            res.append(loop.run_until_complete(run_step(i, 0.0)))
            log(f"[bench] config3 step {i}: {res[-1]['ok']}/{res[-1]['n']} requests in {res[-1]['wall']:.2f} s")
        return res
    res, clocks = timed(region)
    ctr = [e.batch_counters(reset=True) for e in engines]
    n_req = sum(r["n"] for r in res)
    assert all(r["ok"] == r["n"] for r in res), "a request failed"
    assert all(r["chunks"] == r["n"] * (N_GEN + 1) for r in res), "stream chunk count"
    gen_tokens = float(n_req * N_GEN)
    dev_s = max((c["step_ns"] + c["prefill_ns"]) * 1e-9 for c in ctr)      # the slowest worker of this process
    wall_s = sum(r["wall"] for r in res)
    agg = multirank.aggregate_throughput(gen_tokens, dev_s, wall_s, dist)
    # the same workload once more with the reference's 1 s dispatch tick (JobScheduler.ts:128-135), reported beside the headline
    tick1 = loop.run_until_complete(run_step(500, 1.0))
    log(f"[bench] config3 1 s-tick pass: {tick1['wall']:.2f} s, {tick1['ticks']} ticks")
    for e in engines:
        e.batch_counters(reset=True)
    # roofline of the batched step: weights are read once per step for all B sequences
    ms_step, nl_step, wbytes = engines[0].time_batch_step(B, N_PROMPT + N_GEN // 2, 16)
    info = engines[0].info
    bpt = int(info.decode_bytes_per_token)
    kv_bytes = 2 * info.n_layer * info.n_head_kv * info.head_dim * 2 * (N_PROMPT + N_GEN // 2) * B       # fp16 K and V of every cached position
    achieved = (bpt + kv_bytes) / (ms_step * 1e-3) / 1e9
    steps_total = sum(c["steps"] for c in ctr)
    rows_total = sum(c["rows"] for c in ctr)
    launches = int(sum(c["launches"] for c in ctr))
    for s in svcs:
        s.close()
    return {"value": agg["value"], "ms_per_step": agg["device_s"] / args.steps * 1e3, "n_gpus": world * n_local,
            "dtype": "fp16 tensor-core GEMMs (fp32 accumulate) over q4_K/q6_K weights, fp16 KV",
            "e2e": {"value": agg["e2e"], "unit": "tokens/s", "h2d_bytes_per_step": B * n_local * (N_PROMPT * 4 + 64),
                    "d2h_bytes_per_step": B * n_local * N_GEN * 16, "api": "NativeWorker.handleJobMessage -> NativeInferenceService.generateStreamResponse -> "
                    "gl_seq_open / gl_batch_step (C ABI, host buffers); wall clock from first submission to last result, scheduler tick 0"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": f"one batched decode step, B = {B}, ctx {N_PROMPT + N_GEN // 2} (weight GEMMs + paged attention)",
                         "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "peak_source": peaks["src"],
                         "algorithmic_bytes_per_step": bpt + kv_bytes, "algorithmic_weight_bytes": bpt, "algorithmic_kv_bytes": kv_bytes,
                         "weight_bytes_this_path_reads": int(wbytes), "ms_per_batched_step": ms_step, "launches_per_batched_step": nl_step,
                         "tokens_per_s_at_this_step_time": B / (ms_step * 1e-3), "traffic": None},
            "clocks": clocks,
            "extra": {"config3": {"requests": n_req, "workers_in_process": n_local, "workers_used": res[-1]["workers_used"],
                                  "mean_batch": rows_total / max(1, steps_total), "batched_steps": steps_total,
                                  "prefill_device_s": sum(c["prefill_ns"] for c in ctr) * 1e-9, "decode_device_s": sum(c["step_ns"] for c in ctr) * 1e-9,
                                  "ttft_median_s": res[-1]["ttft_median_s"],
                                  "wall_tick0": {"tokens_per_s": gen_tokens / wall_s, "seconds_per_step": wall_s / args.steps},
                                  "wall_tick1s": {"tokens_per_s": tick1["n"] * N_GEN / tick1["wall"], "seconds": tick1["wall"], "ticks": tick1["ticks"],
                                                  "note": "the reference's 1 000 ms dispatch tick (JobScheduler.ts:128-135), MAX_CONCURRENT_JOBS_PER_WORKER = batch"}}}}


# ---------------------------------------------------------------------------------------------------------------------
def run_config4(args, N, path, rank, local_rank, world, dist, timed, peaks, extra):
    from gridllm_b200 import multirank
    T, S = 2048, 32
    eng = N.Engine(path, device=local_rank, max_ctx=T + 16)
    info = eng.info
    for w in range(max(1, args.warmup)):
        eng.generate(prompt_for(77_000 + w, T), num_predict=1, ignore_eos=True)

    def region():
        dev_ns = wall = launches = 0
        for i in range(args.steps):
            gens = []
            for s in range(S):
                p = prompt_for(2000 + multirank.request_seeds(rank, i, 1)[0] * S + s, T)
                t0 = time.perf_counter()
                g = eng.generate(p, num_predict=1, ignore_eos=True)
                wall += time.perf_counter() - t0
                dev_ns += g.stats.prompt_eval_duration_ns
                launches += g.stats.kernel_launches
                gens.append(g)
        return dev_ns, wall, launches, gens
    (dev_ns, wall_s, launches, gens), clocks = timed(region)
    tokens = float(args.steps * S * T)
    agg = multirank.aggregate_throughput(tokens, dev_ns * 1e-9, wall_s, dist)
    qd, kvd = info.n_head * info.head_dim, info.n_head_kv * info.head_dim
    lin_params = info.n_layer * ((qd + 2 * kvd) * info.n_embd + info.n_embd * qd + 3 * info.n_ff * info.n_embd)
    flops_seq = 2.0 * lin_params * T + 2.0 * T * T * qd * info.n_layer + 2.0 * info.n_vocab * info.n_embd      # linear + causal attention + one lm_head row
    achieved = flops_seq * S * args.steps / (dev_ns * 1e-9) / 1e12
    eng.close()
    return {"value": agg["value"], "ms_per_step": agg["device_s"] / args.steps * 1e3,
            "dtype": "fp16 tensor cores (tcgen05, fp32 accumulate in TMEM); bf16 weights converted once at load (exact inside fp16's range)",
            "e2e": {"value": agg["e2e"], "unit": "tokens/s", "h2d_bytes_per_step": S * (T * 4 + 64), "d2h_bytes_per_step": S * 72,
                    "api": "gl_generate(prompt 2048, num_predict 1) x 32 (C ABI, host buffers)"},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "gemm_tc5_kernel (the prefill's linear layers: > 90 % of the step's flops); whole prefill timed",
                         "achieved": achieved, "peak": peaks["tf"], "unit": "TFLOP/s", "frac": achieved / peaks["tf"], "peak_source": peaks["src"],
                         "algorithmic_flops_per_step": flops_seq * S, "traffic": None},
            "clocks": clocks, "extra": {},
            "outputs": {"ids": np.concatenate([g.ids for g in gens]), "logprobs": np.concatenate([g.logprobs for g in gens])}}


def run_config5(args, N, path, rank, local_rank, world, dist, timed, peaks, extra):
    from gridllm_b200 import multirank
    eng = N.Engine(path, device=local_rank, max_ctx=4096)
    info = eng.info
    pack = 16                                                           # documents per gl_embed call (/api/embed input: string[])

    def docs(step, k, n):
        base = 3000 + multirank.request_seeds(rank, step, 1)[0] * 100000 + k
        return [prompt_for(base + j, DOC_TOKENS, 32000 - 1) for j in range(n)]
    eng.embed(docs(999, 0, pack))

    def region():
        dev_ns = wall = launches = n = 0
        for i in range(args.steps):
            k, embs = 0, []
            while k < args.docs:
                d = docs(i, k, min(pack, args.docs - k))
                t0 = time.perf_counter()
                emb, st = eng.embed(d)
                wall += time.perf_counter() - t0
                dev_ns += st.prompt_eval_duration_ns
                launches += st.kernel_launches
                n += len(d)
                k += len(d)
                embs.append(emb)
        assert np.isfinite(emb).all()
        return dev_ns, wall, launches, n, embs
    (dev_ns, wall_s, launches, n, embs), clocks = timed(region)
    agg = multirank.aggregate_throughput(float(n), dev_ns * 1e-9, wall_s, dist)
    qd, kvd = info.n_head * info.head_dim, info.n_head_kv * info.head_dim
    lin_params = info.n_layer * ((qd + 2 * kvd) * info.n_embd + info.n_embd * qd + 3 * info.n_ff * info.n_embd)
    flops_doc = 2.0 * lin_params * DOC_TOKENS + 2.0 * DOC_TOKENS * DOC_TOKENS * qd * info.n_layer
    achieved = flops_doc * n / (dev_ns * 1e-9) / 1e12
    eng.close()
    return {"value": agg["value"], "ms_per_step": agg["device_s"] / args.steps * 1e3,
            "dtype": "fp16 tensor cores (fp32 accumulate) over q8_0 weights dequantised once at load",
            "e2e": {"value": agg["e2e"], "unit": "docs/s", "h2d_bytes_per_step": args.docs * (DOC_TOKENS * 4 + 4),
                    "d2h_bytes_per_step": args.docs * info.n_embd * 4, "api": f"gl_embed, {pack} documents per call (C ABI, host buffers)"},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "gemm_tc5_kernel (packed prompt pass); whole gl_embed device time", "achieved": achieved,
                         "peak": peaks["tf"], "unit": "TFLOP/s", "frac": achieved / peaks["tf"], "peak_source": peaks["src"],
                         "algorithmic_flops_per_doc": flops_doc, "traffic": None},
            "clocks": clocks, "extra": {"docs_per_call": pack}, "outputs": {"embeddings": np.concatenate(embs)}}


if __name__ == "__main__":
    main()
