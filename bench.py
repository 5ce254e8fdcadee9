#!/usr/bin/env python
"""bench.py — throughput of the ensemble-SAE training hot path (BASELINE.json metric: activations/sec/GPU).

    python bench.py --gpus N --steps K --warmup W                     # this engine
    python bench.py --impl reference --gpus N --steps K --warmup W    # the reference's own CPU PyTorch path

A "step" is one ``FunctionalEnsemble.step_batch`` over one batch of synthetic activations: forward, losses,
backward and the Adam update of every model of the ensemble (nothing is skipped or cached). The workload at N=1 is
BASELINE config 2: 16 tied SAEs, d_model=512, dict_ratio=8 (n=4096), L1 = logspace(-4,-2,16), batch 8192, fp32
parameters, lr 1e-3. For N>1 every rank trains its own 16-model shard on the same activation stream (config 4:
model-axis sharding, no data-path collective) — weak scaling; value = rows consumed by all ranks' shards per second.

Printed JSON (one line, rank 0): the driver contract plus
  value           K steps on device-resident batches between two CUDA events, NOTHING else in the loop (max over ranks)
  e2e             the same through the public API with HOST (pinned) batches: side-stream H2D of the next batch
                  (train_loop.HostBatchPrefetcher) + step + D2H of the losses every step; `e2e.serial` is the same
                  loop with the copy on the compute stream, with its copy / step split measured by CUDA events
  phases_ms       per-phase device time of a step, measured in a SEPARATE short loop (events recorded inside libsce)
  roofline        dominant kernel (weight-gradient GEMM): algorithmic FLOPs / CUDA-event time vs the measured bf16
                  peak; per-GEMM fractions; DRAM bytes per step from the committed ncu capture
  cpu_baseline    one step of the oracle port of the reference on this box's host cores at the FULL batch
  stock_torch_gpu the same oracle port (the op sequence the reference launches) on THIS GPU, fp32 and TF32
  cfg4_stream     config 4's data path: fp16 chunks from disk -> pinned -> HBM -> device-side gather -> step, with
                  the end-of-chunk metric gather (also a workload of its own: --workload cfg4_stream)

--dump-outputs DIR writes what the last step of the `value` loop returned, and the parameters it left, as .npy files
(see dump_outputs); the inputs depend only on the arguments, so two builds can be compared file by file.
"""
import argparse
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (M, d, n, B, description)
    "cfg2": (16, 512, 4096, 8192, "16 TiedSAE d_model=512 dict_ratio=8 L1=logspace(-4,-2,16) batch=8192 (BASELINE configs[1])"),
    "cfg1": (1, 128, 256, 1024, "1 TiedSAE d_model=128 dict_ratio=2 L1=1e-3 batch=1024 (BASELINE configs[0])"),
    "cfg5": (1, 2048, 32768, 4096, "1 TiedSAE/GPU d_model=2048 dict_ratio=16 batch=4096 (BASELINE configs[4])"),
    "cfg3": (32, 768, None, 8192, "32 TopK d_model=768 dict_ratio in {4,8,16} (11+11+10 models) k in {16,32,64} batch=8192 (BASELINE configs[2])"),
    "cfg3g": (12, 768, 6144, 8192, "12 TopK d_model=768 dict_ratio=8 k in {16,32,64} batch=8192 (one shape group of BASELINE configs[2])"),
    "cfg4_stream": (16, 512, 4096, 8192, "16 TiedSAE/GPU d_model=512 dict_ratio=8, fp16 activation chunks of [2^21, 512] streamed from disk (BASELINE configs[3])"),
}
CFG3_GROUPS = ((3072, 11), (6144, 11), (12288, 10))       # (dict size, models): 32 models in three shape groups
METRIC = "activations/sec (whole job; rows consumed by every resident model)"


def l1_grid(M):
    return [1e-3] if M == 1 else [float(a) for a in np.logspace(-4, -2, M)]


def make_models(sig, M, d, n, seed):
    torch.manual_seed(seed)
    if getattr(sig, "variant", None) == "topk":
        return [sig.init(d, n, (16, 32, 64)[i % 3]) for i in range(M)]
    return [sig.init(d, n, a) for a in l1_grid(M)]


ACT_FP16 = True   # --act-precision: values as the reference caches them (fp16, activation_dataset.py:404-412) or raw fp32


def synth_batches(n_batches, B, d, seed, pin=False):
    """Sparse-mixture activations (the distribution of sc_datasets/random_dataset.py:76-142): a few unit features
    per row + noise, so that ReLU sparsity is non-trivial. Returns CPU fp32 tensors; with ACT_FP16 the VALUES are
    rounded to fp16 first, which is what a chunk written by the reference's harvester and loaded by big_sweep.py
    (`torch.load(chunk_loc).to(device="cpu", dtype=torch.float32)`, big_sweep.py:358) contains."""
    gen = torch.Generator().manual_seed(seed)
    feats = torch.randn(2048, d, generator=gen)
    feats /= feats.norm(dim=-1, keepdim=True)
    out = []
    for _ in range(n_batches):
        codes = (torch.rand(B, 2048, generator=gen) < 0.01).float() * torch.rand(B, 2048, generator=gen)
        x = codes @ feats + 0.05 * torch.randn(B, d, generator=gen)
        if ACT_FP16:
            x = x.half().float()
        out.append(x.pin_memory() if pin else x)
    return out


def _die_with_parent():
    """Runs in the sampler's child before exec: the kernel sends it SIGTERM when bench.py exits, also on an exception
    or a kill, so a failed run leaves no sampling nvidia-smi behind."""
    import ctypes
    import signal
    PR_SET_PDEATHSIG = 1
    ctypes.CDLL(None).prctl(PR_SET_PDEATHSIG, signal.SIGTERM)


class ClockSampler:
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        """Started at process start: nvidia-smi needs about a second before its first sample, the timed region of a
        20-step run is 0.1 s."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL,
                                         preexec_fn=_die_with_parent)
        except OSError:
            self.proc = None

    @staticmethod
    def _ts(text):
        import datetime
        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, windows):
        """``windows``: {name: (t_begin, t_end)} in time.time() seconds; the first one is the timed region of `value`
        and gives sm_mhz / reasons; every window gets its own summary (a 0.1 s region may hold only a few samples, the
        longer ones back it up)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [t.strip() for t in line.split(",")]
            if len(f) < 9:
                continue
            ts = self._ts(f[0])
            try:
                rows.append((ts, float(f[1]), float(f[2]), float(f[3]),
                             [n for n, v in zip(names, f[5:9]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        os.unlink(self.path)

        def summary(lo, hi):
            sel = [r for r in rows if r[0] is not None and lo - 0.01 <= r[0] <= hi + 0.01]
            if not sel:
                return None
            return {"sm_mhz": float(np.median([r[1] for r in sel])), "sm_max_mhz": float(max(r[2] for r in sel)),
                    "power_w_max": float(max(r[3] for r in sel)), "samples": len(sel),
                    "reasons": sorted({n for r in sel for n in r[4]})}

        out = None
        extra = {}
        for i, (name, (lo, hi)) in enumerate(windows.items()):
            s = summary(lo, hi)
            if i == 0:
                out = s
            elif s is not None:
                extra[name] = s
        if out is None:                     # the timed region fell between two samples: report the enclosing load window
            for name, s in extra.items():
                out = dict(s, window=name)
                break
        if out is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        out["other_windows"] = extra
        return out


class _StdoutGuard:
    """stdout must carry exactly ONE JSON line. Libraries (NCCL's version banner, for one) write to file descriptor
    1 behind Python's back, so fd 1 is pointed at stderr for the whole run and the JSON goes to a saved duplicate of
    the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, obj):
        sys.stdout.flush()
        os.write(self.real, (json.dumps(obj) + "\n").encode())


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"bf16_tflops": p.get("bf16_tflops_sustained", p.get("bf16_tflops")), "hbm_gbs": p.get("hbm_gbs"),
                "source": "measured (MEASURED_PEAKS.json, sustained bf16)"}
    return {"bf16_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic():
    """DRAM bytes per launch of every kernel of a step from the committed `ncu --set full` capture (profiles/)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    return json.load(open(path)) if os.path.exists(path) else None


DUMP_BYTES = 60_000_000                 # with the .npy headers, under 64 MB in all


def dump_outputs(folder, enss, results):
    """Writes, as float32 ``folder/<name>.npy``, what one step returned to its caller — every loss term [M], the mean
    L0 [M] and the code [M, B, n] of ``aux["c"]`` — and every parameter the step left ([M, n, d] / [M, n]); names
    carry a ``g<i>_`` prefix when the workload steps several ensembles. An array larger than its share of
    DUMP_BYTES is cut along axis 1 (batch rows of the code, dictionary rows of a parameter) to a seeded, sorted subset
    of indices, the same on every run. Returns {name: shape written}."""
    arrays = {}
    for g, (e, (losses, aux)) in enumerate(zip(enss, results)):
        pre = f"g{g}_" if len(enss) > 1 else ""
        arrays.update({pre + k: v for k, v in losses.items()})
        arrays[pre + "mean_l0"] = aux["c"].count_nonzero(dim=-1).float().mean(dim=-1)
        arrays[pre + "code"] = aux["c"]                       # CodeProxy: read back from the engine when indexed
        arrays.update({pre + k: v for k, v in e.params.items()})
    os.makedirs(folder, exist_ok=True)
    budget, left, shapes = DUMP_BYTES, len(arrays), {}
    for name, v in sorted(arrays.items(), key=lambda kv: math.prod(kv[1].shape)):
        share = budget // left                                # small arrays leave their unused share to the large
        left -= 1
        size = 4 * math.prod(v.shape)
        if size > share:
            keep = max(1, share // (size // v.shape[1]))
            idx = torch.randperm(v.shape[1], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            v = v[:, idx.to(v.device)]
        a = v.float().cpu().numpy()
        np.save(os.path.join(folder, name + ".npy"), a)
        budget -= a.nbytes
        shapes[name] = list(a.shape)
    return shapes


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own PyTorch path (oracle port) on host cores
# ----------------------------------------------------------------------------------------------------------------
class _CpuReference:
    """The restated reference step (vmap(grad(loss)) + Adam, fp32, host threads) for the FULL ensemble, run as
    groups of models so that the [m, B, n] fp32 temporaries (about a dozen live copies) stay within host memory at
    the full batch: the arithmetic and the total work per step are those of one 16-model vmap."""

    def __init__(self, M, d, n, B, mem_bytes=20e9):
        from oracle import sae_oracle as O
        from sparse_coding_b200 import FunctionalTiedSAE
        models = make_models(FunctionalTiedSAE, M, d, n, 0)
        per_model = 12 * 4 * B * n
        group = int(max(1, min(M, mem_bytes // per_model)))
        self.groups = [O.RefPortEnsemble(models[i:i + group], O.SIG_LOSSES["tied"], lr=1e-3) for i in range(0, M, group)]
        self.group = group

    def step(self, chunk, B):
        batch = chunk[torch.randperm(chunk.shape[0])[:B]]       # the reference's CPU gather (big_sweep.py:168)
        for g in self.groups:
            g.step_batch(batch)


def _pick_threads(ref, probe_chunk, Bp):
    """Oversubscribing SMT siblings can be slower than fewer threads: time one small step per candidate count."""
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    ref.step(probe_chunk, Bp)                            # one-off tracing / allocator warm-up, not timed
    best = None
    for th in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
        torch.set_num_threads(th)
        t0 = time.perf_counter()
        ref.step(probe_chunk, Bp)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, th)
    torch.set_num_threads(best[1])
    return best


def cpu_reference_rate(M, d, n, B_full, budget_s, steps=1, warmup=0):
    """Times ``steps`` steps of the restated reference on this box's host cores. The batch is the FULL one when
    (steps + warmup) of them fit ``budget_s`` (estimated from a 256-row probe), else the largest multiple of 64 rows
    that does. Returns (activations/s, sample description, cores, seconds per step, rows per step)."""
    ref = _CpuReference(M, d, n, B_full)
    Bp = min(B_full, 256)
    probe = synth_batches(1, max(Bp, 64), d, 123)[0]
    probe_dt, cores = _pick_threads(ref, probe, Bp)
    per_row = probe_dt / Bp
    Bs = B_full if per_row * B_full * (steps + warmup) <= budget_s else \
        max(64, int(budget_s / max(steps + warmup, 1) / per_row) // 64 * 64)
    Bs = min(Bs, B_full)
    chunk = synth_batches(1, Bs, d, 124)[0]
    for _ in range(warmup):
        ref.step(chunk, Bs)
    t0 = time.perf_counter()
    for _ in range(steps):
        ref.step(chunk, Bs)
    dt = (time.perf_counter() - t0) / steps
    sample = (f"{steps} step(s) of the full {M}-model ensemble (vmap groups of {ref.group}) at batch {Bs} of {B_full} "
              f"rows (fp32, torch CPU, gather included)")
    return Bs / dt, sample, cores, dt, Bs


def run_reference(args, rank, world, out):
    if rank != 0:
        return
    wl = "cfg2" if args.workload in ("cfg4_stream",) else args.workload
    M, d, n, B, desc = WORKLOADS[wl]
    if n is None:
        raise SystemExit("--impl reference: use a single-shape workload (cfg1, cfg2, cfg3g is TopK: cfg2 is the arm's config)")
    K, W = max(args.steps, 1), max(args.warmup, 0)
    # the whole K + W run has to end within a few minutes: full batches when they fit ~150 s, else a bounded sample
    rate, sample, cores, dt, Bs = cpu_reference_rate(M, d, n, B, budget_s=150.0, steps=K, warmup=min(W, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "activations/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl}: {desc}", "parallelism": "host CPU threads", "batch_timed": Bs,
                   "same_config": bool(Bs == B)},
        "cpu_baseline": {"value": rate, "unit": "activations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "activations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if Bs != B:
        # one extra step at the full batch, outside the K timed ones, so that a like-for-like number exists
        ref = _CpuReference(M, d, n, B)
        chunk = synth_batches(1, B, d, 125)[0]
        t0 = time.perf_counter()
        ref.step(chunk, B)
        full_dt = time.perf_counter() - t0
        line["full_batch_step"] = {"value": B / full_dt, "unit": "activations/s", "seconds": full_dt, "batch": B,
                                   "same_config": True}
    out.emit(line)


# ----------------------------------------------------------------------------------------------------------------
# config 4's data path: chunks streamed from disk
# ----------------------------------------------------------------------------------------------------------------
def _scratch_dir(need_bytes):
    for base in ("/dev/shm", tempfile.gettempdir()):
        try:
            if shutil.disk_usage(base).free > need_bytes * 1.3:
                return tempfile.mkdtemp(prefix="sce_chunks_", dir=base), base
        except OSError:
            continue
    return None, None


def _write_chunks(folder, n_chunks, rows, d, dev):
    """Synthesise fp16 activation chunks on the GPU (same sparse mixture as synth_batches) and write them in the
    reference's on-disk format: {i}.pt, fp16 [rows, d] (activation_dataset.py:499-503)."""
    gen = torch.Generator(device=dev).manual_seed(4242)
    feats = torch.randn(2048, d, generator=gen, device=dev)
    feats /= feats.norm(dim=-1, keepdim=True)
    piece = 1 << 16
    for c in range(n_chunks):
        host = torch.empty(rows, d, dtype=torch.float16)
        for lo in range(0, rows, piece):
            r = min(piece, rows - lo)
            codes = (torch.rand(r, 2048, generator=gen, device=dev) < 0.01).float() * torch.rand(r, 2048, generator=gen, device=dev)
            x = codes @ feats + 0.05 * torch.randn(r, d, generator=gen, device=dev)
            host[lo:lo + r] = x.half().cpu()
        torch.save(host, os.path.join(folder, f"{c}.pt"))


def run_stream(S, dist, rank, world, dev, M, d, n, B, n_chunks, rows, feed, resident_ms_per_step):
    """16 tied models per rank trained over `n_chunks` chunk files with train_on_chunks: disk -> pinned -> HBM (side
    stream, overlapped with the previous chunk's steps) -> device-side permutation gather + fp16->fp32 -> step, metric
    all_gather at the end of every chunk. Timed from before the first chunk is requested to the end of the last
    chunk's gather (wall clock bracketed by device synchronisation, max over ranks); the export at the end is timed
    separately."""
    from sparse_coding_b200.sharding import gather_metrics
    from sparse_coding_b200.train_loop import ChunkStreamer, train_on_chunks  # noqa: F401
    need = n_chunks * rows * d * 2
    info = [None, None, None]
    if rank == 0:
        folder, base = _scratch_dir(need)
        info = [folder, base, None]
        if folder is not None:
            t0 = time.perf_counter()
            _write_chunks(folder, n_chunks, rows, d, dev)
            info[2] = time.perf_counter() - t0
    if world > 1:
        dist.broadcast_object_list(info, src=0)
    folder, base = info[0], info[1]
    if folder is None:
        return {"skipped": f"no scratch directory with {need / 2**30:.1f} GiB free"}
    outdir = tempfile.mkdtemp(prefix=f"sce_out_{rank}_")
    try:
        ens = S.FunctionalEnsemble(make_models(S.FunctionalTiedSAE, M, d, n, seed=100 + rank), S.FunctionalTiedSAE, S.adam,
                                   {"lr": 1e-3}, device=dev)
        ens.step_batch(torch.randn(B, d, device=dev))                   # plan + workspace outside the timed region
        marks = []

        def on_chunk_end(i, chunk_idx, e):
            local = torch.stack([e._last_loss, e._last_nnz], dim=1) if hasattr(e, "_last_loss") else \
                torch.zeros(M, 2, device=dev)
            allm = gather_metrics(local)                                 # the path's only collective: [M_total, 2]
            torch.cuda.synchronize()
            marks.append((time.perf_counter(), int(allm.shape[0])))

        # keep the last step's per-model metrics for the gather (what the reference logs per chunk)
        orig = ens.step_batch

        def step_and_keep(x):
            losses, aux = orig(x)
            ens._last_loss = losses["loss"]
            ens._last_nnz = aux["c"].count_nonzero(dim=-1).float().mean(dim=-1)
            return losses, aux

        ens.step_batch = step_and_keep
        # the same number of steps from ONE device-resident chunk first (same gather + step code path, nothing
        # streamed): an equally long, equally power-limited run to compare the streamed one with, and its warm-up
        from sparse_coding_b200.train_loop import gather_rows
        steps_per_chunk = (rows + B - 1) // B
        res_chunk = torch.load(os.path.join(folder, "0.pt"), map_location="cpu", mmap=True).to(dev)
        perm = torch.randperm(rows, device=dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for c in range(n_chunks):
            for j in range(steps_per_chunk):
                ens.step_batch(gather_rows(res_chunk, perm[j * B:(j + 1) * B]))
            on_chunk_end(c, 0, ens)
        t_res = time.perf_counter() - t0
        del res_chunk, perm
        marks.clear()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        train_on_chunks(ens, {"device": str(dev), "dict_size": n, "batch_size": B}, folder, outdir, B, ["dict_size"],
                        ["l1_alpha"], chunk_order=list(range(n_chunks)), feed=feed, on_chunk_end=on_chunk_end,
                        save_schedule="none")
        torch.cuda.synchronize()
        t_all = time.perf_counter()
        t_train = marks[-1][0] - t0
        t = torch.tensor([t_train, t_all - marks[-1][0], marks[-1][0] - marks[0][0], t_res], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_train, t_export, t_steady, t_res = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        chunk_seconds = [marks[0][0] - t0] + [marks[i][0] - marks[i - 1][0] for i in range(1, len(marks))]
        total_rows = n_chunks * rows
        out = {
            "value": world * total_rows / t_train, "unit": "activations/s",
            "per_gpu": total_rows / t_train, "chunks": n_chunks, "chunk_shape": [rows, d], "chunk_dtype": "fp16",
            "chunk_store": base, "feed": feed, "steps": n_chunks * steps_per_chunk, "seconds": t_train,
            "ms_per_step": t_train / (n_chunks * steps_per_chunk) * 1e3,
            # chunks 1.. only: the first chunk's load is not hidden behind anything
            "steady_ms_per_step": (t_steady / ((n_chunks - 1) * steps_per_chunk) * 1e3) if n_chunks > 1 else None,
            "export_seconds": t_export, "metric_gather_rows": marks[-1][1], "chunk_seconds": chunk_seconds,
            "resident_chunk_ms_per_step": t_res / (n_chunks * steps_per_chunk) * 1e3,
            "vs_resident_chunk": (t_res / n_chunks) / (t_steady / (n_chunks - 1)) if n_chunks > 1 else None,
            "vs_resident_chunk_note": "steady-state streamed chunk time against an equally long run of the same gather + "
                                      "step loop over ONE device-resident chunk (equal power / clock conditions); "
                                      "vs_resident_pool compares with the short `value` burst instead",
            "includes": "torch.load(mmap) + pinned copy + H2D on a side stream, device-side permutation gather with "
                        "fp16->fp32, step, end-of-chunk all_gather of per-model metrics; excludes chunk synthesis and "
                        "the final learned_dicts.pt export (export_seconds)",
        }
        if resident_ms_per_step:
            out["vs_resident_pool"] = (resident_ms_per_step / out["steady_ms_per_step"]) if out["steady_ms_per_step"] else None
        if info[2] is not None:
            out["chunk_synthesis_seconds"] = info[2]
        return out
    finally:
        shutil.rmtree(outdir, ignore_errors=True)
        if world > 1:
            dist.barrier()
        if rank == 0:
            shutil.rmtree(folder, ignore_errors=True)


# ----------------------------------------------------------------------------------------------------------------
# stock PyTorch on the same GPU (the op sequence the reference launches), as the library comparator
# ----------------------------------------------------------------------------------------------------------------
def stock_torch_gpu(M, d, n, B, dev, pool):
    from oracle import sae_oracle as O
    import sparse_coding_b200 as S
    out = {}
    for name, tf32 in (("fp32", False), ("tf32", True)):
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        try:
            models = [({k: v.to(dev) for k, v in p.items()}, {k: v.to(dev) for k, v in b.items()})
                      for p, b in make_models(S.FunctionalTiedSAE, M, d, n, 0)]
            ref = O.RefPortEnsemble(models, O.SIG_LOSSES["tied"], lr=1e-3)
            for i in range(3):
                ref.step_batch(pool[i % len(pool)])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(5):
                ref.step_batch(pool[i % len(pool)])
            e1.record()
            torch.cuda.synchronize()
            out[name + "_ms_per_step"] = e0.elapsed_time(e1) / 5
            del ref, models
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
        torch.cuda.empty_cache()
    out["what"] = ("oracle port of the reference step (vmap(grad(loss)) + Adam, stock PyTorch ops, cuBLAS) on this GPU, "
                   "3 warm-up + 5 timed steps; 'tf32' = torch.backends.cuda.matmul.allow_tf32 (the reference never sets it)")
    return out


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--bwd-passes", type=int, default=3, choices=[1, 3])
    ap.add_argument("--arith", default="auto", choices=["auto", "bf16x3", "f16f8"],
                    help="operand arithmetic (include/sce.h sce_arith); auto = f16f8 where the shape allows")
    ap.add_argument("--act-precision", default="fp16", choices=["fp16", "fp32"],
                    help="synthetic activation VALUES: fp16-representable (the reference's chunk format; default) or "
                         "arbitrary fp32. The tensors fed to the engine are fp32 either way.")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the informational single-pass-backward run")
    ap.add_argument("--no-stock", action="store_true", help="skip the stock-PyTorch-on-this-GPU comparator")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-4 chunk-streaming extras")
    ap.add_argument("--stream-timeout", type=float, default=240.0, help="watchdog of the config-4 extras, seconds")
    ap.add_argument("--stream-chunks", type=int, default=3)
    ap.add_argument("--stream-rows", type=int, default=1 << 21, help="rows per streamed chunk (reference: 2^21 at d=512)")
    ap.add_argument("--feed", default="per_rank", choices=["per_rank", "broadcast", "both"],
                    help="cfg4_stream: every rank reads/copies its own chunk, or rank 0 reads and NCCL broadcasts")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs and parameters to DIR/<name>.npy (rank 0, engine only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs writes the engine's outputs: use it with --impl engine")
    global ACT_FP16
    ACT_FP16 = args.act_precision == "fp16"

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    out = _StdoutGuard()
    if args.impl == "reference":
        run_reference(args, rank, world, out)
        return

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    import torch.distributed as dist
    import sparse_coding_b200 as S
    from sparse_coding_b200.train_loop import HostBatchPrefetcher

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL announces its version on stdout; stdout must carry exactly one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    stream_only = args.workload == "cfg4_stream"
    M, d, n, B, desc = WORKLOADS[args.workload]
    K, W = args.steps, max(args.warmup, 3)
    topk = args.workload in ("cfg3", "cfg3g")

    # every rank owns its own shard of the sweep: same shapes, different seeds (model-axis sharding)
    sig = S.TopKEncoder if topk else S.FunctionalTiedSAE
    if args.workload == "cfg3":
        # the three shape groups of config 3 are three stacked ensembles stepped one after the other on the same batch
        # (the reference builds one ensemble per dict size, big_sweep_experiments.py:232-262)
        enss = [S.FunctionalEnsemble(make_models(sig, m, d, nn, seed=rank * 10 + gi), sig, S.adam, {"lr": 1e-3}, device=dev,
                                     bwd_passes=args.bwd_passes, arith=args.arith, no_stacking=True)
                for gi, (nn, m) in enumerate(CFG3_GROUPS)]
    else:
        enss = [S.FunctionalEnsemble(make_models(sig, M, d, n, seed=rank), sig, S.adam, {"lr": 1e-3}, device=dev,
                                     bwd_passes=args.bwd_passes, arith=args.arith)]
    ens = enss[0]
    n_pool = 8
    host = synth_batches(n_pool, B, d, seed=1000, pin=True)        # identical stream on every rank
    pool = [x.to(dev) for x in host]                                 # resident copies for the device-timed run

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_all(x):
        """(losses, aux) of every ensemble, in order."""
        return [e.step_batch(x) for e in enss]

    # ---------------- device-resident run: `value` (nothing but step_batch calls between the two events)
    windows = {}
    for i in range(W):
        step_all(pool[i % n_pool])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.time()
    e0.record()
    for i in range(K):
        results = step_all(pool[i % n_pool])
    e1.record()
    barrier()
    windows["value"] = (t_begin, time.time())
    ms = e0.elapsed_time(e1)
    launches = K * sum(e.gpu_launches_last_call() for e in enss)
    final_loss = results[-1][0]["loss"].detach().clone()
    arith_resolved = ens.resolved_arith()
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(args.dump_outputs, enss, results)
    del results

    # ---------------- per-phase device times: a separate short loop with libsce's events switched on
    for e in enss:
        e.profile_begin()
    t_begin = time.time()
    n_prof = min(max(K, 10), 40)
    for i in range(n_prof):
        step_all(pool[i % n_pool])
    phase_list = [e.profile_end() for e in enss]
    windows["phases"] = (t_begin, time.time())
    steps_prof = max(phase_list[0]["steps"], 1)
    per_phase = {k: sum(p[k] for p in phase_list) / steps_prof for k in phase_list[0] if k != "steps"}

    # ---------------- end-to-end runs through the public API with host batches: `e2e`
    barrier()
    h2d = B * d * 4

    def e2e_loop(prefetch):
        evs = []
        src = HostBatchPrefetcher((host[i % n_pool] for i in range(K + 2)), dev) if prefetch else \
            (host[i % n_pool] for i in range(K + 2))
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        got = nnz = None
        for i, x in enumerate(src):
            if i == 2:
                barrier()
                e2.record()
            if not prefetch and i >= 2:
                a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                a.record()
                x = x.to(dev, non_blocking=True)                          # pinned host -> device on the compute stream
                b.record()
            losses, aux = step_all(x)[-1]
            if not prefetch and i >= 2:
                c.record()
                evs.append((a, b, c))
            got = {k: v.cpu() for k, v in losses.items()}                 # D2H of the step's result, every step
            nnz = aux["c"].count_nonzero(dim=-1).float().mean(dim=-1).cpu()
        e3.record()
        barrier()
        d2h = sum(v.numel() * 4 for v in got.values()) + nnz.numel() * 4
        split = None
        if evs:
            split = {"h2d_ms": float(np.mean([a.elapsed_time(b) for a, b, _ in evs])),
                     "step_device_ms": float(np.mean([b.elapsed_time(c) for _, b, c in evs]))}
        return e2.elapsed_time(e3), d2h, split

    t_begin = time.time()
    ms_e2e, d2h, _ = e2e_loop(prefetch=True)
    windows["e2e"] = (t_begin, time.time())
    ms_serial, _, serial_split = e2e_loop(prefetch=False)

    # ---------------- informational: the same workload with single-pass bf16 backward GEMMs (NOT the headline)
    ms_alt = float("nan")
    if world == 1 and args.bwd_passes == 3 and args.workload == "cfg2" and not args.no_alt:
        alt = S.FunctionalEnsemble(make_models(S.FunctionalTiedSAE, M, d, n, seed=rank), S.FunctionalTiedSAE, S.adam,
                                   {"lr": 1e-3}, device=dev, bwd_passes=1, arith=args.arith)
        for i in range(3):
            alt.step_batch(pool[i % len(pool)])
        e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e4.record()
        for i in range(K):
            alt.step_batch(pool[i % len(pool)])
        e5.record()
        barrier()
        ms_alt = e4.elapsed_time(e5)
        del alt

    t = torch.tensor([ms, ms_e2e, ms_serial], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # end-of-chunk metric gather (the only collective on this path): every model's final loss to every rank
        gathered = [torch.empty_like(final_loss) for _ in range(world)]
        dist.all_gather(gathered, final_loss)
        final_loss = torch.cat(gathered)
    ms, ms_e2e, ms_serial = float(t[0]), float(t[1]), float(t[2])
    clocks = sampler.stop(windows) if rank == 0 else None

    line = None
    if rank == 0:
        pk = peaks()
        arith = arith_resolved
        # tensor work issued per fp32-equivalent GEMM, in bf16-pass equivalents: three kind::f16 passes, or one
        # kind::f16 pass + two kind::f8f6f4 passes at twice the rate
        full_passes = 3 if arith == "bf16x3" else 2
        bwd_eq = full_passes if args.bwd_passes == 3 else 1
        # f16f8 + fp16-representable activations: x has no residual plane, so the x.l8 * W.h8 term of encode and the
        # dz.h8 * x.l8 term of the dz^T x half of dW are skipped on the device (one 8-bit pass = 1/2 pass equivalent)
        x_skip = arith == "f16f8" and ACT_FP16
        enc_eq = full_passes - (0.5 if x_skip else 0.0)
        dw_eq = (bwd_eq - (0.25 if x_skip else 0.0)) if args.bwd_passes == 3 else 1
        arith_text = {
            "bf16x3": "fp32 parameters/moments/accumulation; every GEMM operand is an exact-to-2^-17 (hi, lo) bf16 pair "
                      "and every product 3 tensor-core passes (hi*hi + hi*lo + lo*hi)",
            "f16f8": "fp32 parameters/moments/accumulation; every GEMM operand is an fp16 plane plus two e5m2 planes "
                     "(value, scaled residual); every product = one kind::f16 pass (h*h) + two kind::f8f6f4 passes for "
                     "the cross terms (2 bf16-pass equivalents), rescaled in the accumulator",
        }[arith] + "; parity <= 1e-4 rel vs the fp32 reference on x_hat and losses (tests/test_scale_parity_gpu.py at this size)"
        value = world * B * K / (ms * 1e-3)
        e2e_value = world * B * K / (ms_e2e * 1e-3)
        if args.workload == "cfg3":
            mnd = sum(m * nn for nn, m in CFG3_GROUPS) * d         # sum over models of n * d
        else:
            mnd = M * n * d
        dw_ms = per_phase["dw"]
        alg_flops_dw = 4.0 * B * mnd                  # dW = dz^T x + c^T g: two GEMMs of 2*B*n*d per model
        achieved = alg_flops_dw / (dw_ms * 1e-3) / 1e12 if dw_ms > 0 else None
        step_flops = 10.0 * B * mnd
        gemms = {}
        for ph, units, passes in (("encode", 1, enc_eq), ("decode", 1, full_passes), ("dcode", 1, bwd_eq), ("dw", 2, dw_eq)):
            if per_phase[ph] > 0:
                alg = units * 2.0 * B * mnd / (per_phase[ph] * 1e-3) / 1e12
                gemms[ph] = {"ms": per_phase[ph], "alg_tflops": alg, "frac": alg / pk["bf16_tflops"],
                             "issued_tflops": alg * passes, "frac_of_peak_issued": alg * passes / pk["bf16_tflops"]}
        line = {
            "metric": METRIC, "value": value, "unit": "activations/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32",
            "data": "synthetic (sparse mixture + noise); values " +
                    ("rounded to fp16 as the reference caches activations (activation_dataset.py:404-412), "
                     if ACT_FP16 else "arbitrary fp32, ") + "fed as fp32 tensors",
            "config": {"workload": f"{args.workload}: {desc}", "models_per_gpu": M,
                       "activation_values": args.act_precision, "d_model": d, "dict_size": n,
                       "batch": B, "parallelism": f"ensemble-shard x{world}" if world > 1 else "single GPU",
                       "arith": arith, "arithmetic": arith_text, "pass_equivalents_per_gemm": full_passes,
                       "x_residual_term_skipped": bool(x_skip),
                       "fwd_passes": 3, "bwd_passes": args.bwd_passes,
                       "adam_count_mode": "frozen_t1 (the reference's step_batch drops torchopt's incremented count, "
                                          "ensemble.py:185-189 — an unverified reading, torchopt is not installable here; "
                                          "'standard' is selectable and costs the same)",
                       "l2": "per-step working set (code + code-gradient, 4.3 GB) and the 8-batch input pool "
                             "(134 MB) both exceed the 126 MB L2; no explicit flush",
                       "timed_loop": "value: step_batch calls only (no profiling events, no host reads)"},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "activations/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / K,
                    "how": "pinned host batches through train_loop.HostBatchPrefetcher (copy of batch i+1 on a side "
                           "stream during step i) -> step_batch -> .cpu() of every loss term and of the mean nnz, every step",
                    "serial": dict({"value": world * B * K / (ms_serial * 1e-3), "ms_per_step": ms_serial / K,
                                    "how": "same loop, H2D on the compute stream (step_batch(host_tensor)); the split is "
                                           "measured with CUDA events around the copy and the step: a step between two "
                                           "host synchronisations runs on a cooler, higher-clocked GPU than the "
                                           "back-to-back steps of `value`"}, **(serial_split or {}))},
            "roofline": {"bound": "tensor", "kernel": "gemm_split_kernel<EpiStoreF32,MN,MN> (weight gradient)",
                         "achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": achieved / pk["bf16_tflops"] if achieved else None, "traffic": None,
                         "peak_source": pk["source"], "alg_flops_per_launch": alg_flops_dw,
                         "ms_per_launch": dw_ms,
                         "issued_tflops": alg_flops_dw * dw_eq / (dw_ms * 1e-3) / 1e12 if dw_ms > 0 else None,
                         "issued_note": f"{dw_eq} bf16-pass equivalents per fp32 FLOP of this kernel ({arith}"
                                        + (", x residual term skipped" if x_skip else "") + f"): frac <= 1/{dw_eq} x "
                                        "(tensor-pipe utilisation = issued_tflops / peak; `peak` is cuBLAS's sustained "
                                        "bf16 rate under the power cap, which kind::f8f6f4 passes can exceed)",
                         "step_alg_tflops": step_flops / (ms / K * 1e-3) / 1e12,
                         "step_frac": step_flops / (ms / K * 1e-3) / 1e12 / pk["bf16_tflops"],
                         "per_gemm_frac": {k: v["frac"] for k, v in gemms.items()}},
            "phases_ms": per_phase,
            "phases_note": f"separate loop of {steps_prof} steps with libsce's per-phase events on; their sum is "
                           f"{sum(per_phase.values()):.3f} ms",
            # every GEMM phase against the same peak: algorithmic (fp32-equivalent) and issued (x passes) TFLOP/s
            "gemms": gemms,
            "final_loss_mean": float(final_loss.mean()),
        }
        if dumped is not None:
            line["dump_outputs"] = {"dir": args.dump_outputs, "shapes": dumped,
                                    "what": f"step {W + K} (the last of `value`); axis 1 sampled where an array "
                                            "exceeds its share of 60 MB"}
        tr = (ncu_traffic() or {}).get(arith)
        if tr and args.workload == "cfg2":
            line["roofline"]["traffic"] = tr["dw_dram_bytes_per_launch"]
            line["roofline"]["traffic_source"] = tr["source"]
            # dz and c at 4 B / element (3 B for dz when x's residual term is skipped: its h8 plane is not read) + dW
            line["roofline"]["alg_bytes_per_launch"] = (8.0 - (1.0 if x_skip else 0.0)) * M * B * n + 4.0 * M * n * d
            if "dram_bytes_per_step" in tr:
                line["roofline"]["dram_bytes_per_step"] = tr["dram_bytes_per_step"]
                line["roofline"]["dram_bytes_per_kernel"] = tr.get("dram_bytes_per_kernel")
                line["roofline"]["alg_bytes_per_step"] = 4.0 * B * d + 24.0 * M * n * d
        if ms_alt == ms_alt:
            line["alt_precision"] = {"note": "informational only: backward GEMMs on the 16-bit plane alone (bwd_passes=1); "
                                             "forward, losses and x̂ unchanged; FVU/L0 parity of this mode at this size: "
                                             "tests/test_scale_parity_gpu.py::test_training_quality_at_config2_scale",
                                     "value": B * K / (ms_alt * 1e-3), "ms_per_step": ms_alt / K}
        if world == 1 and not args.no_stock and args.workload in ("cfg2", "cfg1"):
            try:
                line["stock_torch_gpu"] = stock_torch_gpu(M, d, n, B, dev, pool)
                line["stock_torch_gpu"]["speedup_vs_fp32"] = line["stock_torch_gpu"]["fp32_ms_per_step"] / (ms / K)
                line["stock_torch_gpu"]["speedup_vs_tf32"] = line["stock_torch_gpu"]["tf32_ms_per_step"] / (ms / K)
            except Exception as exc:
                line["stock_torch_gpu"] = {"failed": f"{type(exc).__name__}: {exc}"}
        if world == 1 and not args.no_cpu_baseline and n is not None and not topk:
            rate, sample, cores, dt, Bs = cpu_reference_rate(M, d, n, B, budget_s=45.0, steps=1, warmup=0)
            line["cpu_baseline"] = {"value": rate, "unit": "activations/s", "cores": cores, "kind": "port",
                                    "sample": sample, "same_config": bool(Bs == B)}

    # ---------------- config 4's data path (all ranks take part). It runs AFTER the line is complete and under a
    # watchdog: if a rank fails or a collective hangs in here, rank 0 still prints the line (without these extras).
    stream = None
    if (args.workload == "cfg2" and not args.no_stream) or stream_only:
        import threading

        def bail():
            if rank == 0 and line is not None:
                line["cfg4_stream"] = {"failed": f"no result within {args.stream_timeout} s (watchdog)"}
                out.emit(line)
            os._exit(0)

        timer = threading.Timer(args.stream_timeout, bail)
        timer.daemon = True
        timer.start()
        for e in enss:
            e._destroy_plan()
        del pool
        torch.cuda.empty_cache()
        feeds = ["per_rank", "broadcast"] if (args.feed == "both" and world > 1) else \
            [args.feed if (world > 1 or args.feed == "per_rank") and args.feed != "both" else "per_rank"]
        stream = {}
        for feed in feeds:
            try:
                stream[feed] = run_stream(S, dist, rank, world, dev, M, d, n, B, args.stream_chunks, args.stream_rows, feed,
                                          ms / K)
            except Exception as exc:                                      # extras must never cost the headline line
                stream[feed] = {"failed": f"{type(exc).__name__}: {exc}"}
        timer.cancel()

    if rank == 0:
        if stream is not None:
            line["cfg4_stream"] = stream[next(iter(stream))] if len(stream) == 1 else stream
        if stream_only and stream:
            first = stream[next(iter(stream))]
            if "value" in first:                       # this workload's own metric: the streamed rate
                line["resident_pool"] = {"value": line["value"], "ms_per_step": line["ms_per_step"]}
                line["value"], line["ms_per_step"] = first["value"], first["ms_per_step"]
                line["e2e"] = {"value": first["value"], "unit": "activations/s",
                               "h2d_bytes_per_step": int(B * d * 2), "d2h_bytes_per_step": 0,
                               "how": "the streamed run IS end to end: chunk bytes cross PCIe once (fp16), batches are "
                                      "gathered on the device"}
        out.emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
