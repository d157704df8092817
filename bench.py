#!/usr/bin/env python
"""Benchmark of the legacy per-image scoring pass (BASELINE.json metric: images/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of B synthetic 24 MP frames per GPU:
technical metrics (csrc/tech_stats.cu) + perceptual hash (csrc/phash.cu) + CLIP preprocess
(csrc/preprocess.cu, csrc/resample_tc.cu) + ViT-L/14 tower, aesthetic head and tag similarities
(csrc/gemm.cu, csrc/attention_tc.cu, csrc/vit.cu).  After the K steps the duplicate-grouping stage
runs ONCE over everything scored (all-gather across ranks, cosine pairs csrc/gemm.cu +
csrc/similarity.cu, Hamming pairs csrc/hamming.cu) inside the timed region — BASELINE configs[4].
`value` is the whole-job rate with the frames already resident in HBM; `e2e` is the same work
through the reference-shaped call (`BatchProcessor.process_items_streamed`: pinned host frames in,
complete result dicts out; H2D, D2H and the host-side dict building inside the timed region) beside
a copy-only ceiling.  `configs` carries short device-timed legs for BASELINE configs[1..3].
Prints ONE JSON line on rank 0.  `--impl reference` times the reference's CPU path (oracle port;
/root/reference does not exist on the GPU box) on a bounded sample instead.
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

H, W = 4000, 6000
GFLOP_PER_IMAGE = 162.0          # SURVEY.md §8 a12: ViT-L/14 224 px incl. attention and patch embedding
GEMM_GFLOP_PER_IMAGE = 24 * (1.617 + 0.539 + 4.312) + 0.308   # the part the tcgen05 GEMM kernel executes
TECH_BYTES_PER_IMAGE = 3 * H * W


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=128, help="24 MP frames per GPU per step")
    ap.add_argument("--impl", default="facet_b200", choices=["facet_b200", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--clock-period-ms", type=float, default=50.0, help="NVML sampling period during the timed region (0 = off)")
    ap.add_argument("--no-configs", action="store_true", help="skip the short legs for BASELINE configs[1..3]")
    ap.add_argument("--sim-rows", type=int, default=262144, help="embeddings per GPU in the similarity leg (configs[3])")
    ap.add_argument("--e2e-chunk", type=int, default=16, help="frames per staging buffer of the streamed e2e path")
    ap.add_argument("--no-e2e-jpeg", action="store_true", help="skip the e2e leg that starts from JPEG file bytes")
    ap.add_argument("--no-e2e-side", action="store_true", help="skip the e2e leg with leading-lines scores and thumbnails")
    ap.add_argument("--jpeg-restart-blocks", type=int, default=8, help="restart interval (MCUs) of the bench's JPEG streams")
    ap.add_argument("--e2e-jpeg-chunk", type=int, default=32, help="streams per decode launch in the JPEG e2e leg")
    ap.add_argument("--e2e-vit-batch", type=int, default=64, help="frames per ViT launch of the streamed e2e path")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step and the grouping stage computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "facet_b200":
        ap.error("--dump-outputs records the device path (--impl facet_b200)")
    return args


DUMP_BYTES = 64 * 1000 * 1000      # all files of --dump-outputs together


def host_outputs(out, pairs, sims, hpairs):
    """The device results of one step and of the grouping stage as float32 / float64 host arrays.  Integers become
    float64 (exact: the technical sums of a 24 MP frame stay below 2^53); the 64-bit pHash becomes one 0/1 column per
    bit, lowest first.  Pairs index the rows of all timed steps (step k, frame b -> k * batch + b) and are sorted."""
    import numpy as np
    arrays = {}
    for name, t in out.items():
        if t is None:
            continue
        a = t.cpu().numpy()
        if name == "phash":
            name, a = "phash_bits", (a.view(np.uint64)[:, None] >> np.arange(64, dtype=np.uint64)) & 1
        arrays[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    cp = np.column_stack([pairs.cpu().numpy().astype(np.float64), sims.cpu().numpy().astype(np.float64)])
    arrays["cosine_pairs"] = cp[np.lexsort((cp[:, 1], cp[:, 0]))]                 # rows (i, j, cosine)
    hp = hpairs.cpu().numpy().astype(np.float64)
    arrays["hamming_pairs"] = hp[np.lexsort((hp[:, 1], hp[:, 0]))]               # rows (i, j)
    return arrays


def dump_outputs(out_dir, arrays):
    """Writes out_dir/<name>.npy for every array, DUMP_BYTES in all: the smaller arrays are written whole first, and an
    array that does not fit what is left keeps a seeded sample of its rows, in their order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    names = sorted(arrays, key=lambda k: arrays[k].nbytes)
    for i, name in enumerate(names):
        a = arrays[name]
        share = left // (len(names) - i) - 4096          # room for the .npy header
        if a.nbytes > share:
            keep = np.random.default_rng(0).choice(len(a), share // (a.nbytes // len(a)), replace=False)
            a = a[np.sort(keep)]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        left -= os.path.getsize(path)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "MEASURED_PEAKS.json (sustained bf16, copy HBM)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "source": "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"}


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  NVML is queried in-process
    (nvidia_ml_py): one clock read + one reasons read per sample cost microseconds, whereas an `nvidia-smi -lms`
    poller stalls the driver for milliseconds per sample and slows every launch of the step it lands in
    (measured: +20 % on a 10-step run).  Falls back to nvidia-smi if NVML is not importable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_s=0.02):
        self.idx = gpu_index
        self.period = period_s
        self.samples = []          # (sm_mhz, reasons bitmask)
        self.max_mhz = None
        self.proc = None
        self.lines = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "250"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                reasons = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.samples.append((mhz, reasons))
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def reset(self):
        """Drop what was sampled so far (called right before the timed region starts)."""
        self.samples = []

    def _read_smi(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        self.stop_flag.set()
        if self.nvml is not None:
            self.thread.join(timeout=2)
            n = self.nvml
            # every bit NVML defines (nvml.h nvmlClocksEventReason*), so that a clock below the maximum always comes with its reason
            names = {"gpu_idle": 0x1, "applications_clocks_setting": 0x2, "sw_power_cap": 0x4, "hw_slowdown": 0x8, "sync_boost": 0x10,
                     "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake_slowdown": 0x80,
                     "display_clock_setting": 0x100}
            sm = sorted(s[0] for s in self.samples)
            mask = 0
            for _, r in self.samples:
                mask |= r
            reasons = sorted(k for k, bit in names.items() if mask & bit)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                    "sm_max_mhz": self.max_mhz, "reasons": reasons, "reasons_mask": mask, "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                mx = float(parts[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # median of the upper half: samples taken while the GPU was busy
        busy = sm[len(sm) // 2:] if sm else []
        med = busy[len(busy) // 2] if busy else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def make_pool(n, seed, device):
    """n distinct device-resident 24 MP BGR frames (gradients + texture + noise; 1 in 8 pure noise, 1 in 8 flat)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    out = torch.empty((n, H, W, 3), dtype=torch.uint8, device=device)
    yy = torch.linspace(0, 1, H, device=device)[:, None, None]
    xx = torch.linspace(0, 1, W, device=device)[None, :, None]
    for i in range(n):
        kind = i % 8
        if kind == 6:
            out[i] = torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, device=device, generator=g)
            continue
        ph = torch.rand((1, 1, 3), device=device, generator=g) * 6.28
        fr = 1 + 5 * torch.rand((1, 1, 3), device=device, generator=g)
        base = 0.5 + 0.25 * torch.sin(fr * 6.28 * xx + ph) + 0.22 * torch.cos(fr * 4.1 * yy + 2 * ph)
        if kind == 3:
            base = torch.round(base * 5) / 5
        gain = 0.6 + 0.5 * float(torch.rand(1, device=device, generator=g))
        sigma = (0.0, 2.0, 4.0, 1.0, 6.0, 3.0, 0.0, 1.5)[kind]
        noise = torch.randn((H, W, 3), device=device, generator=g) * sigma
        out[i] = (base * 255 * gain + noise).clamp(0, 255).to(torch.uint8)
        if kind == 0:
            out[i, :, :, 0] = out[i, :, :, 1]
            out[i, :, :, 2] = out[i, :, :, 1]
    return out


CPU_SAMPLE_FRAMES = 3            # frames per CPU step: same frames, same ViT batch in `--impl reference` and `cpu_baseline`


def cpu_sample_frames():
    """The bounded CPU sample: three frames of the workload's size from the host-side generator (facet_b200/synth.py)."""
    from facet_b200.synth import synth_image_bgr
    return [synth_image_bgr(2000 + i, H, W) for i in range(CPU_SAMPLE_FRAMES)]


def cpu_arm():
    """(ref_analyzers or None, kind, description).  oracle/_ref holds the reference's own analyzers/technical.py +
    image_cache.py when oracle/build_ref.py ran in the build container; the CLIP tower is the oracle's fp32 restatement
    either way (open_clip is third-party and not installable here)."""
    from oracle import build_ref
    ref = build_ref.load()
    if ref is not None:
        return ref, "reference", ("technical metrics = the reference's own analyzers/technical.py + image_cache.py (oracle/_ref, "
                                  "unmodified); pHash / PIL preprocess / fp32 torch-CPU ViT-L/14 = oracle port (imagehash, open_clip absent)")
    return None, "port", "oracle/cpu_port.py (cv2+NumPy+SciPy technical metrics, PIL preprocess, fp32 torch-CPU ViT-L/14)"


def run_reference(args, rank, world):
    """CPU arm: the reference's CPU path timed on the host cores (oracle/_ref analyzers when present, else the port:
    the same cv2 / NumPy / SciPy / PIL / torch-CPU calls in the order of processing/batch_processor.py:198-233).
    One step = CPU_SAMPLE_FRAMES 24 MP frames, batched through the tower, + the cosine grouping of what was scored so far."""
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm is to use every host thread it can, so the BLAS / OpenMP
    # pools are sized before NumPy / SciPy / torch are imported (nothing above this line imports them)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = str(cores)
    import numpy as np
    import torch
    from facet_b200.models.clip_vit import random_state_dict
    from facet_b200.synth import synth_embeddings
    from oracle import cpu_port, grouping
    torch.set_num_threads(cores)
    try:
        import cv2
        cv2.setNumThreads(cores)
    except ImportError:
        pass
    sd = random_state_dict(0)
    tags = torch.from_numpy(synth_embeddings(240, seed=7, cluster_fraction=0.0))
    ref, kind, desc = cpu_arm()
    frames = cpu_sample_frames()
    embs = []

    def step():
        _, vit = cpu_port.score_images_cpu(frames, sd, tags, ref_analyzers=ref)
        embs.append(vit["embedding"].numpy())
        grouping.cosine_pairs(np.concatenate(embs[-64:], axis=0), 0.9)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = args.steps * len(frames) / dt
    line = {
        "impl": "reference", "metric": "images/sec", "value": val, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.batch),
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": f"{args.steps} steps x {len(frames)} synthetic 24 MP frames (seeds 2000..) per step, ViT batch "
                                   f"{len(frames)}; {desc}"},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(batch):
    return {"workload": "full legacy scoring pass on synthetic 6000x4000 (24 MP) BGR frames: technical metrics + pHash + CLIP "
                        "preprocess + ViT-L/14 224px + MLP aesthetic + tag similarities per image, then ONE duplicate-grouping "
                        "stage (all-gather, cosine and Hamming pairs) over everything scored (BASELINE.json configs[4], per-GPU share)",
            "image": [H, W, 3], "batch_per_gpu": batch, "parallelism": "data-parallel, one rank per GPU",
            "l2": "inputs larger than L2 (pool of batch x 72 MB frames per step)", "weights": "random-init ViT-L/14 (seed 0)",
            "precision": "ViT GEMM operands fp16 (the reference's CUDA precision, `self.model.half()`, scorer.py:515; NOT the bf16 "
                         "BASELINE configs[2] names: bf16 operands miss the 0.01 aesthetic bound, tests/test_gpu_vit.py), fp32 "
                         "accumulate and residual stream; technical metrics / preprocess exact integers"}


def traffic_record():
    """DRAM traffic per launch of the two roofline kernels, from ncu --set full captures (profiles/traffic.json names
    the capture files and their sha256).  Absent file -> None: nothing is hard-coded here."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        return json.load(f)


def device_embeddings(n, dim, seed, device, dup_fraction=0.15):
    """[n, dim] float32 L2-normalised rows on the device with planted near-duplicates (cosine ~0.95)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    e = torch.randn((n, dim), device=device, generator=g)
    e = torch.nn.functional.normalize(e, dim=-1)
    nd = int(n * dup_fraction)
    if nd:
        dst = torch.randperm(n, device=device, generator=g)[:nd]
        src = (torch.rand(nd, device=device, generator=g) * n).long().clamp_(max=n - 1)
        v = e[src] + 0.012 * torch.randn((nd, dim), device=device, generator=g)
        e[dst] = torch.nn.functional.normalize(v, dim=-1)
    return e.contiguous()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from facet_b200 import _lib, ops
    from facet_b200.models.clip_vit import random_state_dict
    from facet_b200.processing.batch_processor import BatchProcessor
    from facet_b200.processing.scorer import Facet
    from facet_b200.synth import synth_embeddings
    from facet_b200.utils.duplicate import all_gather_embeddings, cosine_pairs_sharded

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    from facet_b200.processing.pipeline import bind_to_gpu_numa_node
    orig_affinity = os.sched_getaffinity(0)
    numa_node = bind_to_gpu_numa_node(local_rank)      # pinned e2e buffers local to the GPU's PCIe root
    if world > 1:
        # stdout must carry exactly one JSON line: send NCCL's start-up banner ("NCCL version ...", printed on
        # stdout when the communicator is created) to stderr by redirecting fd 1 during initialisation
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            warm = torch.zeros(1, device=device)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.load()

    B, K = args.batch, args.steps
    tags = synth_embeddings(240, seed=7, cluster_fraction=0.0)
    scorer = Facet(random_state_dict(0), text_embeddings=tags, tag_names=[f"tag{i // 4}" for i in range(240)], device=device)
    pool = make_pool(B, seed=2000 + 17 * rank, device=device)
    emb_all = torch.empty((K * B, 768), dtype=torch.float32, device=device)
    hash_all = torch.empty((K * B,), dtype=torch.int64, device=device)
    torch.cuda.synchronize()

    def step(k):
        """One batch of B frames through the per-image pass; embeddings / hashes are kept for the grouping stage.
        No communication, no host synchronisation."""
        out = scorer.score_images_device(pool)                      # technical + pHash + preprocess + ViT/heads/tags
        emb_all[k * B:(k + 1) * B].copy_(out["embedding"])
        hash_all[k * B:(k + 1) * B].copy_(out["phash"])
        return out

    def grouping(emb, hashes):
        """The duplicate-grouping stage over everything scored (configs[4]): ONE all-gather of the embedding shards and of
        the hashes, then every rank scans its balanced share of the pair triangle."""
        pairs, sims = cosine_pairs_sharded(emb, 0.90)              # bf16 gather -> scan, f32 gather overlapped -> recheck
        h = all_gather_embeddings(hashes.view(-1, 1)).view(-1) if world > 1 else hashes
        hp = ops.hamming_pairs(h, 6, part=rank, nparts=world)      # duplicate rule of utils/duplicate.py:94-119
        return pairs, sims, hp

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(max(args.warmup, 3)):
        step(k % K)
    grouping(emb_all, hash_all)
    barrier()
    # ---- timed region: K steps + the grouping stage, CUDA events on the launching stream -------------------
    launches0 = int(lib.fb_launch_count())
    # one sampler per node (rank 0's GPU): concurrent pollers slow every rank's launches
    sampler = ClockSampler(local_rank, period_s=max(args.clock_period_ms, 1.0) * 1e-3)
    if rank == 0 and args.clock_period_ms > 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    e0, e1, eg = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    sampler.reset()
    e0.record()
    for k in range(K):
        last = step(k)
    eg.record()
    pairs, sims, hpairs = grouping(emb_all, hash_all)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    ms_group = eg.elapsed_time(e1)
    clocks = sampler.stop()
    launches = int(lib.fb_launch_count()) - launches0
    if world > 1:
        t = torch.tensor([ms_total, ms_group], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_group = (float(v) for v in t.tolist())
    ms_step = ms_total / K
    value = world * B * K / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, host_outputs(last, pairs, sims, hpairs))

    # ---- per-kernel device times of the SAME work: the library records a CUDA-event pair around each of its
    # launches on the launching stream (fb_profile_*); K more steps + grouping, identical inputs ----------------
    _lib.profile_enable(True)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for k in range(K):
        step(k)
    grouping(emb_all, hash_all)
    pe1.record()
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    ms_step_profiled = pe0.elapsed_time(pe1) / K
    # the same K steps with the LayerNorm fold switched off (49 separate LayerNorm launches, plain GEMM epilogues): the GEMM
    # figure of the fold carries the LayerNorm work, this one is the GEMM alone
    unfused = None
    if not os.environ.get("FB_VIT_NO_LN_FOLD"):
        os.environ["FB_VIT_NO_LN_FOLD"] = "1"
        try:
            step(0)
            _lib.profile_enable(True)
            qe0, qe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            qe0.record()
            for k in range(K):
                step(k)
            qe1.record()
            prof_u = _lib.profile_read()
            _lib.profile_enable(False)
            unfused = {"step_ms_with_event_pairs": qe0.elapsed_time(qe1) / K, "gemm_ms_per_step": prof_u["gemm"][0] / K,
                       "layernorm_ms_per_step": prof_u["layernorm"][0] / K, "layernorm_launches_per_step": prof_u["layernorm"][1] / K}
        finally:
            del os.environ["FB_VIT_NO_LN_FOLD"]
    per_step = {k: (v[0] / K, v[1] / K) for k, v in prof.items() if v[1]}
    ms_tech, ms_pre = per_step["technical"][0], per_step["preprocess"][0]
    ms_phash = per_step.get("other", (0.0, 0))[0]
    ms_vit = sum(per_step[k][0] for k in ("im2col", "gemm", "layernorm", "attention", "vit_tail") if k in per_step)
    gemm_ms, gemm_launches = per_step["gemm"]
    stages = {"technical_ms": ms_tech, "phash_ms": ms_phash, "preprocess_ms": ms_pre, "vit_ms": ms_vit,
              "grouping_ms_total": ms_group, "grouping_rows": world * K * B,
              "kernel_ms_per_step": {k: round(v[0], 4) for k, v in per_step.items()},
              "launches_per_step": {k: round(v[1], 2) for k, v in per_step.items()},
              "step_ms_with_event_pairs": ms_step_profiled,
              "technical_gbs": B * TECH_BYTES_PER_IMAGE / (ms_tech * 1e-3) / 1e9,
              "vit_tflops": B * GFLOP_PER_IMAGE * 1e9 / (ms_vit * 1e-3) / 1e12}
    peaks = measured_peaks()
    gemm_tflops = B * GEMM_GFLOP_PER_IMAGE * 1e9 / (gemm_ms * 1e-3) / 1e12
    tr = traffic_record()
    roofline = {"bound": "tensor", "kernel": f"gemm_bf16_kernel (tcgen05), {gemm_launches:.0f} launches per step",
                "achieved": gemm_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": gemm_tflops / peaks["bf16_tflops"],
                "traffic": (tr["gemm"]["dram_bytes_per_layer_at_batch_128"] * 24 * B / 128) if tr else None,
                "traffic_source": tr["gemm"]["source"] if tr else None,
                "algorithmic_flops_per_step": B * GEMM_GFLOP_PER_IMAGE * 1e9, "kernel_ms_per_step": gemm_ms,
                "timing": "CUDA-event pairs around every launch of the kernel, on the launching stream, over K steps",
                "peak_source": peaks["source"], "share_of_step": gemm_ms / ms_step_profiled,
                "note": "the GEMM epilogues carry the LayerNorm work of the tower (fold: 16-bit copy of the residual stream + row sums out of "
                        "the residual epilogues, normalisation finished in the QKV / fc epilogues; 1 LayerNorm launch per step instead of 49)",
                "with_separate_layernorm": None if unfused is None else dict(
                    unfused, achieved=B * GEMM_GFLOP_PER_IMAGE * 1e9 / (unfused["gemm_ms_per_step"] * 1e-3) / 1e12,
                    frac=B * GEMM_GFLOP_PER_IMAGE * 1e9 / (unfused["gemm_ms_per_step"] * 1e-3) / 1e12 / peaks["bf16_tflops"],
                    note="same K steps with FB_VIT_NO_LN_FOLD=1: plain GEMM epilogues + 49 layernorm_kernel launches"),
                "technical_kernel": {"bound": "hbm", "achieved": stages["technical_gbs"], "peak": peaks["hbm_gbs"],
                                     "unit": "GB/s", "frac": stages["technical_gbs"] / peaks["hbm_gbs"],
                                     "algorithmic_bytes_per_step": B * TECH_BYTES_PER_IMAGE,
                                     # SURVEY 8(d) counts the frame read only; in the step the same launch also WRITES the
                                     # Pillow luma plane the pHash pass consumes (H W bytes / image), so `traffic` is to be
                                     # held against read + write, not against the read alone
                                     "algorithmic_bytes_with_outputs_per_step": B * (TECH_BYTES_PER_IMAGE + H * W),
                                     "achieved_with_outputs": B * (TECH_BYTES_PER_IMAGE + H * W) / (ms_tech * 1e-3) / 1e9,
                                     "frac_with_outputs": B * (TECH_BYTES_PER_IMAGE + H * W) / (ms_tech * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                     "traffic": (tr["technical"]["dram_bytes_per_frame"] * B) if tr else None,
                                     "traffic_source": tr["technical"]["source"] if tr else None}}

    # ---- the other BASELINE configs, each a short device-timed leg (best of 3) ------------------------------
    def best_ms(fn, reps=3):
        best = 1e30
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b))
        return best

    configs = {}
    if not args.no_configs:
        # configs[1]: technical metrics only, 64-frame pool (4.6 GB >> L2), no luma plane
        n1 = min(64, B)
        ops.tech_stats_raw(pool[:n1])
        ms1 = best_ms(lambda: ops.tech_stats_raw(pool[:n1]))
        configs["tech_only"] = {"baseline_config": 1, "frames_per_launch": n1, "ms": ms1, "images_per_s_per_gpu": n1 / (ms1 * 1e-3),
                                "GB_s": n1 * TECH_BYTES_PER_IMAGE / (ms1 * 1e-3) / 1e9,
                                "frac_of_measured_hbm": n1 * TECH_BYTES_PER_IMAGE / (ms1 * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                "note": "pool of distinct device-resident 24 MP frames cycled (10k-image runs repeat this launch)"}
        # configs[2]: ViT-L/14 + head, batch 512 (fp16 operands, see config.precision)
        g = torch.Generator(device=device).manual_seed(3 + rank)
        clip_in = torch.randn((512, 3, 224, 224), device=device, generator=g)
        scorer.model.encode(clip_in)
        ms2 = best_ms(lambda: scorer.model.encode(clip_in))
        tf2 = 512 * GFLOP_PER_IMAGE * 1e9 / (ms2 * 1e-3) / 1e12
        configs["vit_b512"] = {"baseline_config": 2, "batch": 512, "ms": ms2, "images_per_s_per_gpu": 512 / (ms2 * 1e-3),
                               "TFLOP_s": tf2, "frac_of_sustained_bf16": tf2 / peaks["bf16_tflops"], "dtype": "fp16"}
        del clip_in
        # configs[3]: all-pairs cosine over n3 x 768 embeddings per GPU (gathered: world x n3 rows)
        n3 = args.sim_rows
        e_loc = device_embeddings(n3, 768, 11 + rank, device)

        def sim():
            return cosine_pairs_sharded(e_loc, 0.90)

        sim()
        barrier()
        ms3 = best_ms(sim)
        if world > 1:
            t = torch.tensor([ms3], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms3 = float(t.item())
        ntot = world * n3
        configs["similarity"] = {"baseline_config": 3, "rows_per_gpu": n3, "rows_total": ntot, "dim": 768, "tau": 0.90, "ms": ms3,
                                 "pair_comparisons_per_s": ntot * (ntot - 1) / 2 / (ms3 * 1e-3),
                                 "TFLOP_s_total": ntot * (ntot - 1) * 768 / (ms3 * 1e-3) / 1e12,
                                 "all_gather_bytes_per_rank": (world - 1) * n3 * 768 * (2 + 4) if world > 1 else 0,
                                 "all_gather_note": "bf16 shards first (the scan starts on them), float32 shards on the NCCL stream during the scan"}
        del e_loc

    # ---- e2e: the reference-shaped call.  B items per step ({'path', 'img_cv'} with frames in pinned host memory)
    # -> BatchProcessor.process_items_streamed -> the complete result dicts of batch_processor.py:298-355; then the
    # grouping stage on the embeddings / hashes of those dicts.  H2D, D2H and all host work inside the timed region. ----
    e2e = None
    if not args.no_e2e:
        bp = BatchProcessor(scorer, batch_size=B)
        eb = min(B, 32)              # pinned pool: 32 frames (2.3 GB per rank) referenced B/32 times per step
        reps = max(1, B // eb)
        host = torch.empty((eb, H, W, 3), dtype=torch.uint8, pin_memory=True)
        host.copy_(pool[:eb])
        torch.cuda.synchronize()
        views = [host[i].numpy() for i in range(eb)]
        n_e2e = max(2, min(K, 8))
        # the job's items arrive as ONE stream, like `process_files(paths)` of the reference receives a directory:
        # n_e2e steps x B frames (the pinned pool is referenced repeatedly; every item is copied and scored)
        items = [{"path": f"/bench/rank{rank}/img_{j:06d}.jpg", "img_cv": views[j % eb]} for j in range(eb * reps * n_e2e)]
        chunk, vit_batch = args.e2e_chunk, args.e2e_vit_batch
        bp.process_items_streamed(items[:max(eb, vit_batch)], chunk=chunk, vit_batch=vit_batch)          # warm-up
        barrier()
        bp.metrics["h2d_bytes"] = bp.metrics["d2h_bytes"] = 0
        extra_h2d = extra_d2h = 0
        t0 = time.perf_counter()
        res_all = bp.process_items_streamed(items, chunk=chunk, vit_batch=vit_batch)
        assert all("error" not in r for r in res_all), "e2e: a frame failed"
        emb = torch.from_numpy(np.frombuffer(b"".join(r["clip_embedding"] for r in res_all), dtype=np.float32).reshape(-1, 768).copy()).to(device)
        hh = torch.from_numpy(np.array([int(r["phash"], 16) for r in res_all], dtype=np.uint64).view(np.int64)).to(device)
        p_, _, q_ = grouping(emb, hh)
        extra_h2d = emb.numel() * 4 + hh.numel() * 8
        extra_d2h = int(p_.cpu().numel() + q_.cpu().numel()) * 4
        barrier()
        ms_e = (time.perf_counter() - t0) * 1e3
        # copy-only ceiling: the same pinned frames through the same staging buffers, no kernels, all ranks at once
        stage = [torch.empty((chunk, H, W, 3), dtype=torch.uint8, device=device) for _ in range(2)]
        cs = torch.cuda.Stream(device=device)
        barrier()
        t1 = time.perf_counter()
        with torch.cuda.stream(cs):
            for j in range(eb * reps * 2):
                stage[(j // chunk) & 1][j % chunk].copy_(host[j % eb], non_blocking=True)
        cs.synchronize()
        barrier()
        ms_c = (time.perf_counter() - t1) * 1e3
        if world > 1:
            t = torch.tensor([ms_e, ms_c], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_e, ms_c = (float(v) for v in t.tolist())
        frames_per_step = eb * reps
        e2e_val = world * frames_per_step * n_e2e / (ms_e * 1e-3)
        ceiling = world * frames_per_step * 2 / (ms_c * 1e-3)
        e2e = {"value": e2e_val, "unit": "images/s", "steps": n_e2e, "frames_per_step_per_gpu": frames_per_step,
               "api": "BatchProcessor.process_items_streamed -> result dicts (batch_processor.py:298-355 columns incl. aggregate inputs, tags, "
                      "pHash, embedding bytes), then the grouping stage on their embeddings / hashes",
               "timing": "wall clock between synchronised points (host dict building is inside), max over ranks",
               "chunk_frames": chunk, "vit_batch": vit_batch, "numa_node_rank0": numa_node,
               "h2d_bytes_per_step": bp.metrics["h2d_bytes"] // n_e2e + extra_h2d // n_e2e,
               "d2h_bytes_per_step": bp.metrics["d2h_bytes"] // n_e2e + extra_d2h // n_e2e,
               "h2d_ceiling_images_per_s": ceiling, "h2d_ceiling_GB_s_per_gpu": 2 * frames_per_step * TECH_BYTES_PER_IMAGE / (ms_c * 1e-3) / 1e9,
               "frac_of_h2d_ceiling": e2e_val / ceiling,
               "ceiling_note": "copy-only leg: the same pinned frames into the same staging buffers on one copy stream, no kernels, all "
                               "ranks concurrently"}
        del stage

        # ---- the same call with the two side products of the reference's loop switched on: leading-lines score per image
        # (batch_processor.py:245) and the 640-px thumbnail JPEG (scorer.py:1681-1686).  Edge maps / thumbnail pixels come from
        # the device in the same visit of the frame (the thumbnail as a finished JPEG stream); OpenCV's Hough transform runs on host threads ----
        if not args.no_e2e_side:
            workers = max(2, min(16, (os.cpu_count() or 2) // max(1, world)))
            bps = BatchProcessor(scorer, batch_size=B, num_workers=workers, leading_lines=True)
            # without the pool's pure-noise frames (1 in 8): 8 M edge pixels make cv2.HoughLinesP take seconds per frame — in
            # the reference as well (9.7 s per such frame for its detect_leading_lines on one core) — which no photograph does
            sitems = [it for j, it in enumerate(items[:min(len(items), 2 * B + B // 2)]) if (j % eb) % 8 != 6][:2 * B]
            bps.process_items_streamed(sitems[:max(chunk, 16)], chunk=chunk, vit_batch=vit_batch, thumbnails=True)      # warm-up
            barrier()
            bps.metrics["h2d_bytes"] = bps.metrics["d2h_bytes"] = 0
            t0 = time.perf_counter()
            sres = bps.process_items_streamed(sitems, chunk=chunk, vit_batch=vit_batch, thumbnails=True)
            barrier()
            ms_s = (time.perf_counter() - t0) * 1e3
            assert all("error" not in r and r.get("thumbnail") for r in sres), "e2e side products: a frame failed"
            if world > 1:
                t = torch.tensor([ms_s], device=device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_s = float(t.item())
            e2e["with_leading_lines_and_thumbnails"] = {
                "value": world * len(sitems) / (ms_s * 1e-3), "unit": "images/s", "images_per_gpu": len(sitems), "host_threads_per_gpu": workers,
                "h2d_bytes_per_step": bps.metrics["h2d_bytes"] * B // len(sitems), "d2h_bytes_per_step": bps.metrics["d2h_bytes"] * B // len(sitems),
                "note": "gray / 5x5 blur / Canny (csrc/canny.cu, bit-exact with OpenCV) and the thumbnail pixels (4x4 box sums emitted by the "
                        "technical pass, csrc/thumbnail.cu) on the device; the 24 MB edge map and the thumbnail pixels leave on the D2H "
                        "stream, the thumbnails as JPEG streams encoded on the device (csrc/jpeg_encode.cu); cv2.HoughLinesP on host threads bounds this leg; the pool's pure-noise frames are "
                        "left out of this leg (seconds of HoughLinesP each, in the reference too)"}

        # ---- e2e from FILE BYTES: the same call with items that carry JPEG streams (what the reference's loader reads from
        # disk, utils/image_loading.py:90) in pinned host memory; decoding happens on the device (csrc/jpeg_decode.cu) ----
        if not args.no_e2e_jpeg:
            import io
            from concurrent.futures import ThreadPoolExecutor
            from PIL import Image
            n_src = min(16, eb)
            rgb = [host[i].numpy()[:, :, ::-1].copy() for i in range(n_src)]
            jchunk = args.e2e_jpeg_chunk

            def jpeg_leg(restart_blocks):
                def enc(a):
                    buf = io.BytesIO()
                    kw = {"restart_marker_blocks": restart_blocks} if restart_blocks else {}
                    Image.fromarray(a).save(buf, "JPEG", quality=90, **kw)
                    return buf.getvalue()

                t_enc = time.perf_counter()
                with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
                    streams = list(ex.map(enc, rgb))
                t_enc = time.perf_counter() - t_enc
                t_dec = time.perf_counter()
                Image.open(io.BytesIO(streams[0])).convert("RGB").load()
                pil_decode_ms = (time.perf_counter() - t_dec) * 1e3
                pinned = []
                for st_ in streams:
                    pt = torch.empty(len(st_), dtype=torch.uint8, pin_memory=True)
                    pt.numpy()[:] = np.frombuffer(st_, np.uint8)
                    pinned.append(pt)
                jitems = [{"path": f"/bench/rank{rank}/jpg_{j:06d}.jpg", "jpeg": pinned[j % n_src].numpy()} for j in range(B * n_e2e)]
                bp.process_items_streamed(jitems[:max(2 * jchunk, vit_batch)], chunk=jchunk, vit_batch=vit_batch)        # warm-up
                barrier()
                bp.metrics["h2d_bytes"] = bp.metrics["d2h_bytes"] = 0
                t0 = time.perf_counter()
                jres = bp.process_items_streamed(jitems, chunk=jchunk, vit_batch=vit_batch)
                assert all("error" not in r for r in jres), "e2e_jpeg: a stream failed"
                emb = torch.from_numpy(np.frombuffer(b"".join(r["clip_embedding"] for r in jres), dtype=np.float32).reshape(-1, 768).copy()).to(device)
                hh = torch.from_numpy(np.array([int(r["phash"], 16) for r in jres], dtype=np.uint64).view(np.int64)).to(device)
                grouping(emb, hh)
                barrier()
                ms_j = (time.perf_counter() - t0) * 1e3
                if world > 1:
                    t = torch.tensor([ms_j], device=device)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    ms_j = float(t.item())
                return {"value": world * len(jitems) / (ms_j * 1e-3), "unit": "images/s", "images_per_gpu": len(jitems),
                        "input": f"{n_src} distinct 24 MP frames of the pool as baseline JPEG (Pillow, quality 90, 4:2:0, "
                                 + (f"restart interval {restart_blocks} MCUs" if restart_blocks else "NO restart markers, as cameras write them")
                                 + f"), {sum(len(x) for x in streams) / n_src / 1e6:.2f} MB each, in pinned host memory",
                        "h2d_bytes_per_step": bp.metrics["h2d_bytes"] // n_e2e, "d2h_bytes_per_step": bp.metrics["d2h_bytes"] // n_e2e,
                        "chunk_streams": jchunk, "pillow_decode_ms_per_image_one_core": pil_decode_ms, "pillow_encode_s_total": t_enc}

            e2e["from_jpeg_bytes"] = jpeg_leg(args.jpeg_restart_blocks)
            e2e["from_jpeg_bytes"]["note"] = (
                "same call, items carry the file bytes instead of decoded frames: PCIe moves ~14x fewer bytes and the decode (byte-exact "
                "with Pillow, tests/test_gpu_jpeg.py) runs on the GPU, one thread per restart interval; the reference arm starts from "
                "decoded frames, so the headline e2e above stays the raw-frame figure")
            e2e["from_jpeg_bytes_no_restart_markers"] = jpeg_leg(0)
            e2e["from_jpeg_bytes_no_restart_markers"]["note"] = "entropy decoding by the self-synchronising scheme (csrc/jpeg_decode.cu)"
            del rgb
        del host

    # ---- CPU baseline beside it (rank 0, N=1 only): the same bounded sample `--impl reference` runs -------------
    cpu_baseline = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, orig_affinity)      # the CPU arm may use every host core again
        from oracle import cpu_port
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sd = random_state_dict(0)
        ref, kind, desc = cpu_arm()
        frames = cpu_sample_frames()
        cpu_port.score_images_cpu(frames[:1], sd, torch.from_numpy(tags), ref_analyzers=ref)
        t0 = time.perf_counter()
        tech_cpu, vit_cpu = cpu_port.score_images_cpu(frames, sd, torch.from_numpy(tags), ref_analyzers=ref)
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": len(frames) / dt, "unit": "images/s", "cores": cores, "kind": kind,
                        "sample": f"{len(frames)} synthetic 24 MP frames (seeds 2000..), ViT batch {len(frames)}; {desc}"}
        # parity spot check on those frames (checker only)
        got = scorer.score_images(np.stack(frames))
        cosv = [float(np.dot(np.frombuffer(g["clip_embedding"], np.float32), vit_cpu["embedding"][i].numpy())) for i, g in enumerate(got)]
        cpu_baseline["parity_spot_check"] = {
            "hist_exact": all(g["histogram_data"] == t["histogram"]["histogram_bytes"] for g, t in zip(got, tech_cpu)),
            "phash_equal": all(g["phash"] == t["phash"] for g, t in zip(got, tech_cpu)),
            "min_embedding_cosine": min(cosv)}

    if rank == 0:
        line = {
            "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": K,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16", "data": "synthetic", "config": workload_config(B),
            "clocks": clocks, "gpu_launches": launches, "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "stages": stages, "configs": configs,
            "pairs": {"cosine": int(pairs.shape[0]), "hamming": int(hpairs.shape[0])},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
