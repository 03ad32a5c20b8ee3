#!/usr/bin/env python
"""Throughput of the GigaAM hot path (log-mel -> Conformer encoder -> CTC greedy) on B200.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 2 --warmup 1       # the unmodified reference (oracle/_ref archive) on host cores
    python bench.py --steps 20 --warmup 3 --dump-outputs /tmp/out   # + the last timed step's outputs as /tmp/out/*.npy

Workload (BASELINE.json configs[1]): v2_ctc, batch 64 x 10 s synthetic 16 kHz audio per GPU (weak scaling:
every rank runs its own 64 utterances, hypotheses all-gathered to every rank over NCCL when N > 1), seeded
random weights of the reference's shape (no checkpoints offline).

One JSON line on stdout (rank 0): see the task contract.  `value` = device-resident throughput (CUDA graph of
the whole step, rotating input buffers larger than L2), `e2e` = the same metric through the public API
(`model.forward` + `model.decoding.decode`) from pinned HOST buffers with the H2D / D2H copies inside the timed
region, `roofline` = the dominant kernel class timed live with CUDA events, `cpu_baseline` = the unmodified reference (oracle/_ref, else the oracle port) on the
box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

MODEL = "v2_ctc"
BATCH = 64
SECONDS = 10.0
N_ROT = 4  # rotating input buffers: 4 x 41 MB = 164 MB > 126 MB L2
DUMP_LIMIT = 64_000_000  # bytes of .npy data --dump-outputs may write


def flops_per_utterance(n_samples: int) -> dict:
    """Algorithmic FLOPs (2 x MAC, dense, padding-free) of one utterance -- SURVEY 8(d) formulae."""
    M = n_samples // 160 + 1
    T1 = (M - 1) // 2 + 1
    T = (T1 - 1) // 2 + 1
    d, ff, L, V1 = 768, 3072, 16, 34
    sub = 2 * 9 * d * T1 * 32 + 2 * 6912 * d * T * 16 + 2 * 12288 * d * T
    per_frame = 2 * (2 * d * ff) * 2 + 4 * 2 * d * d + 2 * d * 2 * d + 2 * d * d + 2 * 31 * d + 4 * d * T
    return {"T": T, "M": M, "subsampling": sub, "layers": L * per_frame * T, "head": 2 * d * V1 * T,
            "total": sub + L * per_frame * T + 2 * d * V1 * T,
            "gemm_ffn_up": 2 * d * ff * T, "gemm_ffn_down": 2 * d * ff * T}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0: float = None, t1: float = None) -> dict:
        """Summary of the samples received inside [t0, t1] (the timed region); the sampler itself is started before the
        warm-up so that nvidia-smi's start-up latency does not eat the window."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        inside = [ln for ts, ln in self.lines if t0 is None or (t0 <= ts <= t1 + 0.03)]
        if not inside:
            inside = [ln for _, ln in self.lines[-3:]]
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference(steps: int, warmup: int, batch: int = 4, reps: int = 3, seconds: float = SECONDS):
    """The reference's own CPU PyTorch path on all host cores: log-mel + encoder + CTC greedy incl. host detokenisation,
    fp32, no autocast (gigaam/model.py:34-35).  Runs the UNMODIFIED reference modules byte-compiled into
    oracle/_ref/gigaam_ref.zip (oracle/build_ref.py; kind "reference"); only if that archive is missing does it time the
    oracle port of the same ATen ops (oracle/gigaam_oracle.py; kind "port")."""
    import torch
    from gigaam_b200 import synthetic

    ck = synthetic.synthetic_checkpoint(MODEL, seed=0)
    cfg, sd = ck["cfg"], ck["state_dict"]
    wav, wav_len = synthetic.synthetic_audio(batch, seconds, seed=1234)
    vocab = cfg["decoding"]["vocabulary"]
    try:
        from oracle.ref_loader import build_reference
        ref_root, ref_decoding = build_reference(cfg, sd)
        kind = "reference"

        def forward(w, l):
            mel, mel_len = ref_root.preprocessor(w, l)
            return ref_root.encoder(mel, mel_len)

        def decode(enc, enc_len):
            return [t for t, _, _ in ref_decoding.decode(ref_root.head, enc, enc_len)]
    except ImportError:
        from oracle import gigaam_oracle as orc
        kind = "port"

        def forward(w, l):
            return orc.model_forward(w, l, sd, cfg)

        def decode(enc, enc_len):
            return ["".join(vocab[i] for i in ids) for ids, _ in orc.ctc_greedy(enc, enc_len, sd)]
    # all host threads the process may use: affinity mask capped by the cgroup CPU quota (a 128-thread pool on a
    # quota of a few CPUs thrashes); then keep the fastest of {all, 1/2, 1/4} on a short probe
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            avail = max(1, min(avail, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    probe_wav, probe_len = wav[:1, : 3 * 16000].contiguous(), torch.tensor([3 * 16000])
    best, cores = None, avail
    for n in sorted({avail, max(1, avail // 2), max(1, avail // 4)}, reverse=True):
        torch.set_num_threads(n)
        with torch.inference_mode():
            forward(probe_wav, probe_len)
            t0 = time.perf_counter()
            forward(probe_wav, probe_len)
            dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, n
    torch.set_num_threads(cores)

    # one step = `reps` batches of `batch` utterances: batches of 4 are where the CPU path is fastest on the GPU boxes'
    # hosts (measured 5.2 utt/s at 4 per batch vs 3.2-3.8 at 16: memory-bound), so the baseline is not handicapped
    def step():
        out = []
        for _ in range(reps):
            with torch.inference_mode():
                enc, enc_len = forward(wav, wav_len)
                out += decode(enc, enc_len)
        return out

    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    sec = statistics.median(times)
    return {"value": batch * reps / sec, "unit": "utt/s", "cores": cores, "kind": kind,
            "sample": f"{reps} batches of {batch} x {seconds:g} s utterances of the same workload per step, median of {steps} steps "
                      f"after {warmup} warm-up, torch {torch.__version__} fp32, {cores} threads",
            "rtfx": batch * reps * seconds / sec, "sec_per_step": sec}


def dump_outputs(out_dir: Path, enc, enc_len, ids, frames, counts) -> None:
    """What one step of the timed path returned (encoder output and lengths, CTC hypotheses), written as float32 / float64
    .npy files so that two builds can be compared output for output on the same seeded inputs.  Hypothesis slots past an
    utterance's count hold -1 (the kernels leave them unwritten).  If the encoder output [B, T', d] would not fit in
    DUMP_LIMIT, a fixed seeded sample of utterances is written; enc_utterances.npy lists which."""
    import numpy as np
    import torch

    out_dir.mkdir(parents=True, exist_ok=True)
    counts = counts.cpu().long()
    unwritten = torch.arange(ids.shape[1])[None, :] >= counts[:, None]
    arrays = {"enc_len": enc_len.cpu().double(), "counts": counts.double(),
              "ids": ids.cpu().long().masked_fill(unwritten, -1).double(),
              "frames": frames.cpu().long().masked_fill(unwritten, -1).double()}
    B = enc.shape[0]
    room = (DUMP_LIMIT - 8 * sum(a.numel() for a in arrays.values()) - 8 * B - 4096) // (4 * enc[0].numel())  # 4 KB: headers
    keep = torch.arange(B)
    if room < B:
        keep = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:room].sort().values
    arrays["enc_utterances"] = keep.double()
    arrays["enc"] = enc[keep.to(enc.device)].float().cpu()
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a.numpy())


def c4_strong_scaling(dev, rank: int, world: int, steps: int = 3, total: int = 256, chunk: int = 32, seconds: float = 10.0):
    """BASELINE.json configs[3]: v3_e2e_rnnt, 256 x 10 s in total, sharded across the N GPUs of the job (STRONG scaling:
    the work is fixed, 256 / N utterances per rank, run in device batches of 32 = the per-GPU batch at N = 8), encoder +
    RNN-T greedy loop on every rank, then ONE packed all-gather of all hypotheses (gam_gather_hyps) inside the timed
    region.  Device-timed with CUDA events, max over ranks.  Returns the dict reported under `strong_scaling_c4`."""
    import torch
    import torch.distributed as dist
    import gigaam_b200 as gigaam
    from gigaam_b200.dist import HypothesisGather, shard_bounds, unpack_gathered

    model = gigaam.load_model("v3_e2e_rnnt", device=dev, synthetic=True)
    eng = model._get_engine()
    s0, s1 = shard_bounds(total, rank, world)
    rows = (total + world - 1) // world
    wav, wav_len = gigaam.synthetic_audio(total, seconds, seed=1234)     # the SAME 256 utterances whatever N is ...
    wav, wav_len = wav[s0:s1].to(dev), wav_len[s0:s1].to(dev)            # ... this rank's contiguous shard of them
    T = eng.encoded_frames(eng.logmel_frames(wav.shape[1]))
    W = eng.hyp_width(T)
    gather = HypothesisGather(eng) if world > 1 else None
    packed = eng.packed_hypotheses(rows, T)
    ids_v = packed[: rows * W].view(rows, W)
    frames_v = packed[rows * W: 2 * rows * W].view(rows, W)
    counts_v = packed[2 * rows * W:]

    def step():
        for c0 in range(0, s1 - s0, chunk):
            c1 = min(c0 + chunk, s1 - s0)
            enc, enc_len = model(wav[c0:c1], wav_len[c0:c1])
            ids, frames, counts = model.decoding.decode_device(model.head, enc, enc_len)
            ids_v[c0:c1], frames_v[c0:c1], counts_v[c0:c1] = ids, frames, counts
        if gather is not None:
            return unpack_gathered(gather.all_gather(packed), total, world, rows, W), enc_len
        return (ids_v, frames_v, counts_v), enc_len

    with torch.inference_mode():
        for _ in range(2):
            out, enc_len = step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out, enc_len = step()
        e1.record()
        torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    counts = out[2].cpu()
    assert counts.numel() == total
    return {"metric": "utterances/sec (v3_e2e_rnnt, 256 x 10 s in total, sharded over the job's GPUs)", "value": total / (ms * 1e-3),
            "unit": "utt/s", "ms_per_step": ms, "steps": steps, "global_batch": total, "per_gpu_batch": s1 - s0, "device_batch": chunk,
            "scaling": "strong", "gather_in_timed_region": world > 1,
            "tokens_per_frame": float(counts.sum()) / float(total * T), "rtfx": total * seconds / (ms * 1e-3),
            "api": "model(wav, len) + model.decoding.decode_device(...) per device batch, gam_gather_hyps once per step"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the strong-scaling leg (BASELINE configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 path")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout must carry exactly ONE JSON line: libraries (NCCL prints its version banner on stdout) are diverted to stderr
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    n_samples = int(SECONDS * 16000)
    config = {"workload": f"{MODEL} batch={args.batch}x{SECONDS:g}s per GPU: log-mel + 16-layer Conformer encoder + CTC greedy "
                          "(BASELINE.json configs[1])",
              "global_batch": args.batch * max(world, 1), "audio_seconds": SECONDS, "parallelism": f"dp{max(world, 1)} (utterance sharding)",
              "l2": f"{N_ROT} rotating input buffers ({N_ROT * args.batch * n_samples * 4 / 1e6:.0f} MB > 126 MB L2); >2 GB of "
                    "intermediates + 465 MB weights per step"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        steps = args.steps
        res = cpu_reference(steps, max(1, min(args.warmup, 1)))
        line = {"impl": "reference", "metric": "utterances/sec (10 s audio, v2_ctc)", "value": res["value"], "unit": "utt/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": res["sec_per_step"] * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "rtfx": res["rtfx"],
                "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": res["value"], "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
        return 0

    import torch
    import torch.distributed as dist
    import gigaam_b200 as gigaam

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = gigaam.load_model(MODEL, device=dev, synthetic=True)  # reference defaults: fp16_encoder=True
    eng = model._get_engine()
    B = args.batch
    wavs, lens = [], None
    for i in range(N_ROT):
        w, l = gigaam.synthetic_audio(B, SECONDS, seed=1234 + 17 * i + 1000 * rank)
        wavs.append(w.to(dev))
        lens = l
    wav_len = lens.to(dev)
    M = eng.logmel_frames(n_samples)
    T = eng.encoded_frames(M)
    mel_len = model.preprocessor.out_len(wav_len)
    static_in = torch.empty_like(wavs[0])
    # the path's only exchange (SURVEY 8e): every rank's packed hypotheses to every rank, ONE ncclAllGather issued by the
    # library (gam_gather_hyps) on the compute stream -- inside the CUDA graph below, so replicas are not re-synchronised
    # by host-side collectives between steps
    hyp_gather = None
    if world > 1:
        from gigaam_b200.dist import HypothesisGather
        hyp_gather = HypothesisGather(eng)
    packed = eng.packed_hypotheses(B, T)

    def device_step(wav, collective=True):
        mel = eng.logmel(wav)
        enc, enc_len = eng.encode(mel, mel_len)
        ids, frames, counts = eng.greedy(enc, enc_len, packed)
        if hyp_gather is not None and collective:
            return ids, frames, counts, hyp_gather.all_gather(packed), enc, enc_len
        return ids, frames, counts, None, enc, enc_len

    # ---- warm-up eagerly, then capture the whole step in one CUDA graph (kills ~250 launch gaps)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        for _ in range(2):
            out = device_step(static_in)
        side.synchronize()
        launches0 = eng.launch_count()
        out = device_step(static_in)
        launches_per_step = eng.launch_count() - launches0
    side.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        g_ids, g_frames, g_counts, g_all, g_enc, g_enc_len = device_step(static_in)

    def graph_step(i):
        static_in.copy_(wavs[i % N_ROT], non_blocking=True)  # device->device refill of the static input (41 MB)
        graph.replay()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for i in range(max(args.warmup, 3)):
        graph_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        graph_step(i)
    e1.record()
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    if world > 1:
        dist.barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total / 1e3)
    if args.dump_outputs is not None and rank == 0:
        # before any later leg: the eager runs below write into the same hypothesis buffer
        dump_outputs(args.dump_outputs, g_enc, g_enc_len, g_ids, g_frames, g_counts)

    # ---- end to end through the public API from pinned host memory
    host_wavs = [w.cpu().pin_memory() for w in wavs]
    host_len = lens.clone().pin_memory()

    def api_step(i):
        wav = host_wavs[i % N_ROT].to(dev, non_blocking=True)
        ln = host_len.to(dev, non_blocking=True)
        enc, enc_len = model(wav, ln)                                   # GigaAM.forward
        hyps = model.decoding.decode(model.head, enc, enc_len)          # D2H of ids / frames / counts + detokenise
        return hyps

    for i in range(3):
        api_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        hyps = api_step(i)
    torch.cuda.synchronize()
    e2e_serial_sec = time.perf_counter() - t0
    # same calls, same per-step H2D / D2H, but driven by gigaam_b200.pipeline.BatchPipeline: the copy of step i+1 and the
    # read-back + detokenisation of step i-1 overlap the kernels of step i
    from gigaam_b200.pipeline import BatchPipeline
    pipe = BatchPipeline(model, gather=hyp_gather)      # N > 1: every rank ends up with the hypotheses of all ranks
    n_hyp = sum(len(h) for h in pipe.run((host_wavs[i % N_ROT], host_len) for i in range(3)))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    n_hyp = sum(len(h) for h in pipe.run((host_wavs[i % N_ROT], host_len) for i in range(args.steps)))
    torch.cuda.synchronize()
    e2e_sec = time.perf_counter() - t0
    assert n_hyp == world * B * args.steps
    t = torch.tensor([e2e_sec, e2e_serial_sec], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(t[0].item())
    e2e_serial_value = world * B * args.steps / float(t[1].item())
    h2d = B * n_samples * 4 + B * 8
    d2h = world * (2 * B * T * 4 + B * 4) + B * 4     # ids, frames [B, T'] + counts of every rank's batch, encoded_len [B]; int32

    # ---- dominant kernel, timed live with CUDA events on the launching stream
    roofline = None
    if rank == 0:
        peaks = {}
        pk = ROOT / "MEASURED_PEAKS.json"
        if pk.exists():
            peaks = json.loads(pk.read_text())
        peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
        eng.profile_begin()
        nprof = 3
        for i in range(nprof):
            device_step(wavs[i % N_ROT], collective=False)     # rank 0 only: the kernels without the all-gather
        prof = eng.profile_end()
        fl = flops_per_utterance(n_samples)
        R = B * fl["T"]
        cls_flops = {"gemm_ffn_up_silu": 2 * R * 768 * 3072, "gemm_ffn_down_res": 2 * R * 768 * 3072,
                     "gemm_conv2_implicit": 2 * B * fl["T"] * 16 * 6912 * 768, "gemm_subsample_out": 2 * R * 12288 * 768,
                     "gemm_qkv": None, "gemm_proj_res": 2 * R * 768 * 768, "gemm_pw1_glu": 2 * R * 768 * 1536}
        total_ms = sum(v[0] for v in prof.values())
        dom = max(prof.items(), key=lambda kv: kv[1][0])
        name, (ms_sum, n) = dom
        avg_ms = ms_sum / n
        fpl = cls_flops.get(name)
        achieved = fpl / (avg_ms * 1e-3) / 1e12 if fpl else None
        traffic = None
        tr = ROOT / "profiles" / "ncu_traffic.json"   # dram bytes per launch from the committed ncu --set full capture
        if tr.exists():
            traffic = json.loads(tr.read_text()).get(name)
        roofline = {"kernel": name, "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic,
                    "traffic_source": "profiles/ncu_traffic.json: dram bytes per launch from the committed ncu --set full capture "
                                      "(cold L2), not measured in this run",
                    "classes_note": "per-launch CUDA events around eager launches: the classes sum to more than ms_per_step (one "
                                    "CUDA graph, no launch gaps); use them for shares",
                    "peak_source": peak_src,
                    "avg_launch_ms": avg_ms, "launches_per_step": n // nprof, "share_of_step": ms_sum / total_ms,
                    "flops_per_launch": fpl,
                    "step_tflops": B * fl["total"] / (ms_per_step * 1e-3) / 1e12,
                    "step_frac": B * fl["total"] / (ms_per_step * 1e-3) / 1e12 / peak_tf,
                    "classes_ms_per_step": {k: round(v[0] / nprof, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}

    # ---- varlen leg (N = 1 only, outside the timed region): the same 64-utterance buffer with ragged lengths (uniform in
    # 0.1 .. 1.0 of the 10 s).  Reported as summed kernel time (CUDA events around every launch) next to the full-length
    # step's, because an eager step is paced by the host.  Never fatal: the contract line does not depend on it.
    varlen = None
    if rank == 0 and world == 1 and roofline is not None:
        try:
            gen = torch.Generator().manual_seed(7)
            rag_len = (torch.rand(B, generator=gen) * 0.9 + 0.1).mul(n_samples).long()
            rag_len[0] = n_samples
            rag_len_dev = rag_len.to(dev)
            rag_wav = wavs[0] * (torch.arange(n_samples, device=dev)[None, :] < rag_len_dev[:, None])
            rag_mel_len = model.preprocessor.out_len(rag_len_dev)

            def ragged_step():
                enc, enc_len = eng.encode(eng.logmel(rag_wav), rag_mel_len)
                return eng.greedy(enc, enc_len, packed)
            ragged_step()
            best = float("inf")
            for _ in range(3):
                eng.profile_begin()
                ragged_step()
                best = min(best, sum(ms for ms, _ in eng.profile_end().values()))
            full_ms = sum(v[0] for v in prof.values()) / nprof
            frac = float(rag_len.sum()) / float(B * n_samples)
            varlen = {"workload": f"the same {B} x {SECONDS:g} s buffer, utterance lengths uniform in 0.1 .. 1.0 of it",
                      "audio_fraction": round(frac, 3), "kernel_ms_full_lengths": round(full_ms, 3), "kernel_ms_ragged": round(best, 3),
                      "utt_per_s_of_kernel_time": round(B / best * 1e3, 1),
                      "note": "packed rows (cu_seqlens built on the device): only the frames that exist run through the encoder"}
            del rag_wav
        except Exception as e:  # noqa: BLE001
            varlen = {"error": repr(e)[:300]}
            try:
                eng.profile_end()      # never leave the per-launch event profiler armed
            except Exception:  # noqa: BLE001
                pass

    del pipe, graph
    strong = None if args.no_c4 else c4_strong_scaling(dev, rank, world)
    if rank == 0:
        # the CPU baseline is a property of the box, not of N: timed at N = 1 only (other ranks would idle behind it)
        cpu = None if (args.no_cpu_baseline or world > 1) else cpu_reference(steps=4, warmup=1)   # ~12 s of CPU work
        line = {"metric": "utterances/sec (10 s audio, v2_ctc)", "value": value, "unit": "utt/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16 tensor-core operands, f32 accumulate/residual/norm/head",
                "data": "synthetic", "config": config, "rtfx": value * SECONDS, "rtf": 1.0 / (value * SECONDS),
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "utt/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "api": "gigaam_b200.pipeline.BatchPipeline over model(wav, len) + model.decoding: pinned host wav in, python "
                               "hypotheses out, copies of neighbouring steps overlapped with compute, kernels replayed as one CUDA graph per shape",
                        "serial_value": e2e_serial_value},
                "gpu_launches": launches_per_step * args.steps, "launches_per_step": launches_per_step,
                "roofline": roofline, "varlen": varlen, "strong_scaling_c4": strong,
                "cpu_baseline": ({k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")} if cpu else None)}
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
