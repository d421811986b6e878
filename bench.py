#!/usr/bin/env python
"""bench.py — audio-seconds synthesised per wall-second on the BASELINE.json workload.

  python bench.py --gpus 1 --steps 5 --warmup 3            # our arm (C2: medium, 32 x 256 phonemes)
  python bench.py --impl reference --steps 2 --warmup 1    # reference arm: CPU path on host cores
  torchrun ... bench.py --gpus N ...                        # one rank per GPU, weak scaling (32 utts / GPU)
  python bench.py --steps 5 --warmup 3 --dump-outputs DIR  # also write the last timed step's waveforms to DIR

A "step" is one pass of the phoneme-id -> waveform hot path over one batch of synthetic ids.  The ids, the voice and
the noise (a per-voice call counter seeds it) depend only on the arguments, so two builds can be compared on the
arrays --dump-outputs writes.  The synthetic voices are written to a temporary directory, never into the tree.
`value`   : whole-job audio-s/s, device-resident result (N > 1: incl. the NCCL id broadcast / length all-reduce).
`e2e`     : same metric, host ids in -> host waveforms out: `speak_batch_ids` (N = 1) / `shard.Frontend` (N > 1: one
            frontend on rank 0, results through a page-locked host segment shared by the ranks).
`c5`      : BASELINE config 5 (1024 mixed-length utterances): aggregate audio-s/s and p50 / p99 completion latency.
`secondary`: C1 (single 128-phoneme utterance) and C3 (high voice, 16 x 512) on the same box in the same run (N = 1).
`roofline`: dominant kernel class (HiFi-GAN ResBlock convolutions), CUDA-event timed in the same run.
`cpu_baseline`: the oracle (a port of the reference's onnxruntime graph) on this box's host cores.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

# stdout carries exactly one JSON line: NCCL's own banner / debug output ("NCCL version ...") goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 22050
HOP = 256
DUMP_BUDGET = 64_000_000        # bytes --dump-outputs may write in all


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json), or null."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return None


def dump_outputs(out_dir: str, waves) -> None:
    """The waveforms of one step as its caller receives them: `audio_000.npy`, ... (float32, one per utterance, in
    batch order) and their lengths in samples (`samples.npy`, float64).  When the waveforms exceed DUMP_BUDGET together,
    each is cut to the same fraction of its samples, at sorted positions drawn from a generator seeded with the
    utterance's index: equal lengths give equal positions."""
    os.makedirs(out_dir, exist_ok=True)
    lens = np.array([len(w) for w in waves], dtype=np.float64)
    np.save(os.path.join(out_dir, "samples.npy"), lens)
    room = DUMP_BUDGET - lens.nbytes - 256 * (len(waves) + 1)         # 256: bound on one .npy header
    frac = min(1.0, room / (4.0 * max(lens.sum(), 1.0)))
    for b, w in enumerate(waves):
        w = np.asarray(w, dtype=np.float32)
        if frac < 1.0:
            pick = np.random.default_rng([20261017, b]).choice(len(w), int(len(w) * frac), replace=False)
            w = w[np.sort(pick)]
        np.save(os.path.join(out_dir, f"audio_{b:03d}.npy"), w)


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """samples from here on belong to the timed region"""
        self.first = len(self.lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        first = getattr(self, "first", 0)
        window = "timed region"
        lines = self.lines[first:]
        if not lines:                       # region shorter than one sampling period: use the warm-up samples too
            lines, window = self.lines, "warm-up + timed region"
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def tune_cpu_threads(quality: str, cores: int) -> int:
    """onnxruntime's default (all cores, piper/src/lib.rs:79-86) oversubscribes small B=1 ops on many-core
    hosts; give the CPU arm its best shot: probe a short utterance at a few thread counts and keep the best."""
    best, best_v = min(cores, 8), 0.0
    for t in sorted({min(cores, x) for x in (4, 8, 16, 32, 64)}):
        cpu_reference(quality, 24, 1, t)
        a_, w_ = cpu_reference(quality, 48, 1, t)
        if a_ / w_ > best_v:
            best, best_v = t, a_ / w_
    return best


def cpu_reference(quality: str, n_phonemes: int, n_utts: int, threads: int):
    """Times the oracle (CPU port of the reference's ort graph) B=1 sequentially, like speak_batch
    (piper/src/lib.rs:433-435).  Returns (audio_seconds, wall_seconds)."""
    import torch
    from oracle import vits_oracle as vo
    from sonata_b200 import voicegen, workload
    torch.set_num_threads(threads)
    W = vo.to_torch(voicegen.make_tensors(quality))
    a = vo.arch_of(W)
    g = torch.Generator().manual_seed(5)
    scales = [0.667, 1.0, 0.8]
    audio = 0.0
    t0 = time.perf_counter()
    for u in range(n_utts):
        ids = workload.synthetic_ids(n_phonemes, utt=u)
        ew = torch.randn(1, 2, len(ids), generator=g)
        st = {}
        with torch.inference_mode():
            z_ = None
            # noise for z_p needs y_len: draw after the duration predictor like the graph does
            x, m_p, logs_p = vo.text_encoder(W, torch.as_tensor(ids).view(1, -1), a)
            logw = vo.sdp_reverse(W, x, ew, scales[2], a)
            _, w_ceil, y_len = vo.durations(logw, scales[1])
            ez = torch.randn(1, a["inter"], y_len, generator=g)
            z_p, _ = vo.expand(m_p, logs_p, w_ceil, y_len, ez, scales[0])
            z = vo.flow_reverse(W, z_p, a)
            wav = vo.decoder(W, z, a)
        audio += wav.numel() / SR
    return audio, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2", choices=["C1", "C2", "C3"])
    ap.add_argument("--backend", type=int, default=int(os.environ.get("SB200_BACKEND", "1")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 mixed-length corpus")
    ap.add_argument("--c5-utts", type=int, default=1024)
    ap.add_argument("--no-secondary", action="store_true", help="skip the C1 / C3 secondary lines (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the waveforms of the last one to DIR as .npy (one process only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1 or args.steps < 1):
        ap.error("--dump-outputs needs --impl b200, one process and --steps >= 1")

    from sonata_b200 import workload
    quality, B, NPH = workload.CONFIGS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg_desc = {"workload": f"{args.workload}: synthetic-{quality} (en_US-lessac-{quality} architecture), "
                            f"{B} x {NPH}-phoneme utterances per GPU, scales [0.667,1,0.8]",
                "quality": quality, "batch_per_gpu": B, "phonemes": NPH, "ids_per_utt": 2 * NPH + 2,
                "l2": "working set (>5 GB of activations per step) far exceeds the 126 MB L2",
                "parallelism": (f"dp{world}: one process per GPU; rank 0 is the frontend (NCCL broadcast of ids, all-reduce of frame "
                                "counts; utterances are independent, no collective on the waveform path)" if world > 1 else "dp1")}
    cores = os.cpu_count() or 1

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        n_per_step = 1
        threads = tune_cpu_threads(quality, cores)
        for _ in range(max(args.warmup, 0)):
            cpu_reference(quality, NPH, 1, threads)
        audio, wall = 0.0, 0.0
        for s in range(args.steps):
            a_, w_ = cpu_reference(quality, NPH, n_per_step, threads)
            audio += a_; wall += w_
        v = audio / wall
        print(json.dumps({
            "impl": "reference", "metric": "audio-sec/sec", "value": v, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg_desc,
            "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": threads, "kind": "port", "host_cpus": cores,
                             "sample": f"{n_per_step} utterance(s) of the workload per step, B=1 sequential like speak_batch, "
                                       f"torch threads auto-tuned to {threads} of {cores} host CPUs; "
                                       "PyTorch-CPU restatement of the reference's onnxruntime graph (ort itself is absent offline)"},
            "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return

    # ------------------------------------------------------------------ our arm
    # stdout must carry exactly ONE line (the JSON): native libraries (NCCL's version banner, for one) write to file
    # descriptor 1 directly, so fd 1 points at stderr until the line is printed
    sys.stdout.flush()
    _stdout_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    import sonata_b200
    from sonata_b200 import voicegen, shard
    from sonata_b200.job import SynthesisJob
    from sonata_b200 import _native

    if not os.path.exists(_native.LIB_PATH):
        from sonata_b200 import build as _b
        _b.build()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # every process writes the (seeded, identical) voices into a directory of its own: the tree may be read-only
    voice_dir = tempfile.mkdtemp(prefix="sonata_b200_voices_")
    atexit.register(shutil.rmtree, voice_dir, True)
    cfg_path = voicegen.write_voice(voice_dir, quality)
    model = sonata_b200.from_config_path(cfg_path, device=local_rank)
    model.set_backend(args.backend)
    lib = _native.lib()

    total_utts = B * world
    all_batches = [workload.synthetic_ids(NPH, utt=u) for u in range(total_utts)]
    ids_per_step = sum(len(b) for b in all_batches)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_pair(wall, audio):
        """max-over-ranks wall, sum-over-ranks audio"""
        if world == 1:
            return wall, audio
        t = torch.tensor([wall, audio], dtype=torch.float64, device="cuda")
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        return float(tm[0]), float(ts[1])

    # N > 1: ONE frontend (rank 0) holds every utterance; ids travel by NCCL broadcast, each rank runs its LPT shard, the
    # frame counts are all-reduced, waveforms go device -> host into one page-locked segment shared by the ranks
    # (sonata_b200/shard.py Frontend; SURVEY section 8e).  N = 1: the same public call without a process group.
    fe = shard.Frontend(model) if world > 1 else None
    if fe is not None:
        fe.collect_profile = True

    prof_acc = {}

    def add_profile(regions):
        for r in regions:
            acc = prof_acc.setdefault(r["name"], {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
            for k in ("ms", "flops", "bytes", "launches"):
                acc[k] += r[k]

    def step_device(record, keep=False):
        """device-resident pass (results stay in HBM); returns this rank's (audio seconds, device ms) and, with `keep`
        (N = 1), the job still holding its results, for the caller to close"""
        if fe is None:
            job = SynthesisJob(model, all_batches)
            ms = job.run()
            samples = job.lengths()[1]
            if record:
                add_profile(job.profile())
            if not keep:
                job.close()
            return sum(samples) / SR, ms, (job if keep else None)
        fe.synthesize(all_batches if rank == 0 else None, device_only=True)
        owner, samples = fe.last_table
        if record:
            add_profile(fe.last_profile)
        return float(samples[owner == rank].sum()) / SR, fe.last_device_ms, None

    def step_e2e():
        """host ids in -> host waveforms out, through the public call (N = 1) / the one-frontend path (N > 1); returns
        the audio seconds DELIVERED TO THE CALLER on this rank (all of it on rank 0 when N > 1)"""
        if fe is None:
            auds = model.infer_batch_with_values(all_batches)
            return sum(len(a) for a in auds) / SR
        out = fe.synthesize(all_batches if rank == 0 else None)
        return sum(len(o) for o in out) / SR if rank == 0 else 0.0

    # warm-up (the clock sampler starts here so that nvidia-smi is already streaming when the timed region begins)
    sampler = ClockSampler(local_rank)
    sampler.start()
    W = max(args.warmup, 3)
    for _ in range(W):
        step_device(False)

    barrier()
    launches0 = int(lib.sb200_launch_count())
    sampler.mark()
    t0 = time.perf_counter()
    audio_local, dev_ms, last = 0.0, 0.0, None
    for s in range(args.steps):
        a_, ms, last = step_device(True, keep=bool(args.dump_outputs) and s == args.steps - 1)
        audio_local += a_; dev_ms += ms
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = int(lib.sb200_launch_count()) - launches0
    if last is not None:
        dump_outputs(args.dump_outputs, [a.samples.as_slice() for a in last.fetch()])
        last.close()
    wall_max, audio_total = reduce_pair(wall, audio_local)
    dev_ms_max, _ = reduce_pair(dev_ms, 0.0)
    value = audio_total / wall_max

    # ---------------- e2e ----------------
    step_e2e(); step_e2e()
    barrier()
    e2e_steps = max(args.steps, 10)
    t0 = time.perf_counter()
    e2e_audio = 0.0
    for _ in range(e2e_steps):
        e2e_audio += step_e2e()
    barrier()
    e2e_wall, e2e_audio = reduce_pair(time.perf_counter() - t0, e2e_audio)
    e2e_value = e2e_audio / e2e_wall
    d2h_bytes = int(4 * e2e_audio * SR / e2e_steps)

    # secondary (N > 1): every rank serves its own shard through the public call into its own pinned buffers
    # (independent replicas, no frontend): the upper bound the one-frontend path is measured against
    replicas_value = None
    if world > 1:
        my_idx = shard.lpt_partition([len(b) for b in all_batches], world)[rank]
        local_batches = [all_batches[i] for i in my_idx]
        model.infer_batch_with_values(local_batches)
        barrier()
        t0 = time.perf_counter()
        ra = 0.0
        for _ in range(5):
            ra += sum(len(a) for a in model.infer_batch_with_values(local_batches)) / SR
        barrier()
        rw, ra = reduce_pair(time.perf_counter() - t0, ra)
        replicas_value = ra / rw

    # ---------------- C5: 1024 mixed-length utterances, all arriving at t = 0 (synth/src/benchmarks.rs:55-99) ----------------
    # longest first, in waves of 32 utterances per GPU through the same e2e path; an utterance's latency is the time its
    # wave's audio is in the frontend's hands
    c5 = None
    if quality == "medium" and not args.no_c5:
        nph = workload.mixed_lengths(args.c5_utts)
        c5_ids = [workload.synthetic_ids(int(n), utt=u) for u, n in enumerate(nph)]
        waves = workload.length_buckets([len(x) for x in c5_ids], 32 * world)

        def run_wave(w):
            batch = [c5_ids[i] for i in w]
            if fe is None:
                return sum(len(a) for a in model.infer_batch_with_values(batch)) / SR
            out = fe.synthesize(batch if rank == 0 else None)
            return sum(len(o) for o in out) / SR if rank == 0 else 0.0
        run_wave(waves[0]); run_wave(waves[-1])
        barrier()
        t0 = time.perf_counter()
        done, audio = [], []
        for w in waves:
            audio.append(run_wave(w))
            done.append(time.perf_counter() - t0)
        barrier()
        if rank == 0:
            p50, p99, agg = workload.completion_stats(waves, done, audio)
            c5 = {"workload": f"{args.c5_utts} utterances, N ~ U{{64..512}} phonemes (seed 7), longest first, waves of {32 * world}",
                  "value": agg, "unit": "audio-s/s", "latency_p50_s": p50, "latency_p99_s": p99, "wall_s": done[-1],
                  "audio_s": float(sum(audio)), "waves": len(waves)}

    # ---------------- C1 / C3 as secondary lines (N = 1; same box, same run, own clock record) ----------------
    secondary = {}
    if world == 1 and args.workload == "C2" and not args.no_secondary:
        for name in ("C1", "C3"):
            q2, B2, N2 = workload.CONFIGS[name]
            m2 = model if q2 == quality else sonata_b200.from_config_path(
                voicegen.write_voice(voice_dir, q2), device=local_rank)
            m2.set_backend(args.backend)
            bt = [workload.synthetic_ids(N2, utt=u) for u in range(B2)]
            steps2 = 30 if name == "C1" else 4
            smp = ClockSampler(local_rank); smp.start()
            for _ in range(3):
                m2.infer_batch_with_values(bt)
            torch.cuda.synchronize()
            l0 = int(lib.sb200_launch_count())
            smp.mark()
            t0 = time.perf_counter(); a2 = 0.0
            for _ in range(steps2):
                a2 += sum(len(a) for a in m2.infer_batch_with_values(bt)) / SR
            torch.cuda.synchronize()
            w2 = time.perf_counter() - t0
            l1 = int(lib.sb200_launch_count())
            dms = 0.0
            for _ in range(steps2):
                j = SynthesisJob(m2, bt); dms += j.run(); j.close()
            secondary[name] = {"workload": f"{name}: synthetic-{q2}, {B2} x {N2} phonemes", "e2e_audio_s_per_s": a2 / w2,
                               "e2e_ms_per_step": 1e3 * w2 / steps2, "device_ms_per_step": dms / steps2,
                               "launches_per_step": (l1 - l0) / steps2, "steps": steps2, "clocks": smp.stop()}
            if m2 is not model:
                m2.close()

    if rank == 0:
        peaks = read_peaks()
        # dominant kernel class: HiFi-GAN ResBlock convolutions (dec.mrf*)
        mrf = {k: v for k, v in prof_acc.items() if k.startswith("dec.mrf")}
        mrf_ms = sum(v["ms"] for v in mrf.values()); mrf_l = sum(v["launches"] for v in mrf.values())
        mrf_bytes = sum(v["bytes"] for v in mrf.values()); mrf_flops = sum(v["flops"] for v in mrf.values())
        all_ms = sum(v["ms"] for v in prof_acc.values())
        ach_gbs = mrf_bytes / (mrf_ms * 1e-3) / 1e9 if mrf_ms else 0.0
        arch = voicegen.ARCH[quality]
        frames_rank0 = audio_local * SR / HOP              # frames this rank decoded in the timed steps
        fused_bytes, U_, C_ = 0.0, 1, arch["up_init"]
        for u_ in arch["up_rates"]:
            U_ *= u_; C_ //= 2
            fused_bytes += 2.0 * frames_rank0 * U_ * C_ * 4
        roofline = {
            "bound": "hbm", "kernel": ("conv_tc_kernel" if args.backend >= 1 else "conv_simt_kernel") + " on dec.mrf* (HiFi-GAN ResBlock dilated Conv1d + residual; largest share of the step)",
            "achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach_gbs / peaks["hbm_gbs"],
            "peak_source": f"{peaks['source']} (MEASURED_PEAKS.json hbm_gbs)" if peaks["source"] == "measured" else "fallback 6.65 TB/s",
            "traffic": ncu_traffic(),
            "launches": mrf_l, "avg_launch_ms": mrf_ms / mrf_l if mrf_l else None,
            "bytes_per_launch": mrf_bytes / mrf_l if mrf_l else None,
            "share_of_step": mrf_ms / all_ms if all_ms else None,
            "achieved_tflops": mrf_flops / (mrf_ms * 1e-3) / 1e12 if mrf_ms else 0.0,
            "tensor_peak_tflops": peaks["bf16_tflops_sustained"],
            # the same time against the bytes of a FUSED stage (x in + mean out once per stage, fp32): how far the
            # layer-wise formulation is from what a fully fused ResBlock stage would have to move (DESIGN.md section 3
            # explains why the stages stay layer-wise: shared-memory capacity)
            "fused_stage_bytes_per_step": fused_bytes / args.steps if mrf_ms else None,
            "fused_stage_frac": (fused_bytes / (mrf_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if mrf_ms else None,
            "note": "algorithmic bytes = each conv's input + output (+ the residual when it is NOT the conv input, + the accumulated buffer when read-modify-written) once, fp32, + weights; "
                    "FLOPs at 2/MAC over valid rows",
        }
        regions = {k: {"ms_per_step": v["ms"] / args.steps, "tflops": v["flops"] / max(v["ms"], 1e-9) / 1e9,
                       "gbs": v["bytes"] / max(v["ms"], 1e-9) / 1e6, "launches_per_step": v["launches"] / args.steps}
                   for k, v in prof_acc.items()}
        cpu_base = None
        if not args.no_cpu_baseline and world == 1:
            n_s = 4
            threads = tune_cpu_threads(quality, cores)
            a_, w_ = cpu_reference(quality, NPH, n_s, threads)
            cpu_base = {"value": a_ / w_, "unit": "audio-s/s", "cores": threads, "kind": "port", "host_cpus": cores,
                        "sample": f"{n_s} utterances of the workload ({NPH} phonemes each), B=1 sequential like speak_batch, "
                                  f"PyTorch-CPU port of the reference graph, torch threads auto-tuned to {threads} of {cores}"}
        backend_desc = {1: "tcgen05: bf16x2 split (flow, decoder) + chunk-flushed 3xTF32 (text encoder, duration predictor)",
                        2: "tcgen05 bf16x2 (flow, decoder), fp32 CUDA cores (encoder, duration predictor)", 0: "fp32-simt"}[args.backend]
        line = {
            "metric": "audio-sec/sec", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": 1e3 * wall_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 io; tcgen05 with split operands (2 x bf16 flow/decoder, 3 x tf32 encoder/predictor), fp32 accumulate",
            "data": "synthetic", "config": cfg_desc,
            "device_ms_per_step": dev_ms_max / args.steps, "audio_s_per_step": audio_total / args.steps,
            "backend": backend_desc, "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": int(8 * ids_per_step),
                    "d2h_bytes_per_step": d2h_bytes, "steps": e2e_steps,
                    "path": ("public call speak_batch_ids: host ids -> pinned host waveforms" if world == 1 else
                             "ONE frontend on rank 0: NCCL broadcast of the ids, per-rank batched pass, NCCL all-reduce of the frame "
                             "counts, device->host copies into one page-locked host segment shared by the ranks"),
                    "per_rank_replicas": replicas_value},
            "roofline": roofline, "regions": regions, "cpu_baseline": cpu_base, "c5": c5, "secondary": secondary or None,
        }
        sys.stdout.flush()
        os.dup2(_stdout_fd, 1)
        print(json.dumps(line), flush=True)
        sys.stdout.flush()
        os.dup2(2, 1)
    if fe is not None:
        fe.close()
    model.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
