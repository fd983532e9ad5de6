#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: concurrent audio streams x frames / second on N B200s.

A "step" is one pass of the hot path (frontend + MixedNet, `mww_predict_clip`) over one batch of
synthetic 16 kHz int16 audio: 65 536 streams x 3 s (= 300 ten-ms frames, 100 model steps per stream)
per GPU -- BASELINE.json configs[1].  Streams are independent, so N GPUs run N shards of 65 536
streams each with no data-path collective (weak scaling; configs[4] = 8 x 65 536 = 524 288 streams).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--model f32|int8] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  Keys beyond the driver contract:
  roofline      dominant kernel (K1 spectral) achieved algorithmic GB/s vs MEASURED_PEAKS.json
  kernels       per-kernel-class device ms/step from CUDA events recorded by the library on the launch stream
  cpu_baseline  the CPU oracle (the reference's own native dependencies are not installable: "port") on the
                box's host cores, bounded sample
  e2e           same metric through mww_predict_clip_host with pinned HOST buffers (H2D + D2H inside the timed region)
"""

from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
STREAMS_PER_GPU = 65536
SAMPLES_PER_STEP = 48000          # 3 s -> 300 frames / stream / step
FRAMES_PER_STEP = SAMPLES_PER_STEP // 160
K1_ALG_BYTES_PER_FRAME = 320      # 160 new int16 samples per 10 ms frame: the only mandatory HBM traffic of K1 (DESIGN.md)
METRIC = "streams_x_frames_per_sec"
UNIT = "frames/s"
DUMP_BYTES = 64 * 10**6           # --dump-outputs: at most this much in all


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="f32", choices=["f32", "int8"])
    ap.add_argument("--streams", type=int, default=STREAMS_PER_GPU, help="streams per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-wc", type=int, default=0, help="e2e leg: 1 = the host AUDIO buffer is write-combined pinned memory (mww_host_alloc_wc)")
    ap.add_argument("--ingest-mode", default="auto", choices=["auto", "direct", "staged"],
                    help="N > 1: how a rank reads its block of the ingest rank's buffer -- direct: the frontend kernel reads the peer-mapped "
                         "buffer in place over NVLink; staged: the rank's copy engine pulls tile t+1 while tile t computes; auto: staged once "
                         "the pull alone is slower than a rank's compute (the ingest GPU's NVLink egress is the bottleneck), else direct")
    ap.add_argument("--ingest-share", type=float, default=None,
                    help="N > 1: the ingest rank's share of the streams as a fraction of an equal share (default 1; 0 = it only feeds its peers)")
    ap.add_argument("--tiles", type=int, default=0, help="pipeline tiles per rank of the N > 1 ingest (0 = library default, 16)")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the legs for the other BASELINE.json configurations (the other model dtype in clip mode, live 30 ms steps "
                         "for both dtypes, feature extractor only)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the probabilities the last timed step returned as DIR/probs.npy (float32); the "
                         "input audio is seeded, so runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the GPU path (--impl b200)")
    return args


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy in float32.  An array larger than its share of DUMP_BYTES keeps a fixed sample
    of its rows (streams): np.random.default_rng(0).choice(rows, k, replace=False), in stream order, so every run with the
    same arguments writes the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096            # room for the .npy header
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > share:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], share // a[0].nbytes, replace=False))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def model_blob(kind: str) -> bytes:
    with open(os.path.join(GOLDEN, "okay_nabu_synth_%s.mww" % kind), "rb") as f:
        return f.read()


def config_dict(args, world):
    return {
        "workload": "configs[1]: %d synthetic 16 kHz streams x %d frames (3 s) per step per GPU, okay_nabu mixednet %s, clip mode"
                    % (args.streams, FRAMES_PER_STEP, "int8 (TFLite semantics)" if args.model == "int8" else "fp32"),
        "streams_per_gpu": args.streams, "streams_total": args.streams * world, "frames_per_stream_per_step": FRAMES_PER_STEP,
        "samples_per_stream_per_step": SAMPLES_PER_STEP, "parallelism": "independent stream shards x%d, no collective" % world,
        "l2": "inputs %.1f GB per GPU per step >> 126 MB L2 (no flush needed)" % (args.streams * SAMPLES_PER_STEP * 2 / 1e9),
        "weights": "synthetic okay_nabu seed 0 (tests/golden)",
    }


# --------------------------------------------------------------------------------------------
# CPU oracle legs

def cpu_sample(n_streams: int) -> np.ndarray:
    from microwakeword_b200.synth_audio import synth_audio
    base = np.stack([synth_audio(SAMPLES_PER_STEP, 7000 + i) for i in range(64)])
    reps = (n_streams + 63) // 64
    return np.ascontiguousarray(np.tile(base, (reps, 1))[:n_streams])


def host_cores():
    """(threads to use, facts about the host): the affinity mask rather than os.cpu_count(), and the cgroup CPU quota when
    the container has one -- a 128-thread box whose container may only burn 32 CPUs' worth of time is a 32-core baseline."""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    facts = {"os_cpu_count": os.cpu_count(), "affinity": n}
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        facts["cgroup_cpu_max"] = "%s %s" % (quota, period)
        if quota != "max":
            facts["cgroup_cpus"] = float(quota) / float(period)
    except (OSError, ValueError):
        pass
    # threads to use = what the container may actually burn: oversubscribing a 16-CPU quota with 128 threads cost the r01
    # baseline a third of its throughput (VERDICT r01)
    if facts.get("cgroup_cpus"):
        n = min(n, max(int(facts["cgroup_cpus"] + 0.999), 1))
    facts["threads_used"] = max(n, 1)
    return max(n, 1), facts


def time_cpu_single_thread(kind: str) -> float:
    """frames/s of ONE oracle thread (a few hundred ms): shows how the multi-thread figure scales on this host"""
    import oracle
    audio = cpu_sample(16)
    t0 = time.perf_counter()
    oracle.run_pipeline(model_blob(kind), audio, want_features=False, threads=1)
    return audio.shape[0] * 298 / max(time.perf_counter() - t0, 1e-6)


def time_cpu(kind: str, cores: int, target_s: float = 12.0):
    """Times the CPU oracle (frontend + MixedNet) over a bounded sample with `cores` threads."""
    import oracle
    blob = model_blob(kind)
    probe = cpu_sample(2 * cores)
    t0 = time.perf_counter()
    oracle.run_pipeline(blob, probe, want_features=False, threads=cores)
    dt = max(time.perf_counter() - t0, 1e-3)
    rate = probe.shape[0] * 298 / dt
    n_streams = int(min(16384, max(4 * cores, rate * target_s / 298)))
    n_streams = max(cores, n_streams // cores * cores)
    audio = cpu_sample(n_streams)
    t0 = time.perf_counter()
    oracle.run_pipeline(blob, audio, want_features=False, threads=cores)
    dt = time.perf_counter() - t0
    frames = n_streams * 298
    return frames / dt, "%d streams x 3 s (298 frames each from reset), %d threads, %.1f s" % (n_streams, cores, dt)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores, host = host_cores()
    single = time_cpu_single_thread(args.model)
    vals, sample = [], ""
    for i in range(args.warmup + args.steps):
        v, sample = time_cpu(args.model, cores, target_s=max(2.0, min(12.0, 120.0 / max(args.warmup + args.steps, 1))))
        if i >= args.warmup:
            vals.append(v)
    value = statistics.median(vals) if vals else 0.0
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.model == "f32" else "int8", "data": "synthetic",
        "config": config_dict(args, max(args.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "single_thread_value": single, "host": host,
                         "note": "the reference's own CPU path (tf.lite.Interpreter + pymicro_features) is not installable here; "
                                 "this is the C oracle restating it, one stream per thread"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------
# GPU arm

def synth_audio_device(torch, n_streams, n_samples, seed, device):
    """Gaussian noise with log-uniform level + two tone bursts per stream; 64 edge-case streams overwritten."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n_streams, n_samples), dtype=torch.int16, device=device)
    t = torch.arange(n_samples, device=device, dtype=torch.float32)
    chunk = 4096 if n_samples > 4096 else 1 << 18
    for s0 in range(0, n_streams, chunk):
        n = min(chunk, n_streams - s0)
        sigma = torch.exp(torch.empty(n, 1, device=device).uniform_(np.log(50.0), np.log(8000.0), generator=g))
        x = torch.randn((n, n_samples), device=device, generator=g) * sigma
        for _ in range(2):
            f = torch.empty(n, 1, device=device).uniform_(200.0, 4000.0, generator=g)
            a = torch.empty(n, 1, device=device).uniform_(500.0, 12000.0, generator=g)
            start = torch.empty(n, 1, device=device).uniform_(0, max(n_samples - 8000, 1), generator=g)
            length = torch.empty(n, 1, device=device).uniform_(1600, 8000, generator=g)
            mask = (t[None, :] >= start) & (t[None, :] < start + length)
            x += mask * a * torch.sin(2 * np.pi * f * t[None, :] / 16000.0)
        out[s0:s0 + n] = x.round_().clamp_(-32768, 32767).to(torch.int16)
    from microwakeword_b200.synth_audio import edge_case_audio
    edge = torch.from_numpy(edge_case_audio(n_samples)).to(device)
    k = min(edge.shape[0], n_streams)
    out[:k] = edge[:k]
    return out


class ClockSampler:
    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.path = tempfile.mktemp(prefix="mww_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None
        atexit.register(self.stop)          # the sampler must not outlive a benchmark that fails before stop()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        proc, self.proc = self.proc, None
        if proc is None:
            return out
        proc.terminate()
        try:
            proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            proc.kill()
            proc.wait()
        sm, mx, reasons = [], [], set()
        try:
            for ln in open(self.path):
                p = [x.strip() for x in ln.split(",")]
                if len(p) < 8:
                    continue
                try:
                    sm.append(float(p[1])); mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per K1 launch from the committed ncu --set full capture summary, if present."""
    p = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def issue_roofline(tipf, frames_per_launch, kernel_ms, clock_info):
    sm_hz = ((clock_info or {}).get("sm_mhz") or 1965.0) * 1e6
    peak_issue = 148 * 4 * 32 * sm_hz            # 4 schedulers/SM x 1 warp-instruction/clk x 32 threads
    ach = tipf * frames_per_launch / (kernel_ms / 1e3)
    return {"thread_instr_per_frame": tipf, "achieved_thread_instr_per_s": ach, "peak_thread_instr_per_s": peak_issue,
            "frac": ach / peak_issue, "source": "instructions per frame from the committed ncu capture; duration live from CUDA events"}


def k1_roofline(prof, S, steps, clock_info):
    """HBM roofline of the dominant kernel (the spectral frontend kernel) from the library's own CUDA events."""
    peak, peak_src = measured_peaks()
    k1_ms, k1_n = prof["k1_spectral"]
    if not k1_n:
        return None
    frames_per_launch = S * FRAMES_PER_STEP * steps / k1_n
    per_launch_ms = k1_ms / k1_n
    achieved = K1_ALG_BYTES_PER_FRAME * frames_per_launch / (per_launch_ms / 1e3) / 1e9
    tr = ncu_traffic()
    roof = {"bound": "hbm", "kernel": (tr or {}).get("kernel", "k1_spectral_kernel"), "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": peak_src, "traffic": ((tr or {}).get("dram_bytes_per_unit") or 0) * frames_per_launch or None,
            "traffic_source": (tr or {}).get("source"),
            "alg_bytes_per_frame": K1_ALG_BYTES_PER_FRAME, "frames_per_launch": frames_per_launch,
            "share_of_step": k1_ms / max(sum(v[0] for v in prof.values()), 1e-9),
            "note": "the frontend kernel is integer-ALU bound by construction (~30k thread-instructions per 320-byte frame, ncu): the HBM "
                    "fraction is low because the kernel is instruction-issue bound; see `issue`, DESIGN.md and profiles/"}
    tipf = (tr or {}).get("thread_instr_per_unit")
    if tipf:
        roof["issue"] = issue_roofline(tipf, frames_per_launch, per_launch_ms, clock_info)
    return roof


def run_gpu(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and "CUDA_VISIBLE_DEVICES" not in os.environ:
        # a rank only ever needs the GPUs of its own job: nothing (NCCL topology probing, IPC, a stray context) can touch the
        # box's other GPUs (r01: blips on GPUs 4-7 during the 2-GPU run)
        os.environ["CUDA_VISIBLE_DEVICES"] = ",".join(str(i) for i in range(int(os.environ.get("LOCAL_WORLD_SIZE", world))))
    import torch
    import torch.distributed as dist

    from microwakeword_b200.engine import StreamEngine, bind_host_thread, host_array

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    affinity_before = os.sched_getaffinity(0)
    numa_node = bind_host_thread(local_rank)           # before anything pins host memory: buffers land next to this rank's GPU
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, reps):
        """max over ranks of the CUDA-event time of `reps` calls, in ms per call"""
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b)) / reps

    S = args.streams
    n_probs = FRAMES_PER_STEP // 3 + 1
    eng = StreamEngine(model_blob(args.model), n_streams=S, device=local_rank)
    audio = synth_audio_device(torch, S, SAMPLES_PER_STEP, 1234 + rank, device)
    probs = torch.empty((S, n_probs), dtype=torch.float32, device=device)
    frames_per_step_all = S * FRAMES_PER_STEP * world

    # ---- the shard's own audio already resident in HBM: `value` at N = 1, `value_presharded` at N > 1 ----
    eng.reset()
    clocks = ClockSampler(local_rank) if rank == 0 else None           # samples every 100 ms from warm-up on
    for _ in range(max(args.warmup, 1)):
        eng.predict_clip(audio, out=probs)
    barrier()
    l0 = eng.launch_count
    eng.profile(True)
    last = {}

    def resident_step():
        last["probs"] = eng.predict_clip(audio, out=probs)
    ms_resident = timed(resident_step, args.steps)
    launches = (eng.launch_count - l0)
    prof = eng.profile_read()
    eng.profile(False)
    # what the last timed step returned, copied before the legs below reuse `probs`
    outputs = {"probs": last["probs"].cpu().numpy()} if args.dump_outputs and world == 1 else None
    checksum = float(probs[:, :100].double().sum().item())
    kernels = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps} for k, v in prof.items()}

    # ---- N > 1, BASELINE.json configs[4] as SURVEY.md 8(d) defines it: audio originates on rank 0, every rank pulls its
    # block over NVLink while it computes (copy engines, CUDA IPC peer mapping; DESIGN.md section 5), scores are gathered
    # back on rank 0 (NCCL) -- scatter, compute and gather all inside the timed region ----
    ingest_info, ms_per_step = None, ms_resident
    if world > 1:
        from microwakeword_b200.sharding import IngestBuffer, ShardedEngine, gather_probs, ingest_shares, scatter_audio
        from microwakeword_b200 import _lib as lib_mod
        import ctypes
        total = S * world
        ingest = IngestBuffer(total, SAMPLES_PER_STEP, src=0, device=device)
        if rank == 0:
            ingest.buffer[:S].copy_(audio)
            for r in range(1, world):                  # rank 0 holds every stream's audio (each block has its own seed)
                ingest.buffer[r * S:(r + 1) * S].copy_(synth_audio_device(torch, S, SAMPLES_PER_STEP, 1234 + r, device))
        torch.cuda.synchronize()
        cur = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        # (i) where the time can go: the pull alone (copy engines, no kernels), equal blocks
        stage = torch.empty((max(S // 16, 1), SAMPLES_PER_STEP), dtype=torch.int16, device=device)

        def pull_only():
            dist.barrier()
            rows = stage.shape[0]
            for s0 in range(0, S if rank != 0 else 0, rows):
                n = min(rows, S - s0)
                lib_mod.check(None, lib_mod.lib().mww_copy_async(stage.data_ptr(), ingest.block_ptr(rank * S + s0), n * SAMPLES_PER_STEP * 2, cur()))
        pull_only()
        pull_ms = timed(pull_only, 2)
        del stage
        # the ingest rank's share of the streams: equal by default.  (Measured at N = 8, staged mode: equal shares 54.9 ms, the
        # ingest rank feeding only 63.7 ms -- all 8 S streams then cross its NVLink instead of 7 S; DESIGN.md section 5.)
        src_share = 1.0 if args.ingest_share is None else float(args.ingest_share)
        why = "equal shares (default)" if args.ingest_share is None else "--ingest-share"
        egress_bound = pull_ms > ms_resident
        mode = args.ingest_mode if args.ingest_mode != "auto" else ("staged" if egress_bound else "direct")
        ingest_tiles = 0 if mode == "direct" else (args.tiles or 16)
        shares = ingest_shares(total, world, 0, src_share)
        sh = ShardedEngine(model_blob(args.model), total, local_rank, shares=None if src_share == 1.0 else shares)
        my_probs = torch.empty((max(sh.count, 1), n_probs), dtype=torch.float32, device=device) if sh.count != S else probs
        torch.cuda.synchronize()
        gathered = None

        def ingest_step():
            nonlocal gathered
            gathered = sh.predict_clip_ingest(ingest, tiles=ingest_tiles, out=my_probs[:sh.count] if sh.count else None)

        count_launches = lambda: sh.engine.launch_count if sh.engine is not None else 0
        sh.reset()
        ingest_step()
        for _ in range(max(args.warmup, 1)):
            ingest_step()
        l0 = count_launches()
        ms_per_step = timed(ingest_step, args.steps)
        if args.dump_outputs and rank == 0:
            outputs = {"probs": gathered.cpu().numpy()}
        lt = torch.tensor([count_launches() - l0], dtype=torch.int64, device=device)
        dist.all_reduce(lt, op=dist.ReduceOp.MAX)
        launches = int(lt.item())                      # per rank (the ingest rank launches nothing when its share is 0)
        # who is the slow one: every rank's own device time for the same steps (the timed value is the max)
        barrier()
        r0e, r1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0e.record()
        for _ in range(args.steps):
            ingest_step()
        r1e.record()
        torch.cuda.synchronize()
        mine_ms = torch.tensor([r0e.elapsed_time(r1e) / args.steps], dtype=torch.float64, device=device)
        all_ms = [torch.zeros_like(mine_ms) for _ in range(world)]
        dist.all_gather(all_ms, mine_ms)
        per_rank_ms = [float(t.item()) for t in all_ms]
        ingest_checksum = float(gathered[:S, :100].double().sum().item()) if rank == 0 else 0.0
        # per-rank tile timeline of one more step (CUDA events on the library's copy and compute streams)
        max_tiles = 64
        tl = torch.full((max_tiles, 4), -1.0, dtype=torch.float32, device=device)
        if sh.engine is not None:
            sh.engine.profile(True)
        ingest_step()
        if sh.engine is not None:
            t_np = sh.engine.timeline_read(max_tiles)
            sh.engine.profile_read()
            sh.engine.profile(False)
            tl[:len(t_np)] = torch.from_numpy(t_np).to(device)
        all_tl = [torch.zeros_like(tl) for _ in range(world)]
        dist.all_gather(all_tl, tl)
        timelines = [[[round(float(x), 3) for x in row] for row in t.cpu().tolist() if row[0] >= 0] for t in all_tl]
        # every rank's block through the ingest path == the same block computed from resident audio (both from reset state)
        sh.reset()
        ingest_step()
        same = audio_same = True
        diff = 0.0
        if sh.count:
            mine = torch.empty((sh.count, SAMPLES_PER_STEP), dtype=torch.int16, device=device)
            lib_mod.check(None, lib_mod.lib().mww_copy_async(mine.data_ptr(), ingest.block_ptr(sh.start), sh.count * SAMPLES_PER_STEP * 2, cur()))
            # the block this rank pulled is the audio the owning seeds synthesise (generated here, on another GPU of the same kind)
            for r in range(world):
                lo, hi = max(sh.start, r * S), min(sh.start + sh.count, (r + 1) * S)
                if lo < hi:
                    ref = audio if r == rank else synth_audio_device(torch, S, SAMPLES_PER_STEP, 1234 + r, device)
                    audio_same = audio_same and torch.equal(mine[lo - sh.start:hi - sh.start], ref[lo - r * S:hi - r * S])
                    del ref
            chk = eng if sh.count == S else StreamEngine(model_blob(args.model), n_streams=sh.count, device=local_rank)
            chk.reset()
            resident = chk.predict_clip(mine)
            pulled = my_probs[:sh.count, :resident.shape[1]]
            same = torch.equal(resident, pulled)
            diff = float((resident - pulled).abs().max().item())
            if chk is not eng:
                chk.close()
            del mine, resident
        diag = torch.tensor([1 if same else 0, 1 if audio_same else 0], dtype=torch.int32, device=device)
        dist.all_reduce(diag, op=dist.ReduceOp.MIN)
        max_diff = torch.tensor([diff], dtype=torch.float64, device=device)
        dist.all_reduce(max_diff, op=dist.ReduceOp.MAX)
        eng.reset()

        # (ii) the plain serialised NCCL scatter -> compute -> gather (equal blocks)
        def nccl_serial():
            local = scatter_audio(ingest.buffer if rank == 0 else None, total, SAMPLES_PER_STEP, src=0, device=device)
            gather_probs(eng.predict_clip(local, out=probs), total, dst=0)
        nccl_serial()
        nccl_ms = timed(nccl_serial, 2)
        ingest_info = {
            "how": "audio for all %d streams in rank 0's HBM, mapped into every rank with CUDA IPC; " % total + (
                   "every rank's frontend kernel reads its block in place over NVLink (zero-copy, no staging)" if mode == "direct" else
                   "every rank's copy engine pulls its block tile by tile over NVLink while the previous tile computes (mww_predict_clip_remote, "
                   "staged)") + "; scores gathered to rank 0 with NCCL; a one-element all-reduce per step orders the reads after the ingest rank's writes",
            "mode": mode, "mode_rule": "%s (pull alone %.1f ms %s pre-sharded compute %.1f ms)" % (
                args.ingest_mode, pull_ms, ">" if egress_bound else "<=", ms_resident),
            "streams_per_rank": shares, "ingest_rank_share": src_share, "ingest_rank_share_rule": why,
            "tiles_per_rank": ingest_tiles, "per_rank_ms_per_step": per_rank_ms,
            "nvlink_bytes_out_of_rank0_per_step": (total - shares[0]) * SAMPLES_PER_STEP * 2,
            "egress_floor_ms": pull_ms, "pull_only_gbs_out_of_rank0": S * SAMPLES_PER_STEP * 2 * (world - 1) / (pull_ms / 1e3) / 1e9,
            "egress_floor_note": "the pull alone with EQUAL blocks (S (N - 1) streams leave rank 0); with ingest_rank_share 0 all N S streams leave it",
            "value_presharded": frames_per_step_all / (ms_resident / 1e3), "ms_per_step_presharded": ms_resident,
            "nccl_serial": {"value": frames_per_step_all / (nccl_ms / 1e3), "ms_per_step": nccl_ms,
                            "note": "torch.distributed scatter of int16 audio from rank 0, compute, gather of float32 scores (NCCL), serialised"},
            "probs_checksum_rank0_block": ingest_checksum,
            "every_rank_block_equals_resident_path": bool(int(diag[0].item()) == 1),
            "every_rank_pulled_audio_equals_own_synthesis": bool(int(diag[1].item()) == 1),
            "max_abs_prob_difference_to_resident_path": float(max_diff.item()),
            "tile_timeline_ms": {"columns": ["copy_start", "copy_end", "kernels_start", "kernels_end"],
                                 "note": "one step, per rank, per tile; ms after that rank's first copy started", "ranks": timelines},
        }
        torch.cuda.synchronize()
        barrier()
        ingest.close()
        del sh

    clock_info = clocks.stop() if clocks else None
    value = frames_per_step_all / (ms_per_step / 1e3)
    roof = k1_roofline(prof, S, args.steps, clock_info)

    # ---- e2e through the host-buffer C-ABI call (pinned buffers on this GPU's NUMA node) ----
    e2e = None
    if not args.no_e2e:
        ha = host_array((S, SAMPLES_PER_STEP), np.int16, local_rank, write_combined=bool(args.e2e_wc))
        hp = host_array((S, n_probs), np.float32, local_rank)
        torch.from_numpy(ha).copy_(audio)
        torch.cuda.synchronize()
        eng.reset()
        for _ in range(2):
            eng.predict_clip_host(ha, out=hp)
        e2e_steps = max(2, min(args.steps, 4))
        t0 = time.perf_counter()
        e2e_ms = timed(lambda: eng.predict_clip_host(ha, out=hp), e2e_steps)
        wall_ms = (time.perf_counter() - t0) * 1e3
        e2e = {"value": frames_per_step_all / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": S * SAMPLES_PER_STEP * 2 * world,
               "d2h_bytes_per_step": S * (FRAMES_PER_STEP // 3) * 4 * world, "ms_per_step": e2e_ms, "steps": e2e_steps,
               "h2d_gbs_per_gpu": S * SAMPLES_PER_STEP * 2 / (e2e_ms / 1e3) / 1e9,
               "api": "mww_predict_clip_host (pinned host int16 audio in, float32 probabilities out; buffers from mww_host_alloc)",
               "audio_buffer_write_combined": bool(args.e2e_wc), "host_buffers_numa_node": ha.base.base.numa_node, "rank_bound_to_numa_node": numa_node,
               "checksum_matches_device_path": bool(abs(float(hp[:, :100].astype(np.float64).sum()) - checksum) < 1e-3 * max(1.0, abs(checksum)))}
        del ha, hp

    # ---- the other single-GPU configurations of BASELINE.json, each with its own roofline (rank-local, every rank runs them) ----
    def live_traffic(kind, n_streams):
        """DRAM bytes per launch of the fp32 live NN kernel, from the committed ncu --set full capture (per stream-step x streams)"""
        path = os.path.join(ROOT, "profiles", "live_traffic.json")
        if kind != "f32" or not os.path.exists(path):
            return None
        return json.load(open(path))["dram_bytes_per_unit"] * n_streams

    def live_leg(kind, n_live=480):
        """live mode: step() calls with `n_live` new samples per stream; the ring state round-trips HBM on every call"""
        le = eng if kind == args.model else StreamEngine(model_blob(kind), n_streams=S, device=local_rank)
        calls = max(SAMPLES_PER_STEP // n_live, 1)
        le.reset()
        chunks = [audio[:, i * n_live:(i + 1) * n_live].contiguous() for i in range(min(calls, 8))]
        for c in chunks[:4]:
            le.predict_clip(c, out=probs)
        state = {"i": 0}

        def one():
            le.predict_clip(chunks[state["i"] % len(chunks)], out=probs)
            state["i"] += 1
        le.profile(True)
        live_ms = timed(one, calls)
        lp = le.profile_read()
        le.profile(False)
        frames = S * world * (n_live // 160)
        # live-step NN, algorithmic bytes per stream-step (SURVEY.md 8d): every ring row read once (4 176 elements), one new
        # row per ring + the 2-row first-conv ring written (368 elements), 3 uint16 feature rows in, one probability out
        nn_ms = lp["mixednet"][0] / max(lp["mixednet"][1], 1)
        eb = 4 if kind == "f32" else 1
        step_bytes = 4176 * eb + 368 * eb + 3 * 80 + 4
        peak, peak_src = measured_peaks()
        nn_gbs = S * step_bytes / (nn_ms / 1e3) / 1e9 if nn_ms else None
        out = {"workload": "configs[1]/[2] streams stepped live: %d calls of %d new samples (one model step) for %d streams, %s" % (calls, n_live, S, kind),
               "samples_per_call": n_live, "calls": calls, "value": frames / (live_ms / 1e3), "unit": UNIT, "ms_per_call": live_ms,
               "kernels_ms_per_call": {k: v[0] / calls for k, v in lp.items()},
               "roofline": {"bound": "hbm", "kernel": "nn_f32_live3_kernel" if kind == "f32" else "nn_i8_live_kernel", "achieved": nn_gbs, "peak": peak,
                            "unit": "GB/s", "frac": nn_gbs / peak if nn_gbs else None, "peak_source": peak_src,
                            "alg_bytes_per_stream_step": step_bytes, "kernel_ms": nn_ms, "traffic": live_traffic(kind, S)},
               "realtime_streams_capacity": S * world * (n_live / 16.0) / live_ms}
        if le is not eng:
            le.close()
        return out

    def clip_leg(kind):
        ce = StreamEngine(model_blob(kind), n_streams=S, device=local_rank)
        for _ in range(3):
            ce.predict_clip(audio, out=probs)
        ce.profile(True)
        steps = max(3, min(args.steps, 5))
        ms = timed(lambda: ce.predict_clip(audio, out=probs), steps)
        cp = ce.profile_read()
        ce.profile(False)
        out = {"workload": "configs[2]: %d streams x %d frames per step, okay_nabu mixednet %s, clip mode" % (S, FRAMES_PER_STEP, kind),
               "dtype": kind, "value": S * FRAMES_PER_STEP * world / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
               "kernels": {k: {"ms_per_step": v[0] / steps} for k, v in cp.items()}, "roofline": k1_roofline(cp, S, steps, clock_info)}
        ce.close()
        return out

    def features_leg():
        """BASELINE.json configs[3]: the feature extractor alone on 1 M 30 ms windows (streaming and stateless)"""
        feat = {}
        peak, peak_src = measured_peaks()
        tr = ncu_traffic() or {}
        for name, fs, fn in (("streaming_4096x256", 4096, 160 * 256 + 320), ("stateless_1048576x480", 1 << 20, 480)):
            fe = StreamEngine(None, n_streams=fs, device=local_rank)
            fa = synth_audio_device(torch, fs, fn, 99 + rank, device)
            n_fr = (fn - 480) // 160 + 1
            fo = torch.empty((fs, n_fr, 40), dtype=torch.uint16, device=device)

            def one():
                fe.reset()                                   # every pass starts from the reset frontend state, like a new clip
                fe.features(fa, out=fo)
            for _ in range(3):
                one()
            f_ms = timed(one, 10)
            windows = fs * n_fr * world
            alg = (fn * 2 + n_fr * 80) / n_fr
            gbs = fs * (fn * 2 + n_fr * 80) / (f_ms / 1e3) / 1e9
            feat[name] = {"windows": windows, "ms": f_ms, "windows_per_s": windows / (f_ms / 1e3), "alg_bytes_per_window": alg,
                          "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "peak_source": peak_src,
                                       "traffic": None,
                                       "issue": issue_roofline(tr["thread_instr_per_unit"], fs * n_fr, f_ms, clock_info) if tr.get("thread_instr_per_unit") else None,
                                       "note": "integer-ALU bound like the clip frontend: the issue-slot fraction is the binding one"}}
            fe.close()
            del fa, fo
        return feat

    extras = {}
    if not args.no_extra:
        other = "int8" if args.model == "f32" else "f32"
        extras[other] = clip_leg(other)
        extras["live"] = live_leg(args.model)
        extras["live_" + other] = live_leg(other)
        extras["features_only"] = features_leg()

    # ---- CPU baseline beside it (rank 0, N = 1 only; all the host cores the container may use) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, affinity_before)
        cores, host = host_cores()
        v, sample = time_cpu(args.model, cores)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
               "single_thread_value": time_cpu_single_thread(args.model), "host": host}

    if rank == 0:
        cfg = config_dict(args, world)
        if world > 1:
            cfg["workload"] = "configs[4]: %d synthetic 16 kHz streams x %d frames (3 s) per step on %d GPUs (65 536 per rank), audio originating on rank 0 " \
                              "(pulled over NVLink inside the timed region), scores gathered on rank 0; okay_nabu mixednet %s, clip mode" \
                              % (S * world, FRAMES_PER_STEP, world, args.model)
            cfg["parallelism"] = "independent stream shards x%d; scatter (copy-engine pull over NVLink) + NCCL gather inside the timed region" % world
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.model == "f32" else "int8", "data": "synthetic",
            "config": cfg, "clocks": clock_info, "gpu_launches": int(launches),
            "kernels": kernels, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "ingest": ingest_info,
            "probs_checksum": checksum, "realtime_streams_capacity": value / 100.0,
        }
        line.update(extras)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True     # the project's modules are imported below this point: no __pycache__ in the (maybe read-only) tree
    # libraries print to stdout on their own (NCCL's version banner, for one): keep the real stdout for the ONE JSON line and
    # send everything else to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
