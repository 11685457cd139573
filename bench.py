#!/usr/bin/env python
"""
bench.py -- utterances/second of the mask-based MVDR beamformer hot path.

Workload (BASELINE.json configs[1], "metric"): 4-channel MVDR, oracle IRM mask,
16 kHz, 10 s utterances (N = 160000), 512-point STFT / hop 256 / hann /
center, batch = 256 utterances per GPU per step.  A "step" is one pass of the
hot path over one resident batch:

    setk_stft_cov (fused STFT + Rs/Rn) -> setk_weights (fp64 MVDR) ->
    setk_apply_istft_pcm16 (fused beamform + iSTFT + peak normalisation + the wav
    writer's float -> PCM-16 conversion)

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by torch.distributed.run, one rank per GPU; utterances shard
across ranks with no data-path collective ("scaling": "weak").  EVERY batch's
enhanced audio (PCM-16, what the wav files would hold) is gathered to rank 0 by
NCCL inside the timed region, asynchronously to the kernels (SURVEY.md section 8e).

Prints one JSON line (rank 0).  Keys beyond the base contract:
  roofline      the dominant kernel (fused STFT+covariance): algorithmic bytes
                per launch / CUDA-event time of that call, vs MEASURED_PEAKS.json
  cpu_baseline  the reference's CPU path (oracle port; the reference's own modules
                when its tree is present) on this box's host cores (N = 1 only)
  e2e           same metric through the public API with HOST (pinned) buffers: PCM-16
                audio + float32 masks in, PCM-16 enhanced audio out, every step
  configs       the other BASELINE.json configurations (3, 4, 5) at this GPU count
`--impl reference` times the reference's CPU implementation of the path with all
host cores and prints the same JSON line with "impl": "reference".
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "utts/sec 4-ch MVDR 10s@16kHz at 1/2/4/8 B200; STFT+cov HBM GB/s vs peak"   # BASELINE.json
UNIT = "utts/s"
C, N, FRAME_LEN, HOP, NFFT = 4, 160000, 512, 256, 512
BATCH = 256
F = NFFT // 2 + 1
T = 1 + N // HOP            # center=True
WORKLOAD = "cfg2: 4-ch MVDR, IRM mask, 16 kHz x 10 s, 512/256 hann center, batch 256 per GPU"


def config_dict(world, batch=BATCH):
    """The workload both arms are measured on (identical in both JSON lines)."""
    return {"workload": WORKLOAD, "batch_per_gpu": batch, "global_batch": batch * world,
            "parallelism": f"utterance-sharded x{world}, no data-path collective; every batch's "
                           f"PCM-16 result gathered to rank 0 inside the timed region",
            "l2": f"inputs {batch * (C * N + T * F) * 4 / 1e6:.0f} MB per step exceed the 126 MB L2 "
                  f"(no flush needed)"}


def algorithmic_bytes_stft_cov(c=C, n=N, n_fft=NFFT, hop=HOP):
    """SURVEY.md section 8d: audio f32 + mask f32 + Rs,Rn c64, per utterance."""
    f, t = n_fft // 2 + 1, 1 + n // hop
    return 4 * c * n + 4 * t * f + 2 * 8 * f * c * c


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(batch):
    """
    dram__bytes_read + dram__bytes_write of the dominant kernel per launch, from the
    committed `ncu --set full` capture (profiles/r2_traffic.json); only valid for the
    batch it was captured on, else null.
    """
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                d = json.load(fh)
            if batch * algorithmic_bytes_stft_cov() == d["algorithmic_bytes_per_launch"]:
                return d["traffic_bytes_per_launch"]
        except Exception:
            continue
    return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6),
                                  ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        # median over the upper half of the samples = the clock under load (the sampler also
        # sees the idle gaps between the timed phases)
        busy = sm[len(sm) // 2:] if sm else []
        med = busy[len(busy) // 2] if busy else None
        return {"sm_mhz": med, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_model():
    try:
        with open("/proc/cpuinfo") as fh:
            for ln in fh:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ------------------------------------------------------------------ CPU arm ---
def cpu_steps(steps, warmup, budget_s, cores):
    """
    The reference's CPU path for `steps` steps.  A step is the GPU step's 256 utterances when
    the whole run fits `budget_s` at ~20 utterances/s/core, else a bounded sample of it (a
    multiple of the worker count); the line says which.
    """
    from oracle import cpu_bench
    fit = int(budget_s * 20.0 * cores / max(1, steps + warmup))
    ups = BATCH if fit >= BATCH else max(cores, (fit // cores) * cores)
    return cpu_bench.run_steps(C, N, steps, warmup, ups, cores)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.cpu_bench import usable_cores
    cores = usable_cores()
    t0 = time.time()
    r = cpu_steps(args.steps, args.warmup, args.cpu_budget, cores)
    sample = (f"each step = {r['utts_per_step']} utterances of the {BATCH}-utterance GPU step"
              f"{'' if r['utts_per_step'] == BATCH else ' (bounded sample)'}, spread over {r['workers']} "
              f"single-threaded worker processes (run.pl nj={r['workers']}), distinct utterances, "
              f"compute only")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "utts_per_step": r["utts_per_step"],
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (STFT/cov/apply), f64 (per-bin weight solve)",
        "data": "synthetic",
        "config": config_dict(max(1, args.gpus), args.batch),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": cores, "kind": r["kind"],
                         "sample": sample, "cpu": cpu_model(), "reference_root": r["reference_root"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "timed_s": r["seconds"], "wall_s": time.time() - t0,
    }
    emit(line)


# --------------------------------------------------------------- NUMA binding ---
def numa_bind(dev_index):
    """
    Pin this rank to the CPUs of its GPU's NUMA node BEFORE any pinned host allocation, so that
    the staging buffers are node-local (first touch) and the ranks of an 8-GPU box do not
    fight over one socket's memory controller.  Returns what was done, for the JSON line.
    """
    info = {"bound": False}
    try:
        import torch
        p = torch.cuda.get_device_properties(dev_index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as fh:
            node = int(fh.read().strip())
        info["gpu_pci"] = bdf
        info["numa_node"] = node
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            spec = fh.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info["bound"] = True
            info["cpus"] = len(cpus)
    except Exception as e:          # no sysfs / no permission: run unbound and say so
        info["error"] = f"{type(e).__name__}: {e}"
    return info


# ------------------------------------------------------------------ GPU arm ---
def gpu_arm(args):
    import torch
    import torch.distributed as dist
    from setk_b200 import _lib, synth
    from setk_b200 import plan as P_
    from setk_b200.engine import BeamformPipeline, HostBatchStreamer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    # CPU baseline first (rank 0, N=1 only): before the GPU gets busy and before the rank is
    # bound to one NUMA node
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle.cpu_bench import usable_cores
        cores = usable_cores()
        r = cpu_steps(2, 1, 20.0, cores)
        cpu_base = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": r["kind"],
                    "sample": f"2 steps x {r['utts_per_step']} utterances of the same synthetic workload "
                              f"({r['workers']} single-threaded processes, distinct utterances), compute "
                              f"only, {r['seconds']:.1f} s",
                    "cpu": cpu_model()}

    numa = numa_bind(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries ONE JSON line: keep NCCL's "NCCL version ..." banner off it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B = args.batch
    pipe = BeamformPipeline(C, "mvdr", frame_len=FRAME_LEN, frame_hop=HOP, center=True,
                            window="hann", max_batch=B, max_samples=N, device=dev)
    # distinct synthetic utterances per rank (tiled to the batch when --unique < batch)
    uniq = min(B, args.unique)
    a_u, m_u = synth.make_batch(uniq, C, N, device=dev, first=rank * uniq)
    reps = (B + uniq - 1) // uniq
    audio = a_u.repeat(reps, 1, 1)[:B].contiguous()
    mask = m_u.repeat(reps, 1, 1)[:B].contiguous()
    del a_u, m_u
    torch.cuda.synchronize()

    def step():
        return pipe.run(audio, mask, pcm16_out=True)

    # ---- the result gather: every batch, PCM-16, asynchronous to the kernels ----
    # First choice: peer copies into a ring on rank 0 (copy engines over NVLink, no kernel on any
    # SM: setk_b200.distributed.PeerResultRing).  --gather nccl, or a box where the peer mapping
    # fails, uses dist.gather on NCCL's stream instead.
    RING = 3
    glists = ring = None
    n_out = pipe.plan.istft_length(T)
    if world > 1:
        if args.gather == "peer":
            from setk_b200.distributed import PeerResultRing
            ring = PeerResultRing.create((B, n_out), torch.int16, dev, slots=RING)
            if ring is None and rank == 0:
                print(f"[bench] peer ring unavailable ({PeerResultRing.last_error}); NCCL gather",
                      file=sys.stderr)
        if ring is None and rank == 0:
            # NCCL has no int16 type: the PCM travels as its uint8 byte view (same bytes, same count)
            glists = [[torch.empty((B, 2 * n_out), dtype=torch.uint8, device=dev) for _ in range(world)]
                      for _ in range(RING)]

    def as_bytes(w):
        return w.view(torch.uint8)

    # Order of the peer delivery (SETK_BENCH_PUSH, measurement knob):
    #   "after" : push batch i right behind its last kernel (default)
    #   "inside": launch the next batch's fused STFT+covariance first, then push batch i, and let the
    #             next apply+iSTFT wait for the copy.  Built to test whether the copy disturbs the launch
    #             of a persistent kernel: it does not -- both orders show the same two regimes at two
    #             GPUs (1.05-1.08 ms per step on most process starts, 2-4 ms on others).
    push_mode = os.environ.get("SETK_BENCH_PUSH", "after")

    def run_steps_inside(k):
        wave = status = None
        for i in range(k):
            Rs_, Rn_, mx_ = pipe.covariances(audio, mask)
            if wave is not None:
                ring.push(wave, i - 1)
            w_, status, _ = pipe.solve(Rs_, Rn_)
            ring.drain()                            # the apply kernel is launched behind the copy
            wave = pipe.plan.apply_istft(audio, w_, norm=mx_, pcm16=True)
        if wave is not None:
            ring.push(wave, k - 1)
        ring.drain()
        return wave, status

    def run_steps(k):
        if ring is not None and push_mode == "inside":
            return run_steps_inside(k)
        works, keep = [], collections.deque(maxlen=RING + 1)
        wave = status = None
        for i in range(k):
            wave, status = step()
            if ring is not None:
                ring.push(wave, i)
            elif world > 1:
                if i >= RING:
                    works[i - RING].wait()          # that ring slot's gather has drained
                keep.append(wave)
                works.append(dist.gather(as_bytes(wave), glists[i % RING] if rank == 0 else None, dst=0,
                                         async_op=True))
        if ring is not None:
            ring.drain()
        for w in works[-RING:]:
            w.wait()
        return wave, status

    wave, status = run_steps(max(args.warmup, 1))
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0, "solver reported failures on the synthetic batch"

    # ---- calibration of the delivery at N > 1 (12 steps per candidate, every rank decides alike) ----
    # Seen at two GPUs: 1.05 ms per step on most process starts, 1.3-4 ms on others, both ranks
    # alike.  Suspected mechanism (DESIGN section 6): delivering a batch is executed by copy kernels on
    # the SMs (the ring slot is a mapping in this rank's own address space, so the runtime treats the copy
    # as device-local); the fused kernels are persistent with static equal runs, and when a copy's
    # CTAs reach the SMs first at a batch boundary, CTAs of the persistent kernel cannot become
    # resident and its time doubles.  A high-priority compute stream makes the block scheduler place
    # the persistent CTAs first.  Nothing of this could be measured before the GPU budget ended, so
    # the run measures it: plain steps, steps + delivery on the default stream, steps + delivery on a
    # high-priority stream; the faster delivery is used, and if even that costs more than 15 % the
    # NCCL gather is used and the line says so.
    compute_ctx = None
    ring_probe = None
    if ring is not None:
        def probe(k, with_push):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            w = None
            for i in range(k):
                w, _ = step()
                if with_push:
                    ring.push(w, i)
            if with_push:
                ring.drain()
            e1.record()
            barrier()
            return max_over_ranks(e0.elapsed_time(e1)) / k

        hp_stream = None
        if os.environ.get("SETK_BENCH_PRIORITY", "1") == "1":
            try:
                hp_stream = torch.cuda.Stream(device=dev, priority=-1)
            except Exception as err:     # noqa: BLE001 -- no stream priorities here: default stream only
                if rank == 0:
                    print(f"[bench] no high-priority compute stream ({err!r})", file=sys.stderr)
        probe(4, True)
        t_plain, t_push = probe(12, False), probe(12, True)
        ring_probe = {"ms_per_step_without_push": round(t_plain, 4), "ms_per_step_with_push": round(t_push, 4)}
        use_hp = False
        if hp_stream is not None:
            try:
                torch.cuda.synchronize()
                with torch.cuda.stream(hp_stream):
                    probe(2, True)
                    t_hp = probe(12, True)
                    torch.cuda.synchronize()
                ring_probe["ms_per_step_with_push_high_priority_stream"] = round(t_hp, 4)
                use_hp = t_hp < t_push
                t_push = min(t_push, t_hp)
            except Exception as err:     # noqa: BLE001 -- the same code on every rank: all take this path
                hp_stream = None
                ring_probe["high_priority_stream_error"] = repr(err)
        if t_push > 1.15 * t_plain or os.environ.get("SETK_BENCH_PROBE_FORCE_REJECT") == "1":
            ring_probe["verdict"] = "rejected: NCCL gather used"
            if rank == 0:
                print(f"[bench] peer ring rejected by the calibration probe ({t_push:.3f} vs "
                      f"{t_plain:.3f} ms per step); NCCL gather", file=sys.stderr)
            ring = None
            use_hp = False
            if rank == 0:
                glists = [[torch.empty((B, 2 * n_out), dtype=torch.uint8, device=dev) for _ in range(world)]
                          for _ in range(RING)]
            run_steps(RING + 1)                  # warm the collective path
            torch.cuda.synchronize()
        else:
            ring_probe["verdict"] = "accepted, " + ("high-priority compute stream" if use_hp else "default stream")
        if use_hp:
            torch.cuda.synchronize()
            compute_ctx = torch.cuda.stream(hp_stream)
            compute_ctx.__enter__()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    def host_state():
        st = {"cuda_mallocs": torch.cuda.memory_stats(dev).get("num_device_alloc", 0), "cpu_s": sum(os.times()[:2])}
        try:
            with open("/sys/fs/cgroup/cpu.stat") as fh:
                kv = dict(l.split() for l in fh)
            st["throttled_ms"] = int(kv.get("throttled_usec", 0)) / 1e3
        except Exception:
            st["throttled_ms"] = None
        return st

    hs0 = host_state()
    ev0.record()
    h0 = time.perf_counter()
    wave, status = run_steps(args.steps)
    host_ms = (time.perf_counter() - h0) * 1e3      # host time to ENQUEUE the steps (no sync inside)
    ev1.record()
    hs1 = host_state()
    if compute_ctx is not None:
        torch.cuda.synchronize()
        compute_ctx.__exit__(None, None, None)
    host_diag = {"cuda_mallocs_in_region": hs1["cuda_mallocs"] - hs0["cuda_mallocs"],
                 "process_cpu_ms_in_region": round((hs1["cpu_s"] - hs0["cpu_s"]) * 1e3, 1),
                 "cgroup_throttled_ms_in_region": (None if hs0["throttled_ms"] is None else
                                                   round(hs1["throttled_ms"] - hs0["throttled_ms"], 1))}
    barrier()
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wave, status)
    ms_mine = ev0.elapsed_time(ev1)
    ms = max_over_ranks(ms_mine)
    value = world * B * args.steps / (ms / 1000.0)
    # per-rank device and host-enqueue times (a rank whose host time reaches its device time is
    # launch-bound: the GPU waits for Python)
    per_rank = [None] * world
    if world > 1:
        dist.all_gather_object(per_rank, (ms_mine / args.steps, host_ms / args.steps, host_diag))
    else:
        per_rank = [(ms_mine / args.steps, host_ms / args.steps, host_diag)]

    # ---- the gather alone (one batch from every rank into rank 0), for the record ----
    gather = None
    if world > 1:
        def gather_once(i):
            if ring is not None:
                ring.push(wave, i)
                ring.drain()
            else:
                dist.gather(as_bytes(wave), glists[0] if rank == 0 else None, dst=0)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        g0.record()
        for i in range(3):
            gather_once(args.steps - 1)           # the slot the run's last batch went to
        g1.record()
        barrier()
        g_ms = max_over_ranks(g0.elapsed_time(g1)) / 3
        # every rank's last batch must be on rank 0, bit for bit: compare checksums
        sums = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sums, wave.to(torch.int64).sum().reshape(1))
        if rank == 0:
            got = ring.slot(args.steps - 1) if ring is not None else \
                torch.stack([g.view(torch.int16) for g in glists[0]])
            assert torch.equal(got[0], wave), "gather: rank 0's own slot differs"
            for r in range(world):
                assert int(got[r].to(torch.int64).sum()) == int(sums[r]), f"gather: rank {r}'s batch differs"
        gbytes = (world - 1) * wave.numel() * 2
        how = (f"device-to-peer copies into a ring of 3 on rank 0 ({ring.mode} mapping of rank 0's buffer, "
               "copy engines over NVLink, side stream; no collective kernel)" if ring is not None else
               "dist.gather on NCCL's stream, ring of 3")
        gather = {"payload": "int16 PCM, every batch of every rank -> rank 0", "how": how,
                  "peer_ring_probe": ring_probe,
                  "bytes_into_rank0_per_step": gbytes, "gather_ms_alone": g_ms,
                  "gather_GBps": gbytes / (g_ms * 1e-3) / 1e9,
                  "needed_GBps_at_value": gbytes / ((ms / args.steps) * 1e-3) / 1e9}
    del glists, ring

    # ---- roofline of the dominant kernel: fused STFT+cov, timed alone ----
    def timed(fn, n):
        fn(); fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, r

    k_ms, (Rs, Rn, mx) = timed(lambda: pipe.covariances(audio, mask), max(10, min(args.steps, 50)))
    peak, peak_src = measured_peaks()
    alg = algorithmic_bytes_stft_cov() * B
    achieved = alg / (k_ms * 1e-3) / 1e9
    w_ms, (w, _, _) = timed(lambda: pipe.solve(Rs, Rn), 5)
    a_ms, _ = timed(lambda: pipe.plan.apply_istft(audio, w, norm=mx, pcm16=True), 5)
    stage = {"stft_cov_ms": k_ms, "weights_ms": w_ms, "apply_istft_pcm16_ms": a_ms}
    alg_apply = (4 * C * N + 8 * F * C + 2 * HOP * (T - 1)) * B
    stage["apply_istft_GBps"] = alg_apply / (a_ms * 1e-3) / 1e9
    del Rs, Rn, w

    # ---- e2e: host pinned buffers in and out, every step ----
    h_pcm = torch.empty(audio.shape, dtype=torch.int16, pin_memory=True)
    h_pcm.copy_(P_.float_to_pcm16(audio))
    h_mask = torch.empty(mask.shape, dtype=mask.dtype, pin_memory=True)
    h_mask.copy_(mask)
    n_out = wave.shape[1]
    h_outs = [torch.empty((B, n_out), dtype=torch.int16, pin_memory=True) for _ in range(2)]

    def make_pipe():
        return BeamformPipeline(C, "mvdr", frame_len=FRAME_LEN, frame_hop=HOP, center=True,
                                window="hann", max_batch=B, max_samples=N, device=dev)

    def time_e2e(streamer, h_a, h_o, steps, h_m=None):
        """H2D + hot path + D2H per step, two lanes so copies overlap compute."""
        h_m = h_mask if h_m is None else h_m
        for i in range(2):
            streamer.submit(h_a, h_m, h_o[i % 2])
        streamer.synchronize()
        barrier()
        x0 = torch.cuda.Event(enable_timing=True)
        x0.record()
        for i in range(steps):
            streamer.submit(h_a, h_m, h_o[i % 2], after=x0 if i < 2 else None)
        ends = streamer.record_all()
        streamer.synchronize()
        barrier()
        e_ms = max_over_ranks(max(x0.elapsed_time(e) for e in ends))
        for lane in streamer.slots:
            assert int(lane["status"].abs().sum()) == 0
        return world * B * steps / (e_ms / 1000.0)

    e2e_steps = max(4, min(args.steps, 8))
    del pipe
    torch.cuda.empty_cache()
    # headline: what the files hold -- PCM-16 wav samples and the masks as a Kaldi archive stores them
    # by default (CompressedMatrix "CM", 1 byte per TF cell; kaldi_io.py:248-281 expands them on the
    # host in the reference, setk_cm_masks on the device here, bit-identical)
    from setk_b200.libs.data_handler import compress_kaldi_cm
    slot = HostBatchStreamer.cm_slot_bytes(T, F)
    h_cm = torch.zeros((B, slot), dtype=torch.uint8, pin_memory=True)
    m_host = mask[:uniq].cpu().numpy()
    for u in range(uniq):
        raw = torch.frombuffer(bytearray(compress_kaldi_cm(m_host[u])), dtype=torch.uint8)
        h_cm[u, :raw.numel()] = raw
    for b in range(uniq, B):
        h_cm[b] = h_cm[b % uniq]
    del m_host
    st = HostBatchStreamer(make_pipe, B, C, N, slots=2, pcm16=True, pcm16_out=True, device=dev, cm_masks=True)
    e2e_val = time_e2e(st, h_pcm, h_outs, e2e_steps, h_cm)
    for lane in st.slots:
        assert int(lane["cm_status"].abs().sum()) == 0
    del st
    torch.cuda.empty_cache()
    # variant: the same with float32 masks on the host (round 2's first e2e definition)
    st = HostBatchStreamer(make_pipe, B, C, N, slots=2, pcm16=True, pcm16_out=True, device=dev)
    e2e_f32mask = time_e2e(st, h_pcm, h_outs, e2e_steps)
    del st
    torch.cuda.empty_cache()
    # variant: float32 samples on the host in both directions (round 1's e2e definition)
    h_f32 = torch.empty(audio.shape, dtype=torch.float32, pin_memory=True)
    h_f32.copy_(audio)
    h_outs_f = [torch.empty((B, n_out), dtype=torch.float32, pin_memory=True) for _ in range(2)]
    st = HostBatchStreamer(make_pipe, B, C, N, slots=2, pcm16=False, pcm16_out=False, device=dev)
    e2e_f32 = time_e2e(st, h_f32, h_outs_f, e2e_steps)
    del st, h_f32, h_outs_f
    h2d = h_pcm.numel() * 2 + h_cm.numel()
    h2d_f32mask = h_pcm.numel() * 2 + h_mask.numel() * 4
    d2h = B * n_out * 2
    del audio, mask, h_pcm, h_mask, h_outs, h_cm
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations at this GPU count ----
    configs = None if args.no_configs else other_configs(dev, world, rank, barrier, max_over_ranks, peak)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (STFT/cov/apply), f64 (per-bin weight solve)", "data": "synthetic",
            "config": config_dict(world, B),
            "run": {"unique_utterances_per_gpu": uniq, "numa": numa,
                    "compute_stream": "high priority" if compute_ctx is not None else "default",
                    "per_rank_ms_per_step": [dict({"device": round(a, 4), "host_enqueue": round(b, 4)}, **hd)
                                             for a, b, hd in per_rank]},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": measured_traffic(B), "peak_source": peak_src,
                         "kernel": "setk_stft_cov (stft_cov_ws_kernel<4> + finalize)",
                         "algorithmic_bytes_per_launch": alg, "kernel_ms": k_ms},
            "cpu_baseline": cpu_base,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps,
                    "how": "pinned host PCM-16 audio (what wav files hold) + Kaldi CompressedMatrix masks "
                           "(what a mask archive holds, 1 byte per TF cell) -> H2D -> int16/32768 and "
                           "kaldi_io uncompress on device -> BeamformPipeline.run -> floor(y*32768) on "
                           "device -> D2H int16, every step; 2 lanes (streams) so copies overlap kernels",
                    "h2d_GBps": e2e_val / world * h2d / B / 1e9,
                    "bound": "host->device link (PCIe)",
                    "f32_mask_variant": {"value": e2e_f32mask, "unit": UNIT, "h2d_bytes_per_step": h2d_f32mask,
                                         "d2h_bytes_per_step": d2h,
                                         "h2d_GBps": e2e_f32mask / world * h2d_f32mask / B / 1e9},
                    "f32_host_variant": {"value": e2e_f32, "unit": UNIT,
                                         "h2d_bytes_per_step": B * (C * N + T * F) * 4,
                                         "d2h_bytes_per_step": B * n_out * 4}},
            "gather": gather,
            "gpu_launches": int(launches),
            "stages": stage,
            "configs": configs,
            "clocks": sampler.summary() if sampler else None,
            "library": _lib.library_path(),
        }
        if sampler:
            sampler.stop()
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def other_configs(dev, world, rank, barrier, max_over_ranks, peak):
    """
    BASELINE.json configs[2..4] (SURVEY.md section 8d shapes), device-resident, a few steps each:
      cfg3  8-ch GEV, 1024-pt STFT, batch 256 per GPU (processed as 4 x 64)
      cfg4  WPE(taps 10, delay 3, 3 iterations) + MVDR, 6 ch, batch 128 in TOTAL (strong scaling)
      cfg5  MVDR 8 ch and 16 ch, 512-pt (4 ch is the headline line)
    value = utterances of all ranks / max-over-ranks device time.
    """
    import torch
    from setk_b200 import synth
    from setk_b200 import plan as P_
    from setk_b200.engine import BeamformPipeline

    out = {}

    def time_steps(fn, n):
        fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / n

    def beamform_cfg(name, ch, frame_len, kind, b, steps=5):
        pipe = BeamformPipeline(ch, kind, frame_len=frame_len, frame_hop=HOP, max_batch=b,
                                max_samples=N, device=dev)
        nf = pipe.plan.n_fft
        a, m = synth.make_batch(min(b, 8), ch, N, device=dev, frame_len=frame_len, n_fft=nf,
                                first=1000 + 8 * rank)
        reps = (b + a.shape[0] - 1) // a.shape[0]
        audio = a.repeat(reps, 1, 1)[:b].contiguous()
        mask = m.repeat(reps, 1, 1)[:b].contiguous()
        del a, m
        ms = time_steps(lambda: pipe.run(audio, mask, pcm16_out=True), steps)
        k_ms = time_steps(lambda: pipe.covariances(audio, mask), steps)
        Rs, Rn, mx = pipe.covariances(audio, mask)
        w_ms = time_steps(lambda: pipe.solve(Rs, Rn), steps)
        w = pipe.solve(Rs, Rn)[0]
        a_ms = time_steps(lambda: pipe.plan.apply_istft(audio, w, norm=mx, pcm16=True), steps)
        alg = algorithmic_bytes_stft_cov(ch, N, nf, HOP) * b
        ach = alg / (k_ms * 1e-3) / 1e9
        out[name] = {"channels": ch, "n_fft": nf, "beamformer": kind, "batch_per_gpu": b,
                     "value": world * b / ms * 1e3, "unit": UNIT, "ms_per_batch": ms,
                     "stages": {"stft_cov_ms": k_ms, "weights_ms": w_ms, "apply_istft_pcm16_ms": a_ms},
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                                  "frac": ach / peak, "algorithmic_bytes_per_launch": alg,
                                  "kernel": "setk_stft_cov"}}
        del pipe, audio, mask, Rs, Rn, w
        torch.cuda.empty_cache()

    beamform_cfg("cfg3_8ch_gev_1024", 8, 1024, "gevd", 64)
    beamform_cfg("cfg5_8ch_mvdr_512", 8, 512, "mvdr", 64)
    beamform_cfg("cfg5_16ch_mvdr_512", 16, 512, "mvdr", 32)

    # cfg4: WPE -> MVDR on the dereverberated STFT, 128 utterances in total over the ranks
    b = max(1, 128 // world)
    ch = 6
    pipe = BeamformPipeline(ch, "mvdr", frame_len=512, frame_hop=HOP, max_batch=b, max_samples=N,
                            device=dev)
    a, m = synth.make_batch(min(b, 4), ch, N, device=dev, first=2000 + 4 * rank)
    reps = (b + a.shape[0] - 1) // a.shape[0]
    audio = a.repeat(reps, 1, 1)[:b].contiguous()
    mask = m.repeat(reps, 1, 1)[:b].contiguous()
    del a, m
    from setk_b200 import _lib

    def wpe_mvdr():
        S = pipe.plan.stft(audio)                                  # (B,C,F,T)
        D, st = P_.wpe_from_stft(S, 10, 3, 1, 3)
        Rs = P_.covariance(D, mask)
        Rn = P_.covariance(D, 1.0 - mask)
        w = P_.weights(_lib.BF_MVDR, Rs, Rn=Rn, out_dtype=torch.complex64)[0]
        enh = P_.apply_weights(D, w)
        return pipe.plan.istft(enh)

    ms = time_steps(wpe_mvdr, 2)
    S = pipe.plan.stft(audio)
    wpe_ms = time_steps(lambda: P_.wpe_from_stft(S, 10, 3, 1, 3), 2)
    out["cfg4_wpe_mvdr_6ch"] = {"channels": ch, "n_fft": 512, "beamformer": "wpe(10,3,1,3)+mvdr",
                                "batch_total": b * world, "batch_per_gpu": b, "scaling": "strong",
                                "value": world * b / ms * 1e3, "unit": UNIT, "ms_per_batch": ms,
                                "stages": {"wpe_ms": wpe_ms}}
    del pipe, audio, mask, S
    torch.cuda.empty_cache()
    return out


DUMP_ROWS = 64     # utterances of the PCM-16 output written by --dump-outputs: 64 x 160000 x 4 B = 41 MB


def dump_outputs(out_dir, wave, status):
    """
    What the last timed step returned to its caller (BeamformPipeline.run with pcm16_out=True), as
    float32 .npy files in `out_dir`:
      pcm16.npy   the enhanced PCM-16 samples of DUMP_ROWS utterances of the batch, picked by a fixed
                  seed (all of them when the batch is smaller), in ascending order; (rows, n_out)
      status.npy  the solver status of every utterance of the batch; (B,)
    The int16 and int32 values are exact in float32.
    """
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    B = wave.shape[0]
    rows = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_ROWS), replace=False))
    pcm = wave.index_select(0, torch.from_numpy(rows).to(wave.device)).float().cpu().numpy()
    np.save(os.path.join(out_dir, "pcm16.npy"), pcm)
    np.save(os.path.join(out_dir, "status.npy"), status.float().cpu().numpy())


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--unique", type=int, default=256,
                    help="distinct synthetic utterances per GPU (tiled to the batch)")
    ap.add_argument("--cpu-budget", type=float, default=150.0,
                    help="seconds of CPU work the --impl reference run may take")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--gather", choices=["peer", "nccl"], default="peer",
                    help="N > 1: how every batch's result reaches rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    # stdout carries ONE JSON line: everything else any library writes to file descriptor 1 (NCCL's
    # version banner comes from C) goes to stderr; emit() writes the line to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
