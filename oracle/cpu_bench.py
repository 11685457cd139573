"""
oracle/cpu_bench.py -- time the reference's CPU path on the host cores, for bench.py's
`cpu_baseline` and `--impl reference` legs.

TEST / MEASUREMENT INFRASTRUCTURE (see oracle/__init__.py).  Mirrors how the reference
scales: `run.pl JOB=1:nj` forks one single-threaded Python per wav.scp shard
(scripts/run_adapt_beamformer.sh:66-92); here `workers` processes each run the
per-utterance loop body of apply_adaptive_beamformer.py:130-177

    forward_stft x C -> MvdrBeamformer.run -> inverse_stft(norm=max|x|) -> PCM-16

on the reference's default dtype path (float32 mask -> complex64 STFT), no file IO in the
timed region, every worker cycling through its own distinct synthetic utterances.

Which code is timed (BASELINE.md section 3): the reference's OWN modules when its tree can be
found -- $SETK_REFERENCE, then <repo>/baseline/_ref/scripts/sptk -- imported under
oracle/ref_shim.py (`kind` = "reference"); otherwise this directory's numpy restatement of the
same files (`kind` = "port").
"""
import multiprocessing as mp
import os
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_root():
    """First existing scripts/sptk directory of the lookup order, or None."""
    cands = []
    env = os.environ.get("SETK_REFERENCE")
    if env:
        cands += [env, os.path.join(env, "scripts", "sptk")]
    cands += [os.path.join(ROOT, "baseline", "_ref", "scripts", "sptk")]
    for c in cands:
        if os.path.isdir(os.path.join(c, "libs")):
            return c
    return None


def _synth(C, N, seed):
    rng = np.random.default_rng(seed)
    env = 0.55 + 0.45 * np.cos(2 * np.pi * 4.0 * np.arange(N) / 16000.0 + rng.uniform(0, 6.28))
    s = rng.standard_normal(N) * env
    taps = np.exp(-np.arange(64) / 8.0)

    def fir(x):
        h = rng.standard_normal(64) * taps
        h[0] = np.sign(h[0]) * (np.abs(h).max() + 0.5)
        return np.convolve(x, h)[:N]

    tgt = np.stack([fir(s) for _ in range(C)])
    noise = np.zeros((C, N))
    for _ in range(C + 2):
        v = rng.standard_normal(N)
        noise += np.stack([fir(v) for _ in range(C)])
    noise += 0.1 * np.std(tgt) * rng.standard_normal((C, N))
    noise *= np.sqrt(np.mean(tgt[0]**2) / (np.mean(noise[0]**2) * 10**0.5))
    mix = tgt + noise
    sc = 0.5 / np.max(np.abs(mix))
    return (mix * sc).astype(np.float32), (tgt[0] * sc).astype(np.float32), \
        (noise[0] * sc).astype(np.float32)


def _make_runner(ref_root):
    """Returns (run(mix, mask) -> int16 samples, kind)."""
    from oracle import stft_oracle as so
    kw = dict(frame_len=512, frame_hop=256, center=True, window="hann", transpose=False)
    if ref_root is not None:
        from oracle import ref_shim
        ref_shim.REFERENCE_SPTK = ref_root
        ref = ref_shim.load_reference()
        bf = ref.beamformer.MvdrBeamformer(257)

        def run(mix, mask):
            stft = np.stack([ref.utils.forward_stft(mix[c], round_power_of_two=True, **kw)
                             for c in range(mix.shape[0])])
            enh = bf.run(np.minimum(mask, 1), stft, mask_n=None, ban=False)
            y = ref.utils.inverse_stft(enh, norm=float(np.max(np.abs(mix))), **kw)
            return so.pcm16_from_float(y)
        return run, "reference"
    from oracle import beamformer_oracle as bo

    def run(mix, mask):
        y, _, _ = bo.enhance_utterance(mix, mask, kind="mvdr", stft_dtype=np.complex64)
        return so.pcm16_from_float(y)
    return run, "port"


def _worker(wid, C, N, share, steps, warmup, seed, distinct, ref_root, barrier, out):
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    from oracle import stft_oracle as so
    run, kind = _make_runner(ref_root)
    kw = dict(frame_len=512, frame_hop=256, center=True, window="hann", transpose=False)
    utts = []
    for u in range(distinct):
        mix, tgt0, noise0 = _synth(C, N, seed + 1000 * wid + u)
        S = so.forward_stft(tgt0, round_power_of_two=True, **kw)
        V = so.forward_stft(noise0, round_power_of_two=True, **kw)
        mask = (np.abs(S) / np.sqrt(np.abs(S)**2 + np.abs(V)**2 + so.EPSILON)).T.astype(np.float32)
        utts.append((mix, mask))
    k = 0
    for _ in range(max(1, warmup) * share):
        run(*utts[k % distinct]); k += 1
    barrier.wait()
    t0 = time.perf_counter()
    for _ in range(steps * share):
        run(*utts[k % distinct]); k += 1
    out.put((wid, time.perf_counter() - t0, kind))


def usable_cores():
    """Cores this process may actually use: affinity mask and cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def run_steps(C, N, steps, warmup, utts_per_step, workers, seed=20240923, distinct=4):
    """
    `steps` timed steps of `utts_per_step` utterances spread over `workers` concurrent
    single-threaded processes (each runs steps x its share back to back after `warmup`
    untimed shares).  Returns dict(value utts/s, seconds, ms_per_step, utts_per_step, kind).
    """
    workers = max(1, min(workers, utts_per_step))
    share = max(1, utts_per_step // workers)
    ups = share * workers
    ref_root = reference_root()
    ctx = mp.get_context("spawn")
    barrier = ctx.Barrier(workers)
    out = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(w, C, N, share, steps, warmup, seed, distinct, ref_root,
                                               barrier, out)) for w in range(workers)]
    for p in procs:
        p.start()
    res = []
    import queue
    while len(res) < len(procs):
        try:
            res.append(out.get(timeout=5.0))
        except queue.Empty:
            dead = [p for p in procs if p.exitcode not in (None, 0)]
            if dead:                       # a worker died: do not wait for the others forever
                for p in procs:
                    p.terminate()
                raise RuntimeError(f"cpu_bench worker exited with code {dead[0].exitcode}")
    for p in procs:
        p.join()
    seconds = max(r[1] for r in res)
    return {"value": steps * ups / seconds, "seconds": seconds, "ms_per_step": 1000.0 * seconds / steps,
            "utts_per_step": ups, "workers": workers, "kind": res[0][2],
            "reference_root": ref_root}


def throughput(C, N, n_utts_per_worker, workers, seed=20240923):
    """utterances / second over `workers` processes, `n_utts_per_worker` timed utterances each."""
    r = run_steps(C, N, n_utts_per_worker, 1, workers, workers, seed)
    return r["value"]
