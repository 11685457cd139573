"""
CPU tier: the Python host layer (the mirror of the reference's sptk.libs API,
the batched engine and the CLI) running on the CPU execution model of the
kernels, against the oracle.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import beamformer_oracle as bo
from oracle import stft_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def libs(emu):
    from setk_b200.libs import beamformer as BF
    from setk_b200.libs import utils as U
    U.set_default_device("cpu")
    yield U, BF
    U.set_default_device(None)


def test_forward_inverse_stft_api(libs):
    U, _ = libs
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(3000) * 0.1).astype(np.float32)
    for kw in (dict(frame_len=512, frame_hop=256, center=True, transpose=False),
               dict(frame_len=400, frame_hop=160, center=True, transpose=True),
               dict(frame_len=256, frame_hop=128, center=False, window="hamming", transpose=True)):
        S = U.forward_stft(x, **kw)
        So = so.forward_stft(x, **kw)
        assert S.shape == So.shape and S.dtype == np.complex64
        assert bo.rel_inf(S, So) <= 2e-5
        y = U.inverse_stft(S, norm=0.3, **kw)
        yo = so.inverse_stft(So, norm=0.3, **kw)
        assert y.shape == yo.shape
        assert bo.rel_inf(y, yo) <= 2e-5
    # defaults are the reference's (utils.py:96-105): 1024 / 256 / center False / transpose True
    S = U.forward_stft(x)
    assert S.shape == (1 + (3000 - 1024) // 256, 513)
    mag = U.forward_stft(x, 512, 256, apply_log=True, transpose=False)
    assert mag.dtype == np.float32 and np.all(np.isfinite(mag))
    with pytest.raises(RuntimeError):
        U.forward_stft(np.zeros((2, 3000), dtype=np.float32))
    # torch in -> torch out
    St = U.forward_stft(torch.from_numpy(x), 512, 256, center=True)
    assert isinstance(St, torch.Tensor) and St.dtype == torch.complex64
    assert U.nextpow2(400) == 512


def test_beamformer_api(libs):
    _, BF = libs
    rng = np.random.default_rng(1)
    C, F, T = 4, 257, 10
    obs = (rng.standard_normal((C, F, T)) + 1j * rng.standard_normal((C, F, T))).astype(np.complex64)
    mask = rng.uniform(0, 1, (T, F)).astype(np.float32)
    obs64, mask64 = obs.astype(np.complex128), mask.astype(np.float64)
    cases = [(BF.MvdrBeamformer(F), "mvdr", {}), (BF.GevdBeamformer(F), "gevd", {}),
             (BF.PmwfBeamformer(F, beta=1, ref_channel=0), "pmwf", dict(beta=1, ref_channel=0)),
             (BF.PmwfBeamformer(F, rank1_appro="eig"), "pmwf", dict(rank1_appro="eig")),
             (BF.MpdrBeamformer(F), "mpdr", {}), (BF.MpdrBeamformer(F, whiten=True), "mpdr-whiten", {})]
    for bf, kind, kw in cases:
        for ban in (False, True):
            enh = bf.run(mask, obs, ban=ban)
            ref = bo.run_supervised(kind, mask64, obs64, ban=ban, **kw)
            assert enh.shape == (F, T) and enh.dtype == np.complex64
            assert bo.rel_inf(bo.align_phase(enh, ref)[0], ref) <= 2e-5, (kind, ban)
    Rs, Rn = bo.compute_covar(obs64, mask64), bo.compute_covar(obs64, 1 - mask64)
    assert bo.rel_inf(BF.compute_covar(obs, mask), Rs) <= 2e-5
    d = BF.solve_pevd(Rs)
    assert d.dtype == np.complex128
    assert bo.rel_inf(bo.align_phase(d, bo.solve_pevd(Rs))[0], bo.solve_pevd(Rs)) <= 1e-9
    assert bo.rel_inf(BF.rank1_constraint(Rs, Rn), bo.rank1_constraint(Rs, Rn)) <= 1e-9
    w = bo.mvdr_weight(Rs, Rn)
    assert bo.rel_inf(BF.do_ban(w, Rn), bo.do_ban(w, Rn)) <= 1e-9
    # error behaviour of the reference
    with pytest.raises(ValueError):
        BF.Beamformer().beamform(w[:, :3], obs)
    with pytest.raises(ValueError):
        BF.MvdrBeamformer(F).compute_covar_mat(mask[:, :100], obs)
    with pytest.raises(RuntimeError):
        BF.PmwfBeamformer(F, ref_channel=7).weight(Rs, Rn)
    with pytest.raises(np.linalg.LinAlgError):
        BF.MvdrBeamformer(F).weight(Rs, np.zeros_like(Rn))
    with pytest.raises(NotImplementedError):
        BF.SupervisedBeamformer(F).weight(Rs, Rn)


def test_online_beamformer(libs):
    _, BF = libs
    rng = np.random.default_rng(2)
    C, F, T = 3, 129, 64
    obs = (rng.standard_normal((C, F, T)) + 1j * rng.standard_normal((C, F, T))).astype(np.complex64)
    mask = rng.uniform(0, 1, (T, F)).astype(np.float32)
    bf = BF.OnlineMvdrBeamformer(F, C, alpha=0.8)
    out = [bf.run(mask[c:c + 32], np.ascontiguousarray(obs[:, :, c:c + 32])) for c in (0, 32)]
    assert out[0].shape == (F, 32)
    # first chunk equals the offline beamformer on that chunk
    ref = bo.run_supervised("mvdr", mask[:32].astype(np.float64),
                            obs[:, :, :32].astype(np.complex128))
    assert bo.rel_inf(bo.align_phase(out[0], ref)[0], ref) <= 2e-5
    # second chunk: the reference's recursion R <- alpha R + R_chunk (phi stays 1,
    # beamformer.py:314-316: `reset` is never cleared there)
    m64, o128 = mask.astype(np.float64), obs.astype(np.complex128)
    Rs = [bo.compute_covar(o128[:, :, c:c + 32], m64[c:c + 32]) for c in (0, 32)]
    Rn = [bo.compute_covar(o128[:, :, c:c + 32], 1 - m64[c:c + 32]) for c in (0, 32)]
    w = bo.mvdr_weight(0.8 * Rs[0] + Rs[1], 0.8 * Rn[0] + Rn[1])
    ref2 = bo.beamform(w, o128[:, :, 32:])
    assert bo.rel_inf(bo.align_phase(out[1], ref2)[0], ref2) <= 5e-5


def test_pipeline_status_maps_to_linalgerror(emu):
    from setk_b200.engine import BeamformPipeline
    pipe = BeamformPipeline(4, "mvdr", max_batch=2, max_samples=2000, device=emu)
    x = torch.zeros(2, 4, 2000)                       # silence: singular covariances
    m = torch.full((2, pipe.plan.num_frames(2000), 257), 0.5)
    wave, status = pipe.run(x, m)
    assert int(status.abs().sum()) != 0
    with pytest.raises(np.linalg.LinAlgError):
        BeamformPipeline.raise_for_status(status, ["a", "b"])


def test_plan_is_destroyed_by_the_library_that_made_it(emu, monkeypatch):
    """A plan outliving a use_library() switch (the plan cache of setk_b200.libs.utils keeps plans until
    the interpreter exits) is destroyed by its own library, not by the one bound now."""
    from setk_b200 import _lib
    from setk_b200.plan import StftPlan
    pl = StftPlan(2, max_batch=1, max_samples=4000, device=emu)
    other = []

    class OtherLibrary:
        def setk_plan_destroy(self, h):
            other.append(h)
            return 0

    monkeypatch.setattr(_lib, "_cdll", OtherLibrary())
    pl.close()
    assert other == [] and pl._h is None


def _write_wav(path, x):
    import scipy.io.wavfile as wavfile
    wavfile.write(path, 16000, so.pcm16_from_float(x.T))


def test_cli_end_to_end(tmp_path, emu_library_path):
    """scripts/sptk/apply_adaptive_beamformer.py with the reference's flags, vs the oracle."""
    from setk_b200 import synth
    x, m = synth.make_batch(1, 4, 4000, device="cpu")
    x, m = x[0].numpy(), m[0].numpy()
    x = so.float_from_pcm16(so.pcm16_from_float(x))            # what the wav file will hold
    _write_wav(str(tmp_path / "utt1.wav"), x)
    np.save(tmp_path / "utt1.npy", m)
    (tmp_path / "wav.scp").write_text(f"utt1 {tmp_path / 'utt1.wav'}\n")
    (tmp_path / "mask.scp").write_text(f"utt1 {tmp_path / 'utt1.npy'}\n")
    env = dict(os.environ, SETK_B200_TEST_LIBRARY=emu_library_path, PYTHONPATH=ROOT)
    runner = (
        "import os, sys, runpy; sys.argv = sys.argv[1:];"
        "from setk_b200 import _lib; _lib.use_library(os.environ['SETK_B200_TEST_LIBRARY']);"
        "from setk_b200.libs import utils; utils.set_default_device('cpu');"
        "runpy.run_path(sys.argv[0], run_name='__main__')")
    import scipy.io.wavfile as wavfile
    # PMWF is phase invariant, so the waveform itself is comparable with the oracle;
    # MVDR's per-bin sign is LAPACK-defined in the reference (checked elsewhere after alignment)
    cases = (("pmwf-0", [], dict(beta=0)),
             ("pmwf-1", ["--ban", "true", "--pmwf-ref", "1"], dict(beta=1, ref_channel=1, ban=True)),
             ("mvdr", ["--post-masking", "true"], None))
    for bf, extra, okw in cases:
        dst = tmp_path / bf
        cmd = [sys.executable, "-c", runner,
               os.path.join(ROOT, "scripts", "sptk", "apply_adaptive_beamformer.py"),
               "--frame-len", "512", "--frame-hop", "256", "--mask-format", "numpy",
               "--batch-size", "0",       # the batched feeder needs CUDA streams: tests/test_gpu_cli.py
               "--beamformer", bf, *extra, str(tmp_path / "wav.scp"), str(tmp_path / "mask.scp"),
               str(dst)]
        subprocess.run(cmd, check=True, env=env, capture_output=True)
        sr, out = wavfile.read(str(dst / "utt1.wav"))
        assert sr == 16000 and out.dtype == np.int16
        assert out.shape == (256 * (so.num_frames(4000, 512, 256, True) - 1),)
        if okw is None:
            assert np.abs(out).max() > 1000
            continue
        y, _, _ = bo.enhance_utterance(x, m, kind="pmwf", **okw)
        ref = so.pcm16_from_float(y)
        d = np.abs(out.astype(np.int64) - ref.astype(np.int64))
        assert d.max() <= 1 and np.mean(d > 0) <= 0.05


def test_batch_planner_sorts_and_cuts():
    """setk_b200/batch_cli.plan_batches: same channel count / dtype per batch, lengths sorted,
    at most batch_size utterances (pure host logic of the batched CLI)."""
    from setk_b200.batch_cli import plan_batches
    rng = np.random.default_rng(3)
    window = []
    for i in range(37):
        C = 4 if i % 5 else 2
        n = int(rng.integers(1000, 9000))
        dt = np.int16 if i % 7 else np.float32
        window.append((f"k{i}", np.zeros((C, n), dtype=dt), np.zeros((3, 5), np.float32), None))
    batches = plan_batches(list(window), 8)
    assert sum(len(b) for b in batches) == 37
    for b in batches:
        assert len(b) <= 8
        assert len({(it[1].shape[0], it[1].dtype) for it in b}) == 1
        lens = [it[1].shape[1] for it in b]
        assert lens == sorted(lens)


def test_cgmm_trainer_mirror_and_cli(tmp_path, emu, emu_library_path):
    """libs.cluster.CgmmTrainer (reference signature) and scripts/sptk/estimate_cgmm_masks.py."""
    from oracle import cgmm_oracle as co
    from setk_b200.libs import utils
    from setk_b200.libs.cluster import CgmmTrainer
    import parity_cases as pc
    utils.set_default_device("cpu")
    rng = np.random.default_rng(11)
    x = pc.structured_audio(rng, 1, 3, 3000)[0]
    x = so.float_from_pcm16(so.pcm16_from_float(x))
    # (a) the trainer on a caller-provided STFT (n_fft = 256: plan-free setk_cgmm_stft)
    obs = so.multichannel_stft(x, frame_len=256, frame_hop=128, center=True, window="hann",
                               round_power_of_two=True, transpose=False, out_dtype=np.complex64)
    gamma = CgmmTrainer(obs, 2).train(3)
    assert isinstance(gamma, np.ndarray) and gamma.shape == (2,) + obs.shape[1:]
    ref = co.cgmm_masks(obs, 2, 3, return_all=True)[1][-1]
    assert np.max(np.abs(gamma - ref)) <= 1e-6
    tr = CgmmTrainer(torch.from_numpy(obs), 2, gamma=ref[0].astype(np.float32), update_alpha=True)
    tr.train(1)
    g2 = tr.train(1)                                     # continues: 2 iterations in all
    ref2 = co.cgmm_masks(obs, 2, 2, init_gamma=ref[0].astype(np.float32).astype(np.float64),
                         update_alpha=True, return_all=True)[1][-1]
    assert torch.is_tensor(g2) and np.max(np.abs(g2.numpy() - ref2)) <= 1e-6
    with pytest.raises(RuntimeError):
        CgmmTrainer(obs, 3)
    # (b) the CLI, documented flags, from a wav file
    _write_wav(str(tmp_path / "utt1.wav"), x)
    (tmp_path / "wav.scp").write_text(f"utt1 {tmp_path / 'utt1.wav'}\n")
    env = dict(os.environ, SETK_B200_TEST_LIBRARY=emu_library_path, PYTHONPATH=ROOT)
    runner = (
        "import os, sys, runpy; sys.argv = sys.argv[1:];"
        "from setk_b200 import _lib; _lib.use_library(os.environ['SETK_B200_TEST_LIBRARY']);"
        "from setk_b200.libs import utils; utils.set_default_device('cpu');"
        "runpy.run_path(sys.argv[0], run_name='__main__')")
    cmd = [sys.executable, "-c", runner, os.path.join(ROOT, "scripts", "sptk", "estimate_cgmm_masks.py"),
           "--frame-len", "512", "--frame-hop", "256", "--num-iters", "3", "--center", "true",
           str(tmp_path / "wav.scp"), str(tmp_path / "masks")]
    subprocess.run(cmd, check=True, env=env, capture_output=True)
    mask = np.load(tmp_path / "masks" / "utt1.npy")
    T = so.num_frames(3000, 512, 256, True)
    assert mask.shape == (T, 257) and mask.dtype == np.float32
    obs512 = so.multichannel_stft(x, frame_len=512, frame_hop=256, center=True, window="hann",
                                  round_power_of_two=True, transpose=False, out_dtype=np.complex64)
    d = np.abs(mask - co.cgmm_masks(obs512, 2, 3))
    assert d.mean() <= 1e-4                              # float32 tile STFT vs float64 oracle STFT


def test_wpe_mirror_and_cli(tmp_path, emu, emu_library_path):
    """libs.wpe.wpe (reference signature) and scripts/sptk/apply_wpe.py."""
    from oracle import wpe_oracle as wo
    from setk_b200.libs import utils
    from setk_b200.libs.wpe import wpe
    import parity_cases as pc
    utils.set_default_device("cpu")
    rng = np.random.default_rng(13)
    x = pc.structured_audio(rng, 1, 2, 2600)[0]
    x = so.float_from_pcm16(so.pcm16_from_float(x))
    kw = dict(frame_len=256, frame_hop=64, center=True, window="hann", round_power_of_two=True,
              transpose=False)
    obs = np.einsum("nft->fnt", so.multichannel_stft(x, out_dtype=np.complex64, **kw))      # F x N x T
    ref = wo.wpe(obs, taps=4, delay=2, context=1, num_iters=2)
    out = wpe(obs, taps=4, delay=2, context=1, num_iters=2)
    assert isinstance(out, np.ndarray) and out.shape == obs.shape
    assert bo.rel_inf(out, ref) <= 2e-6
    out_t = wpe(torch.from_numpy(obs)[None], taps=4, delay=2, context=1, num_iters=2)       # batched tensor
    assert torch.is_tensor(out_t) and bo.rel_inf(out_t[0].numpy(), ref) <= 2e-6
    with pytest.raises(np.linalg.LinAlgError):
        wpe(np.zeros((9, 2, 30), dtype=np.complex64), taps=3, delay=1)
    # the CLI: all channels of the dereverberated signal as one PCM-16 file
    _write_wav(str(tmp_path / "utt1.wav"), x)
    (tmp_path / "wav.scp").write_text(f"utt1 {tmp_path / 'utt1.wav'}\n")
    env = dict(os.environ, SETK_B200_TEST_LIBRARY=emu_library_path, PYTHONPATH=ROOT)
    runner = (
        "import os, sys, runpy; sys.argv = sys.argv[1:];"
        "from setk_b200 import _lib; _lib.use_library(os.environ['SETK_B200_TEST_LIBRARY']);"
        "from setk_b200.libs import utils; utils.set_default_device('cpu');"
        "runpy.run_path(sys.argv[0], run_name='__main__')")
    cmd = [sys.executable, "-c", runner, os.path.join(ROOT, "scripts", "sptk", "apply_wpe.py"),
           "--frame-len", "256", "--frame-hop", "64", "--center", "true", "--taps", "4", "--delay", "2",
           "--num-iters", "2", str(tmp_path / "wav.scp"), str(tmp_path / "out")]
    subprocess.run(cmd, check=True, env=env, capture_output=True)
    import scipy.io.wavfile as wavfile
    sr, y = wavfile.read(str(tmp_path / "out" / "utt1.wav"))
    assert sr == 16000 and y.dtype == np.int16 and y.shape[1] == 2
    yo = np.stack([so.inverse_stft(ref[:, n], frame_len=256, frame_hop=64, center=True, window="hann",
                                   transpose=False) for n in range(2)])
    d = np.abs(y.T.astype(np.int64) - so.pcm16_from_float(yo).astype(np.int64))
    assert d.max() <= 1


def test_archive_writer_and_spatial_cli(tmp_path, emu, emu_library_path):
    """
    ArchiveWriter (Kaldi ark + scp, data_handler.py:564-587), the libs.spatial mirror (reference
    names / axes) and scripts/sptk/compute_ipd_and_linear_srp.py on the CPU execution model.
    """
    import struct
    from oracle import spatial_oracle as sp
    from setk_b200.libs import utils
    from setk_b200.libs import spatial as gs
    from setk_b200.libs.data_handler import ArchiveWriter, ScriptReader
    import parity_cases as pc
    utils.set_default_device("cpu")
    # ---- writer: the bytes the reference's kaldi_io writers produce, read back by ScriptReader ----
    a = np.arange(6, dtype=np.float64).reshape(2, 3) / 7
    v = np.linspace(0, 1, 5)
    with ArchiveWriter(str(tmp_path / "a.ark"), str(tmp_path / "a.scp")) as w:
        w.write("m1", a)
        w.write("v1", v)
        with pytest.raises(RuntimeError):
            w.write("bad", [1, 2, 3])
    raw = (tmp_path / "a.ark").read_bytes()
    expect = (b"m1 \0BFM \x04" + struct.pack("i", 2) + b"\x04" + struct.pack("i", 3) +
              a.astype(np.float32).tobytes() + b"v1 \0BFV \x04" + struct.pack("i", 5) +
              v.astype(np.float32).tobytes())
    assert raw == expect
    lines = (tmp_path / "a.scp").read_text().splitlines()
    assert lines[0] == f"m1\t{tmp_path / 'a.ark'}:3" and lines[1].startswith("v1\t")
    rd = ScriptReader(str(tmp_path / "a.scp"))
    assert np.array_equal(rd["m1"], a.astype(np.float32)) and np.array_equal(rd["v1"], v.astype(np.float32))
    with pytest.raises(RuntimeError):
        ArchiveWriter("")
    # ---- libs.spatial mirror: numpy in -> numpy out, reference dtypes ----
    rng = np.random.default_rng(31)
    x = pc.structured_audio(rng, 1, 3, 2400)[0]
    x = so.float_from_pcm16(so.pcm16_from_float(x))
    kw = dict(frame_len=128, frame_hop=64, center=True, window="hann", round_power_of_two=True,
              transpose=False)
    obs = so.multichannel_stft(x, out_dtype=np.complex64, **kw)                    # C x F x T
    S = np.ascontiguousarray(np.transpose(obs, (0, 2, 1)))                          # C x T x F
    F = S.shape[-1]
    topo = (0.0, 0.1, 0.25)
    gk = dict(num_bins=F, num_doa=21)
    srp = gs.srp_phat_linear(S, topo, **gk)
    ref_srp = sp.srp_phat_linear(S, topo, **gk)
    assert isinstance(srp, np.ndarray) and srp.dtype == ref_srp.dtype and srp.shape == ref_srp.shape
    assert np.max(np.abs(srp - ref_srp)) <= 5e-6 * np.max(np.abs(ref_srp))
    two = gs.srp_phat_linear(S[:2], topo[:2], normalize=False, **gk)               # N == 2: defaults win
    assert np.max(np.abs(two - sp.srp_phat_linear(S[:2], topo[:2], normalize=False, **gk))) <= 5e-6
    got = gs.ipd(S[0], S[2])
    assert got.dtype == np.float32 and pc._wrap_err(got, sp.ipd(S[0], S[2])) <= 5e-6
    assert np.max(np.abs(gs.msc(S, context=2) - sp.msc(S, context=2))) <= 1e-9
    sv = np.exp(1j * rng.uniform(0, 6.28, size=(3, F)))
    assert np.max(np.abs(gs.directional_feats(obs, sv, df_pair=[(0, 2)]) -
                         sp.directional_feats(obs, sv, df_pair=[(0, 2)]))) <= 5e-6
    t = gs.gcc_phat_diag(torch.from_numpy(S[0]), torch.from_numpy(S[1]), 0.4, 0.08, num_doas=13, num_bins=F)
    assert torch.is_tensor(t)
    assert np.max(np.abs(t.numpy() - sp.gcc_phat_diag(S[0], S[1], 0.4, 0.08, num_doas=13, num_bins=F))) <= 5e-6
    with pytest.raises(ValueError):
        gs.srp_phat_linear(S, np.array(topo))
    with pytest.raises(ValueError):
        gs.srp_phat_linear(S, (0.0, 0.1))
    # ---- the CLI, the reference's flags, all three feature types ----
    _write_wav(str(tmp_path / "utt1.wav"), x)
    (tmp_path / "wav.scp").write_text(f"utt1 {tmp_path / 'utt1.wav'}\n")
    env = dict(os.environ, SETK_B200_TEST_LIBRARY=emu_library_path, PYTHONPATH=ROOT)
    runner = (
        "import os, sys, runpy; sys.argv = sys.argv[1:];"
        "from setk_b200 import _lib; _lib.use_library(os.environ['SETK_B200_TEST_LIBRARY']);"
        "from setk_b200.libs import utils; utils.set_default_device('cpu');"
        "runpy.run_path(sys.argv[0], run_name='__main__')")
    script = os.path.join(ROOT, "scripts", "sptk", "compute_ipd_and_linear_srp.py")
    base = [sys.executable, "-c", runner, script, "--frame-len", "128", "--frame-hop", "64",
            "--center", "true"]
    cases = {
        "srp": (["--type", "srp", "--srp.topo", "0,0.1,0.25", "--srp.num_doa", "21"], ref_srp),
        "ipd": (["--type", "ipd", "--ipd.pair", "0,1;0,2", "--ipd.cos", "true"],
                np.hstack([sp.ipd(S[0], S[1], cos=True), sp.ipd(S[0], S[2], cos=True)])),
        "msc": (["--type", "msc", "--msc.ctx", "2"], sp.msc(S, context=2)),
    }
    for name, (flags, ref) in cases.items():
        ark, scp = tmp_path / f"{name}.ark", tmp_path / f"{name}.scp"
        subprocess.run(base + flags + ["--scp", str(scp), str(tmp_path / "wav.scp"), str(ark)], check=True,
                       env=env, capture_output=True)
        feats = ScriptReader(str(scp))["utt1"]
        assert feats.dtype == np.float32 and feats.shape == ref.shape, (name, feats.shape, ref.shape)
        assert np.max(np.abs(feats - ref)) <= 1e-5 * max(1.0, np.max(np.abs(ref))), name
    # ---- directional features from given steer vectors / from a TF-mask ----
    A = np.exp(1j * rng.uniform(0, 6.28, size=(3, 3, F)))                          # A x M x F
    np.save(str(tmp_path / "sv.npy"), A)
    script = os.path.join(ROOT, "scripts", "sptk", "compute_df_on_geometry.py")
    base = [sys.executable, "-c", runner, script, "--frame-len", "128", "--frame-hop", "64", "--center", "true"]
    ark, scp = tmp_path / "dfg.ark", tmp_path / "dfg.scp"
    subprocess.run(base + ["--doa-idx", "0,2", "--df-pair", "0,1;0,2", "--scp", str(scp),
                           str(tmp_path / "wav.scp"), str(tmp_path / "sv.npy"), str(ark)],
                   check=True, env=env, capture_output=True)
    dfs = np.stack([sp.directional_feats(obs, A[i], df_pair=[(0, 1), (0, 2)]) for i in (0, 2)])
    ref = dfs.transpose(1, 0, 2).reshape(dfs.shape[1], -1)
    feats = ScriptReader(str(scp))["utt1"]
    assert feats.shape == ref.shape and np.max(np.abs(feats - ref)) <= 1e-5
    mask = rng.uniform(0.05, 1.0, size=(S.shape[1], F)).astype(np.float32)         # T x F
    np.save(str(tmp_path / "mask.npy"), mask)
    (tmp_path / "mask.scp").write_text(f"utt1 {tmp_path / 'mask.npy'}\n")
    script = os.path.join(ROOT, "scripts", "sptk", "compute_df_on_mask.py")
    base = [sys.executable, "-c", runner, script, "--frame-len", "128", "--frame-hop", "64", "--center", "true"]
    ark, scp = tmp_path / "dfm.ark", tmp_path / "dfm.scp"
    subprocess.run(base + ["--mask-format", "numpy", "--df-pair", "0,2", "--scp", str(scp),
                           str(tmp_path / "wav.scp"), str(tmp_path / "mask.scp"), str(ark)],
                   check=True, env=env, capture_output=True)
    Rs = bo.compute_covar(obs.astype(np.complex128), mask.astype(np.float64))
    sv = bo.solve_pevd(Rs)                                                          # F x N (phase: arbitrary)
    ref = sp.directional_feats(obs, sv.T, df_pair=[(0, 2)])      # phase differences: sign/phase invariant
    feats = ScriptReader(str(scp))["utt1"]
    assert feats.shape == ref.shape and np.max(np.abs(feats - ref)) <= 2e-4
    # ---- SRP for a circular array: mean of the diagonal pairs' GCC-PHAT ----
    script = os.path.join(ROOT, "scripts", "sptk", "compute_circular_srp.py")
    base = [sys.executable, "-c", runner, script, "--frame-len", "128", "--frame-hop", "64", "--center", "true"]
    ark, scp = tmp_path / "csrp.ark", tmp_path / "csrp.scp"
    subprocess.run(base + ["--n", "3", "--d", "0.08", "--diag-pair", "0,2;1,2", "--num-doas", "17",
                           "--scp", str(scp), str(tmp_path / "wav.scp"), str(ark)],
                   check=True, env=env, capture_output=True)
    ref = np.average(np.stack([sp.gcc_phat_diag(S[i], S[j], min(i, j) * np.pi * 2 / 3, 0.08, num_bins=F,
                                                sr=16000, num_doas=17) for i, j in ((0, 2), (1, 2))]), axis=0)
    feats = ScriptReader(str(scp))["utt1"]
    assert feats.shape == ref.shape and np.max(np.abs(feats - ref)) <= 1e-5
    utils.set_default_device(None)


def test_geometry_based_beamformers(libs, tmp_path, emu_library_path):
    """DS / SD / fixed beamformers and beam_pattern vs the reference's own outputs (ref_fixed_bf.npz),
    and scripts/sptk/apply_fixed_beamformer.py (single and multiple beams) vs the oracle."""
    import parity_cases as pc
    from setk_b200.libs import beamformer as BF
    pc.check_fixed_beamformers(torch.device("cpu"))
    rng = np.random.default_rng(17)
    x = pc.structured_audio(rng, 1, 3, 3000)[0]
    x = so.float_from_pcm16(so.pcm16_from_float(x))
    kw = dict(frame_len=256, frame_hop=128, center=True, window="hann", round_power_of_two=True,
              transpose=False)
    obs = so.multichannel_stft(x, out_dtype=np.complex64, **kw)                    # 3 x F x T
    F = obs.shape[1]
    w0 = BF.LinearSDBeamformer([0.0, 0.06, 0.12]).weight(70.0, F)
    w1 = BF.LinearDSBeamformer([0.0, 0.06, 0.12]).weight(120.0, F)
    np.save(str(tmp_path / "w_single.npy"), w0)
    np.save(str(tmp_path / "w_multi.npy"), np.stack([w0, w1]))
    _write_wav(str(tmp_path / "utt1.wav"), x)
    (tmp_path / "wav.scp").write_text(f"utt1 {tmp_path / 'utt1.wav'}\n")
    (tmp_path / "beam.scp").write_text("utt1 1\n")
    env = dict(os.environ, SETK_B200_TEST_LIBRARY=emu_library_path, PYTHONPATH=ROOT)
    runner = (
        "import os, sys, runpy; sys.argv = sys.argv[1:];"
        "from setk_b200 import _lib; _lib.use_library(os.environ['SETK_B200_TEST_LIBRARY']);"
        "from setk_b200.libs import utils; utils.set_default_device('cpu');"
        "runpy.run_path(sys.argv[0], run_name='__main__')")
    script = os.path.join(ROOT, "scripts", "sptk", "apply_fixed_beamformer.py")
    base = [sys.executable, "-c", runner, script, "--frame-len", "256", "--frame-hop", "128", "--center", "true"]
    import scipy.io.wavfile as wavfile
    for tag, wfile, extra, w in (("single", "w_single.npy", [], w0),
                                 ("multi", "w_multi.npy", ["--beam", str(tmp_path / "beam.scp")], w1)):
        subprocess.run(base + extra + [str(tmp_path / "wav.scp"), str(tmp_path / wfile), str(tmp_path / tag)],
                       check=True, env=env, capture_output=True)
        sr, y = wavfile.read(str(tmp_path / tag / "utt1.wav"))
        enh = np.einsum("fn,nft->ft", w.conj(), obs.astype(np.complex128))
        yo = so.inverse_stft(enh, frame_len=256, frame_hop=128, center=True, window="hann", transpose=False,
                             norm=float(np.max(np.abs(x))))
        d = np.abs(y.astype(np.int64) - so.pcm16_from_float(yo).astype(np.int64))
        assert sr == 16000 and y.dtype == np.int16 and d.max() <= 1, (tag, int(d.max()))
    # scripts/sptk/apply_classic_beamformer.py: SD for a linear array (one DoA per utterance) and
    # DS in chunks (online: one DoA per --chunk-len frames), --normalize true
    script = os.path.join(ROOT, "scripts", "sptk", "apply_classic_beamformer.py")
    base = [sys.executable, "-c", runner, script, "--frame-len", "256", "--frame-hop", "128", "--center", "true",
            "--linear-topo", "0,0.06,0.12", "--normalize", "true"]
    T = obs.shape[-1]
    (tmp_path / "utt2doa").write_text("utt1 70\n")
    half = (T + 1) // 2
    runs = (("sd", ["--beamformer", "sd", "--utt2doa", str(tmp_path / "utt2doa")],
             np.einsum("fn,nft->ft", BF.LinearSDBeamformer([0.0, 0.06, 0.12]).weight(70.0, F, c=343).conj(),
                       obs.astype(np.complex128))),
            ("ds_online", ["--beamformer", "ds", "--chunk-len", str(half), "--doa", "30"], None))
    for tag, extra, enh in runs:
        if enh is None:
            (tmp_path / "utt2doa2").write_text("utt1 30 150\n")
            extra = ["--beamformer", "ds", "--chunk-len", str(half), "--utt2doa", str(tmp_path / "utt2doa2")]
            ds = BF.LinearDSBeamformer([0.0, 0.06, 0.12])
            o = obs.astype(np.complex128)
            enh = np.hstack([np.einsum("fn,nft->ft", ds.weight(30.0, F, c=343).conj(), o[:, :, :half]),
                             np.einsum("fn,nft->ft", ds.weight(150.0, F, c=343).conj(), o[:, :, half:])])
        subprocess.run(base + extra + [str(tmp_path / "wav.scp"), str(tmp_path / tag)], check=True, env=env,
                       capture_output=True)
        sr, y = wavfile.read(str(tmp_path / tag / "utt1.wav"))
        yo = so.inverse_stft(enh, frame_len=256, frame_hop=128, center=True, window="hann", transpose=False,
                             norm=float(np.max(np.abs(x))))
        d = np.abs(y.astype(np.int64) - so.pcm16_from_float(yo).astype(np.int64))
        assert sr == 16000 and d.max() <= 1, (tag, int(d.max()))


def test_facted_wpd_mirror(libs):
    """libs.wpe.facted_wpd (reference signature) on the CPU execution model vs the reference's output."""
    import parity_cases as pc
    from setk_b200.libs.wpe import facted_wpd
    err, mean_d, max_d = pc.check_wpd_fixture(torch.device("cpu"), "c3")
    with pytest.raises(RuntimeError):
        facted_wpd(np.zeros((3, 20, 33), dtype=np.float32))
    with pytest.raises(np.linalg.LinAlgError):
        facted_wpd(np.zeros((2, 30, 17), dtype=np.complex64), taps=2, delay=1, wpd_iters=1, cgmm_iters=1)


def test_apply_wpd_cli(tmp_path, emu, emu_library_path):
    """scripts/sptk/apply_wpd.py with the reference's flags vs the oracle's facted_wpd + inverse STFT."""
    from oracle import wpe_oracle as wo
    import parity_cases as pc
    rng = np.random.default_rng(23)
    x = pc.structured_audio(rng, 1, 3, 4000)[0]
    x = so.float_from_pcm16(so.pcm16_from_float(x))
    _write_wav(str(tmp_path / "utt1.wav"), x)
    (tmp_path / "wav.scp").write_text(f"utt1 {tmp_path / 'utt1.wav'}\n")
    env = dict(os.environ, SETK_B200_TEST_LIBRARY=emu_library_path, PYTHONPATH=ROOT)
    runner = (
        "import os, sys, runpy; sys.argv = sys.argv[1:];"
        "from setk_b200 import _lib; _lib.use_library(os.environ['SETK_B200_TEST_LIBRARY']);"
        "from setk_b200.libs import utils; utils.set_default_device('cpu');"
        "runpy.run_path(sys.argv[0], run_name='__main__')")
    cmd = [sys.executable, "-c", runner, os.path.join(ROOT, "scripts", "sptk", "apply_wpd.py"),
           "--frame-len", "256", "--frame-hop", "64", "--center", "true", "--taps", "3", "--delay", "2",
           "--wpd-iters", "2", "--cgmm-iters", "3", "--dump-mask", "true",
           str(tmp_path / "wav.scp"), str(tmp_path / "out")]
    subprocess.run(cmd, check=True, env=env, capture_output=True)
    kw = dict(frame_len=256, frame_hop=64, center=True, window="hann", round_power_of_two=True, transpose=True)
    obs = so.multichannel_stft(x, out_dtype=np.complex64, **kw)                    # N x T x F
    m_ref, e_ref = wo.facted_wpd(obs, cgmm_iters=3, wpd_iters=2, taps=3, delay=2, context=1)
    mask = np.load(str(tmp_path / "out" / "utt1.npy"))
    assert mask.shape == m_ref[..., 0].shape and np.abs(mask - m_ref[..., 0]).mean() <= 1e-5
    import scipy.io.wavfile as wavfile
    sr, y = wavfile.read(str(tmp_path / "out" / "utt1.wav"))
    assert sr == 16000 and y.dtype == np.int16 and y.ndim == 1
    # the output's per-bin phase is the eigenvector convention's (the reference's is LAPACK's):
    # compare the magnitudes of its STFT with the oracle's enhanced spectrum after the same rescale
    yo = so.inverse_stft(e_ref, frame_len=256, frame_hop=64, center=True, window="hann", transpose=True,
                         norm=float(np.max(np.abs(x))))
    assert abs(int(np.abs(y).max()) - int(np.abs(so.pcm16_from_float(yo)).max())) <= 2000
    assert len(y) == len(yo)


def test_permu_aligner_restores_a_scrambled_mask():
    from setk_b200.libs.cluster import permu_aligner
    rng = np.random.default_rng(12)
    K, T, F = 3, 40, 257
    act = (rng.uniform(size=(K, T)) > 0.5).astype(np.float64) + 0.05          # class activity over time
    masks = np.repeat(act[:, :, None], F, axis=2) + 0.02 * rng.uniform(size=(K, T, F))
    masks /= masks.sum(0, keepdims=True)
    scrambled = masks.copy()
    for f in range(F):
        scrambled[..., f] = masks[rng.permutation(K), :, f]
    out = permu_aligner(scrambled)
    # all bins carry one common class order
    ref_order = [int(np.argmax([np.sum(out[k, :, 0] * masks[j, :, 0]) for j in range(K)])) for k in range(K)]
    assert sorted(ref_order) == list(range(K))
    for f in range(F):
        assert np.allclose(out[..., f], masks[ref_order, :, f])
    with pytest.raises(ValueError):
        permu_aligner(np.zeros((2, 5, 100)))


def test_kaldi_matrix_reader(tmp_path):
    import struct
    from setk_b200.libs.data_handler import ScriptReader
    mat = np.arange(12, dtype=np.float32).reshape(3, 4)
    path = tmp_path / "m.ark"
    with open(path, "wb") as f:
        f.write(b"utt1 ")
        off = f.tell()
        f.write(b"\0B" + b"FM " + b"\4" + struct.pack("<i", 3) + b"\4" + struct.pack("<i", 4))
        f.write(mat.tobytes())
    (tmp_path / "m.scp").write_text(f"utt1 {path}:{off}\n")
    rd = ScriptReader(str(tmp_path / "m.scp"))
    assert "utt1" in rd and np.array_equal(rd["utt1"], mat)


def test_kaldi_compressed_matrix_reader(tmp_path):
    """CM / CM2 / CM3 archives (kaldi_io.py:248-318): hand-built bytes, and what the reference's own
    reader decodes from the same bytes (tests/golden/ref_kaldi_io.npz)."""
    import io
    import struct
    from setk_b200.libs.data_handler import ScriptReader, read_kaldi_matrix
    rng = np.random.default_rng(5)
    rows, cols = 7, 5
    blobs = {}
    pch = np.sort(rng.integers(0, 65535, size=(cols, 4)), axis=1).astype("<u2")
    u8 = rng.integers(0, 256, size=(cols, rows)).astype(np.uint8)
    u8[0, :3] = (64, 65, 193)                                    # the three segments' edges
    blobs["CM"] = (b"\0BCM " + struct.pack("<ffii", -3.0, 9.5, rows, cols) + pch.tobytes() + u8.tobytes())
    u16 = rng.integers(0, 65536, size=(rows, cols)).astype("<u2")
    blobs["CM2"] = b"\0BCM2 " + struct.pack("<ffii", 0.25, 4.0, rows, cols) + u16.tobytes()
    u8b = rng.integers(0, 256, size=(rows, cols)).astype(np.uint8)
    blobs["CM3"] = b"\0BCM3 " + struct.pack("<ffii", -1.0, 2.0, rows, cols) + u8b.tobytes()
    # expected values, straight from Kaldi's definition
    p = pch.astype(np.float32).T * np.float32(9.5) / 65535.0 + np.float32(-3.0)
    v = u8.astype(np.float32).T
    exp_cm = np.where(v <= 64, v * (p[1] - p[0]) / 64.0 + p[0],
                      np.where(v >= 193, (v - 192) * (p[3] - p[2]) / 63.0 + p[2], (v - 64) * (p[2] - p[1]) / 128.0 + p[1]))
    expect = {"CM": exp_cm, "CM2": 0.25 + u16.astype(np.float32) * float(4.0 / 65535.0),
              "CM3": -1.0 + u8b.astype(np.float32) * float(2.0 / 255.0)}
    ref = np.load(os.path.join(ROOT, "tests", "golden", "ref_kaldi_io.npz"))
    with open(tmp_path / "c.ark", "wb") as f, open(tmp_path / "c.scp", "w") as scp:
        for key, blob in blobs.items():
            f.write(key.encode() + b" ")
            scp.write(f"{key} {tmp_path / 'c.ark'}:{f.tell()}\n")
            f.write(blob)
    rd = ScriptReader(str(tmp_path / "c.scp"))
    for key, blob in blobs.items():
        got = read_kaldi_matrix(io.BytesIO(blob))
        assert got.shape == (rows, cols) and np.allclose(got, expect[key], rtol=1e-6, atol=1e-6), key
        assert np.array_equal(rd[key], got)
        assert ref[key + "/blob"].tobytes() == blob, key
        assert np.array_equal(ref[key + "/ref"], got), key
    # a mask through compress_kaldi_cm (what bench.py / the streamer ship to setk_cm_masks): the same
    # bytes read by this repo's reader and by the reference's, within the format's quantisation of the input
    from setk_b200.libs.data_handler import compress_kaldi_cm
    m = (rng.random((37, 19)) ** 2).astype(np.float32)
    blob = b"\0BCM " + compress_kaldi_cm(m)
    got = read_kaldi_matrix(io.BytesIO(blob))
    assert got.shape == m.shape and got.dtype == np.float32
    assert np.max(np.abs(got - m)) <= 0.02 * (m.max() - m.min())
    ref_blob = ref["mask_cm/blob"].tobytes()
    assert np.array_equal(read_kaldi_matrix(io.BytesIO(ref_blob)), ref["mask_cm/ref"])


def test_remaining_table_readers(tmp_path):
    """ArchiveReader (file / pipe), DirReader, SegmentWaveReader, BinaryReader, PickleReader, Mat* round trips."""
    import pickle
    from setk_b200.libs.data_handler import (ArchiveReader, ArchiveWriter, BinaryReader, DirReader, MatReader,
                                             MatWriter, PickleReader, SegmentWaveReader)
    a, v = np.arange(12, dtype=np.float32).reshape(3, 4), np.arange(5, dtype=np.float32)
    with ArchiveWriter(str(tmp_path / "x.ark")) as w:
        w.write("a", a)
        w.write("v", v)
    for spec in (str(tmp_path / "x.ark"), f"cat {tmp_path / 'x.ark'} |"):
        got = dict(ArchiveReader(spec))
        assert list(got) == ["a", "v"] and np.array_equal(got["a"], a) and np.array_equal(got["v"], v)
    x = (np.arange(2 * 4000, dtype=np.float32).reshape(2, 4000) % 200 - 100) / 32768.0
    _write_wav(str(tmp_path / "u1.wav"), x)
    (tmp_path / "wav.scp").write_text(f"u1 {tmp_path / 'u1.wav'}\n")
    (tmp_path / "segments").write_text("u1-a u1 100 1100\nu1-b u1 2000 2500\n")
    seg = SegmentWaveReader(str(tmp_path / "wav.scp"), str(tmp_path / "segments"), sr=16000)
    assert len(seg) == 2 and np.array_equal(seg["u1-a"], x[:, 100:1100]) and seg["u1-b"].shape == (2, 500)
    d = DirReader(str(tmp_path), "wav")
    assert list(d.index_keys) == ["u1"]
    v.tofile(str(tmp_path / "v.bin"))
    (tmp_path / "bin.scp").write_text(f"v {tmp_path / 'v.bin'}\n")
    assert np.array_equal(BinaryReader(str(tmp_path / "bin.scp"), length=5)["v"], v)
    with pytest.raises(RuntimeError):
        BinaryReader(str(tmp_path / "bin.scp"), length=4)["v"]
    with open(tmp_path / "o.pkl", "wb") as f:
        pickle.dump({"k": 1}, f)
    (tmp_path / "pkl.scp").write_text(f"o {tmp_path / 'o.pkl'}\n")
    assert PickleReader(str(tmp_path / "pkl.scp"))["o"] == {"k": 1}
    with MatWriter(str(tmp_path / "mats"), str(tmp_path / "mat.scp")) as w:
        w.write("m", a)
    assert np.array_equal(MatReader(str(tmp_path / "mat.scp"), "data")["m"], a)
    with pytest.raises(KeyError):
        MatReader(str(tmp_path / "mat.scp"), "nope")["m"]


def test_config3_fixture_cgmm_mask_gev(emu):
    """config 3 (8 ch, 1024-pt, reference CGMM mask -> GEV) on the CPU execution model."""
    import parity_cases as pc
    pc.check_config_fixture(emu, "cfg3", stft_from_oracle=True)
