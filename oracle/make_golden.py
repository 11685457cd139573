#!/usr/bin/env python
"""
oracle/make_golden.py -- generate tests/golden/*.npz from the REFERENCE's own
code (imported from /root/reference under oracle/ref_shim.py) and pin the
restatement (oracle/{stft,beamformer}_oracle.py) against it.

Run in the build container only (needs /root/reference):
    python -m oracle.make_golden

TEST INFRASTRUCTURE.  Writes:
  tests/golden/doc_adaptive_beamformer.npz
      the reference's shipped example doc/adaptive_beamformer/asset/egs.wav
      (5 ch x 94010, PCM-16), the CGMM mask the documented command produces
      (reference code, 20 iterations, seed 777), the shipped outputs
      {pmwf-0, pmwf-0-eig, pmwf-0-gev, gevd, gevd-ban, mvdr}.wav and the
      reference-code replay statistics of each (in PINNING.json).
  tests/golden/ref_small.npz
      seeded small synthetic cases pushed through the reference's
      forward_stft / compute_covar / solve_pevd / *Beamformer.weight /
      beamform / inverse_stft with float64 masks (complex128 path).
  tests/golden/ref_configs.npz
      BASELINE.json configs 3 (reference CGMM mask -> GEV, 8 ch, 1024-pt) and 4
      (reference WPE -> MVDR, 6 ch) on short seeded utterances.
  tests/golden/ref_restatement.npz
      the reference's forward_stft and Mvdr / Gevd / Pmwf Beamformer.run on a
      seeded 3-channel signal (complex128 path).
  tests/golden/ref_kaldi_io.npz
      CompressedMatrix blobs and what the reference's Kaldi reader decodes.
  tests/golden/PINNING.json
      what matched what, to how many LSB / what rel-inf.
"""
import json
import os
import sys

import numpy as np
import scipy.io.wavfile as wavfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402
from oracle import stft_oracle as so  # noqa: E402
from oracle import beamformer_oracle as bo  # noqa: E402

ASSET = "/root/reference/doc/adaptive_beamformer/asset/"
GOLD = os.path.join(ROOT, "tests", "golden")
STFT_KW = dict(frame_len=512, frame_hop=256, window="hann", center=True,
               transpose=False)


def lsb_stats(a, b):
    d = np.abs(a.astype(np.int64) - b.astype(np.int64))
    return int(d.max()), int(np.count_nonzero(d))


def ref_multichannel_stft(ref, samps, **kw):
    return np.stack([
        ref.utils.forward_stft(np.ascontiguousarray(samps[c]), **kw)
        for c in range(samps.shape[0])
    ])


def doc_example(ref, report):
    sr, egs = wavfile.read(ASSET + "egs.wav")
    assert sr == 16000 and egs.dtype == np.int16
    samps = so.float_from_pcm16(egs.T)                       # (5, 94010) f32
    stft_ref = ref_multichannel_stft(ref, samps, round_power_of_two=True,
                                     **STFT_KW)              # c64 (5,257,368)
    # --- documented mask command: estimate_cgmm_masks.py --num-iters 20
    np.random.seed(777)
    trainer = ref.cluster.CgmmTrainer(stft_ref, 2, gamma=None,
                                      update_alpha=False)
    masks = trainer.train(20)                                # K x F x T
    mask = np.transpose(masks, (0, 2, 1))[0].astype(np.float32)  # T x F
    norm = np.max(np.abs(samps))
    F = stft_ref.shape[1]

    B = ref.beamformer
    variants = {
        "pmwf-0": (B.PmwfBeamformer(F, beta=0, ref_channel=-1,
                                    rank1_appro=""), False),
        "pmwf-0-eig": (B.PmwfBeamformer(F, beta=0, ref_channel=-1,
                                        rank1_appro="eig"), False),
        "pmwf-0-gev": (B.PmwfBeamformer(F, beta=0, ref_channel=-1,
                                        rank1_appro="gev"), False),
        "gevd": (B.GevdBeamformer(F), False),
        "gevd-ban": (B.GevdBeamformer(F), True),
        "mvdr": (B.MvdrBeamformer(F), False),
    }
    out = {"egs_pcm16": egs.T.copy(), "mask": mask}
    speech_mask = np.minimum(mask, 1)
    for name, (bf, ban) in variants.items():
        shipped = wavfile.read(ASSET + name + ".wav")[1]
        enh = bf.run(speech_mask, stft_ref, mask_n=None, ban=ban)
        y = ref.utils.inverse_stft(enh, norm=norm, **STFT_KW)
        pcm = so.pcm16_from_float(y.astype(np.float32))
        mx, nd = lsb_stats(pcm, shipped)
        report["doc/" + name] = {
            "ref_replay_vs_shipped_max_lsb": mx,
            "ref_replay_vs_shipped_ndiff": nd,
            "n": int(shipped.shape[0])
        }
        out["shipped/" + name] = shipped
        # float64 replay (mask as float64 -> complex128 path of the reference)
        enh64 = bf.run(speech_mask.astype(np.float64),
                       stft_ref.astype(np.complex128), mask_n=None, ban=ban)
        # restatement vs reference (same inputs, float64)
        kind = {"pmwf-0": "pmwf", "pmwf-0-eig": "pmwf", "pmwf-0-gev": "pmwf",
                "gevd": "gevd", "gevd-ban": "gevd", "mvdr": "mvdr"}[name]
        r1 = {"pmwf-0-eig": "eig", "pmwf-0-gev": "gev"}.get(name, "")
        enh_o = bo.run_supervised(kind, speech_mask.astype(np.float64),
                                  stft_ref.astype(np.complex128), ban=ban,
                                  beta=0, ref_channel=-1, rank1_appro=r1)
        al, _ = bo.align_phase(enh_o, enh64)
        report["doc/" + name]["oracle_vs_ref64_relinf_aligned"] = bo.rel_inf(
            al, enh64)
        report["doc/" + name]["oracle_vs_ref64_relinf_raw"] = bo.rel_inf(
            enh_o, enh64)
    # end-to-end oracle on the PMWF chain vs shipped vector
    y_o, _, _ = bo.enhance_utterance(samps, mask, kind="pmwf", beta=0,
                                     stft_dtype=np.complex64, **{
                                         k: v for k, v in STFT_KW.items()
                                         if k != "transpose"
                                     })
    pcm = so.pcm16_from_float(y_o)
    mx, nd = lsb_stats(pcm, out["shipped/pmwf-0"])
    report["doc/pmwf-0"]["oracle_e2e_vs_shipped_max_lsb"] = mx
    report["doc/pmwf-0"]["oracle_e2e_vs_shipped_ndiff"] = nd
    # oracle STFT vs the (shimmed) reference STFT: same code path by
    # construction; recorded for completeness
    st_o = so.multichannel_stft(samps, round_power_of_two=True,
                                out_dtype=np.complex64, **STFT_KW)
    report["doc/stft_oracle_vs_refshim_maxabs"] = float(
        np.max(np.abs(st_o - stft_ref)))
    np.savez_compressed(os.path.join(GOLD, "doc_adaptive_beamformer.npz"),
                        **out)


def synth_case(rng, C, N, nsrc=None):
    """Small structured multichannel mixture (dominant target in every bin)."""
    nsrc = C + 2 if nsrc is None else nsrc
    env = 0.55 + 0.45 * np.cos(2 * np.pi * 4.0 * np.arange(N) / 16000.0 +
                               rng.uniform(0, 2 * np.pi))
    s = rng.standard_normal(N) * env
    taps = np.exp(-np.arange(64) / 8.0)

    def fir(x):
        h = rng.standard_normal(64) * taps
        h[0] = np.sign(h[0]) * (np.abs(h).max() + 0.5)
        return np.convolve(x, h)[:N]

    tgt = np.stack([fir(s) for _ in range(C)])
    noise = np.zeros((C, N))
    for _ in range(nsrc):
        v = rng.standard_normal(N)
        noise += np.stack([fir(v) for _ in range(C)])
    noise += 0.1 * np.std(tgt) * rng.standard_normal((C, N))
    g = np.sqrt(np.mean(tgt[0]**2) / (np.mean(noise[0]**2) * 10**(5 / 10)))
    noise *= g
    mix = tgt + noise
    scale = 0.5 / np.max(np.abs(mix))
    return (mix * scale).astype(np.float32), (tgt * scale), (noise * scale)


def small_cases(ref, report):
    rng = np.random.default_rng(20240923)
    out = {}
    cases = [
        # name, C, N, frame_len, hop, center, window
        ("c4_512", 4, 4100, 512, 256, True, "hann"),
        ("c5_400", 5, 3000, 400, 160, True, "hann"),       # pads to 512
        ("c2_256nc", 2, 2500, 256, 128, False, "hamming"),
        ("c8_1024", 8, 6000, 1024, 256, True, "sqrthann"),
    ]
    B = ref.beamformer
    for name, C, N, fl, hop, center, window in cases:
        mix, tgt, noise = synth_case(rng, C, N)
        kw = dict(frame_len=fl, frame_hop=hop, window=window, center=center,
                  transpose=False)
        obs = ref_multichannel_stft(ref, mix, round_power_of_two=True,
                                    **kw).astype(np.complex128)
        # float64 STFT for the "truth" (reference stores c64; oracle can keep
        # c128) -- recorded separately
        obs64 = so.multichannel_stft(mix, round_power_of_two=True,
                                     out_dtype=np.complex128, **kw)
        S = so.forward_stft(tgt[0].astype(np.float32), round_power_of_two=True,
                            **kw)
        V = so.forward_stft(noise[0].astype(np.float32),
                            round_power_of_two=True, **kw)
        # compute_mask.py:85-87,107 IRM
        irm = np.abs(S) / np.sqrt(np.abs(S)**2 + np.abs(V)**2 + so.EPSILON)
        mask = irm.T.astype(np.float64)                          # T x F
        F = obs.shape[1]
        Rs = B.compute_covar(obs, mask)
        Rn = B.compute_covar(obs, 1 - mask)
        w_mvdr = B.MvdrBeamformer(F).weight(Rs, Rn)
        w_gev = B.GevdBeamformer(F).weight(Rs, Rn)
        w_pmwf = B.PmwfBeamformer(F, beta=1, ref_channel=0).weight(Rs, Rn)
        enh = B.Beamformer().beamform(w_mvdr, obs)
        norm = float(np.max(np.abs(mix)))
        y = ref.utils.inverse_stft(enh, norm=norm, **kw)
        out[name + "/mix"] = mix
        out[name + "/mask"] = mask.astype(np.float32)
        out[name + "/Rs"] = Rs
        out[name + "/Rn"] = Rn
        out[name + "/w_mvdr"] = w_mvdr
        out[name + "/w_gev"] = w_gev
        out[name + "/w_pmwf1_ref0"] = w_pmwf
        out[name + "/enh_mvdr"] = enh
        out[name + "/y_mvdr"] = y
        out[name + "/cfg"] = np.array([C, N, fl, hop, int(center)])
        out[name + "/window"] = np.array(window)
        # ---- restatement vs reference, same float64 inputs ----
        rep = {}
        rep["stft_oracle64_vs_ref_c64_relinf"] = bo.rel_inf(obs64, obs)
        Rs_o = bo.compute_covar(obs, mask)
        rep["covar_relinf"] = bo.rel_inf(Rs_o, Rs)
        wm, _ = bo.align_phase(bo.mvdr_weight(Rs, Rn), w_mvdr)
        rep["mvdr_w_relinf_aligned"] = bo.rel_inf(wm, w_mvdr)
        wg, _ = bo.align_phase(bo.gevd_weight(Rs, Rn), w_gev)
        rep["gev_w_relinf_aligned"] = bo.rel_inf(wg, w_gev)
        wp, _ = bo.pmwf_weight(Rs, Rn, beta=1, ref_channel=0)
        rep["pmwf_w_relinf"] = bo.rel_inf(wp, w_pmwf)
        y_o = so.inverse_stft(bo.beamform(w_mvdr, obs), norm=norm, **kw)
        rep["istft_relinf"] = bo.rel_inf(y_o, y)
        ev = np.linalg.eigvalsh(Rs)
        rep["min_eig_gap_Rs"] = float(np.min(ev[:, -1] / np.maximum(
            ev[:, -2], 1e-300)))
        rep["max_cond_Rn"] = float(np.max(np.linalg.cond(Rn)))
        report["small/" + name] = rep
    np.savez_compressed(os.path.join(GOLD, "ref_small.npz"), **out)


def config_cases(ref, report):
    """
    BASELINE.json configs 3 and 4 as parity cases, with the mask producer /
    pre-processor run by the REFERENCE's own code (they are outside the hot path):
      cfg3: 8-ch, 1024-pt, mask = reference CGMM (CgmmTrainer, 20 iterations) -> GEV
      cfg4: 6-ch, 512-pt, STFT dereverberated by the reference WPE
            (taps 10, delay 3, context 1, 3 iterations) -> MVDR with an IRM mask
    """
    rng = np.random.default_rng(20240924)
    out = {}
    B = ref.beamformer
    # ---- config 3 ----
    C, N, fl, hop = 8, 24000, 1024, 256
    mix, tgt, noise = synth_case(rng, C, N)
    kw = dict(frame_len=fl, frame_hop=hop, window="hann", center=True, transpose=False)
    obs = ref_multichannel_stft(ref, mix, round_power_of_two=True, **kw)        # c64 N x F x T
    np.random.seed(777)
    gamma = ref.cluster.CgmmTrainer(obs, 2, gamma=None, update_alpha=False).train(20)
    mask = np.transpose(gamma, (0, 2, 1))[0].astype(np.float32)                  # T x F
    F = obs.shape[1]
    obs64 = obs.astype(np.complex128)
    m64 = np.minimum(mask, 1).astype(np.float64)
    enh = B.GevdBeamformer(F).run(m64, obs64)
    y = ref.utils.inverse_stft(enh, norm=float(np.max(np.abs(mix))), **kw)
    out["cfg3/mix"] = mix
    out["cfg3/mask_cgmm"] = mask
    out["cfg3/enh_gevd"] = enh.astype(np.complex64)
    out["cfg3/y_gevd"] = y.astype(np.float32)
    enh_o = bo.run_supervised("gevd", m64, obs64)
    report["cfg3/oracle_vs_ref_relinf_aligned"] = bo.rel_inf(bo.align_phase(enh_o, enh)[0], enh)
    report["cfg3/mask_mean"] = float(mask.mean())
    # ---- config 4 ----
    C, N, fl, hop = 6, 32000, 512, 256     # T = 126 frames >> 60 prediction taps
    mix, tgt, noise = synth_case(rng, C, N)
    kw = dict(frame_len=fl, frame_hop=hop, window="hann", center=True, transpose=False)
    obs = ref_multichannel_stft(ref, mix, round_power_of_two=True, **kw)
    # apply_wpe.py:45-60: wpe works on F x N x T
    derev = ref.wpe.wpe(np.einsum("nft->fnt", obs), taps=10, delay=3, context=1, num_iters=3)
    derev = np.einsum("fnt->nft", derev).astype(np.complex64)
    S = so.forward_stft(tgt[0].astype(np.float32), round_power_of_two=True, **kw)
    V = so.forward_stft(noise[0].astype(np.float32), round_power_of_two=True, **kw)
    mask = (np.abs(S) / np.sqrt(np.abs(S)**2 + np.abs(V)**2 + so.EPSILON)).T.astype(np.float32)
    F = obs.shape[1]
    enh = B.MvdrBeamformer(F).run(mask.astype(np.float64), derev.astype(np.complex128))
    out["cfg4/stft_wpe"] = derev
    out["cfg4/mask"] = mask
    out["cfg4/enh_mvdr"] = enh.astype(np.complex64)
    enh_o = bo.run_supervised("mvdr", mask.astype(np.float64), derev.astype(np.complex128))
    report["cfg4/oracle_vs_ref_relinf_aligned"] = bo.rel_inf(bo.align_phase(enh_o, enh)[0], enh)
    np.savez_compressed(os.path.join(GOLD, "ref_configs.npz"), **out)


def cgmm_cases(ref, report):
    """
    The CGMM paths the documented command does not take (it is pinned by
    doc_example / config_cases): a start from given posteriors, more than two
    classes, and the prior update -- CgmmTrainer(obs, K, gamma=..., update_alpha=...)
    (cluster.py:396-465) run by the REFERENCE on small mixtures.
    """
    from oracle import cgmm_oracle as co
    rng = np.random.default_rng(20240925)
    out = {}
    kw = dict(frame_len=512, frame_hop=256, window="hann", center=True, transpose=False)
    for name, C, N, K, iters, upd in (("k3_alpha", 3, 6000, 3, 6, True), ("k2_init", 4, 5000, 2, 5, False)):
        mix, _, _ = synth_case(rng, C, N)
        obs = ref_multichannel_stft(ref, mix, round_power_of_two=True, **kw)      # c64 C x F x T
        _, F, T = obs.shape
        if K == 2:
            init = rng.uniform(0.05, 0.95, size=(F, T)).astype(np.float32)
        else:
            init = rng.uniform(size=(K, F, T))
            init = (init / init.sum(0, keepdims=True)).astype(np.float32)
        gamma = ref.cluster.CgmmTrainer(obs, K, gamma=init.astype(np.float64),
                                        update_alpha=upd).train(iters)
        masks = np.transpose(gamma, (0, 2, 1)).astype(np.float32)                  # K x T x F
        out[name + "/mix"] = mix
        out[name + "/init_gamma"] = init
        out[name + "/masks"] = masks
        out[name + "/cfg"] = np.array([K, iters, int(upd)], dtype=np.int64)
        mo = co.cgmm_masks(obs, K, iters, init_gamma=init.astype(np.float64), update_alpha=upd)
        mo = mo[None] if K == 2 else mo
        report["cgmm/" + name + "/oracle_vs_ref_maxabs"] = float(
            np.max(np.abs(mo - np.transpose(gamma, (0, 2, 1))[:mo.shape[0]])))
    np.savez_compressed(os.path.join(GOLD, "ref_cgmm.npz"), **out)


def wpe_cases(ref, report):
    """
    libs/wpe.py wpe() run by the REFERENCE (complex64 in, as apply_wpe.py feeds it)
    on small mixtures; configs chosen so that T > channels * taps.
    """
    from oracle import wpe_oracle as wo
    rng = np.random.default_rng(20240926)
    out = {}
    for name, C, N, fl, hop, taps, delay, ctx, iters in (
            ("c3_t4", 3, 6000, 512, 128, 4, 2, 1, 2),
            ("c4_t10", 4, 20000, 512, 256, 10, 3, 1, 3),
            ("c2_t6_ctx0", 2, 5000, 256, 64, 6, 1, 0, 1)):
        mix, _, _ = synth_case(rng, C, N)
        kw = dict(frame_len=fl, frame_hop=hop, window="hann", center=True, transpose=False)
        obs = ref_multichannel_stft(ref, mix, round_power_of_two=True, **kw)        # c64 C x F x T
        derev = ref.wpe.wpe(np.einsum("nft->fnt", obs), taps=taps, delay=delay, context=ctx,
                            num_iters=iters)                                        # F x N x T
        out[name + "/mix"] = mix
        out[name + "/cfg"] = np.array([fl, hop, taps, delay, ctx, iters], dtype=np.int64)
        out[name + "/derev"] = np.einsum("fnt->nft", derev).astype(np.complex64)
        o32 = wo.wpe(np.einsum("nft->fnt", obs), taps, delay, ctx, iters, dtype=np.complex64)
        o64 = wo.wpe(np.einsum("nft->fnt", obs), taps, delay, ctx, iters, dtype=np.complex128)
        report["wpe/" + name + "/oracle_c64_vs_ref_relinf"] = bo.rel_inf(o32, derev)
        report["wpe/" + name + "/oracle_c128_vs_ref_relinf"] = bo.rel_inf(o64, derev)
    np.savez_compressed(os.path.join(GOLD, "ref_wpe.npz"), **out)


def spatial_cases(ref, report):
    """
    libs/spatial.py run by the REFERENCE on STFTs of small seeded mixtures (complex64, as
    SpectrogramReader feeds it): ipd (3 modes), directional_feats (all pairs / given pairs),
    gcc_phat_linear (DOA and TDOA grids), gcc_phat_diag, srp_phat_linear (2 and 4 mics),
    msc (context 0..2).  The restatement must reproduce every array exactly.
    """
    from oracle import spatial_oracle as sp
    rng = np.random.default_rng(20240927)
    out = {}
    worst = 0.0

    def pin(key, got_ref, got_oracle):
        nonlocal worst
        out[key] = got_ref
        worst = max(worst, float(np.max(np.abs(np.asarray(got_ref) - np.asarray(got_oracle)))))

    for name, C, N, fl, hop in (("c4_512", 4, 9000, 512, 256), ("c3_256", 3, 5000, 256, 128),
                                ("c2_1024", 2, 12000, 1024, 256)):
        mix, _, _ = synth_case(rng, C, N)
        kw = dict(frame_len=fl, frame_hop=hop, window="hann", center=True, transpose=False)
        obs = ref_multichannel_stft(ref, mix, round_power_of_two=True, **kw)        # c64 C x F x T
        F = obs.shape[1]
        S = np.ascontiguousarray(np.transpose(obs, (0, 2, 1)))                      # C x T x F
        out[name + "/mix"] = mix
        out[name + "/cfg"] = np.array([fl, hop], dtype=np.int64)
        pin(name + "/ipd", ref.spatial.ipd(S[0], S[1]), sp.ipd(S[0], S[1]))
        pin(name + "/ipd_cos", ref.spatial.ipd(S[0], S[1], cos=True), sp.ipd(S[0], S[1], cos=True))
        pin(name + "/ipd_cos_sin", ref.spatial.ipd(S[0], S[C - 1], cos=True, sin=True),
            sp.ipd(S[0], S[C - 1], cos=True, sin=True))
        steer = np.exp(-1j * rng.uniform(0, 2 * np.pi, size=(C, F)))                # complex128
        out[name + "/steer"] = steer
        pin(name + "/df", ref.spatial.directional_feats(obs, steer), sp.directional_feats(obs, steer))
        pairs = [(0, C - 1), (C - 1, 0)] if C > 2 else [(1, 0)]
        out[name + "/df_pairs"] = np.array(pairs, dtype=np.int32)
        pin(name + "/df_given_pairs", ref.spatial.directional_feats(obs, steer, df_pair=pairs),
            sp.directional_feats(obs, steer, df_pair=pairs))
        gk = dict(num_bins=F, num_doa=37)
        pin(name + "/gcc", ref.spatial.gcc_phat_linear(S[0], S[1], 0.07, **gk),
            sp.gcc_phat_linear(S[0], S[1], 0.07, **gk))
        pin(name + "/gcc_tdoa_raw",
            ref.spatial.gcc_phat_linear(S[0], S[1], -0.05, normalize=False, apply_floor=False,
                                        samp_doa=False, **gk),
            sp.gcc_phat_linear(S[0], S[1], -0.05, normalize=False, apply_floor=False, samp_doa=False,
                               **gk))
        pin(name + "/gcc_diag", ref.spatial.gcc_phat_diag(S[0], S[1], 0.3, 0.1, num_doas=25, num_bins=F),
            sp.gcc_phat_diag(S[0], S[1], 0.3, 0.1, num_doas=25, num_bins=F))
        d = [0.04 * i for i in range(C)]
        out[name + "/topo"] = np.array(d)
        pin(name + "/srp", ref.spatial.srp_phat_linear(S, d, **gk), sp.srp_phat_linear(S, d, **gk))
        for ctx in (0, 1, 2):
            pin(name + f"/msc_ctx{ctx}", ref.spatial.msc(S, context=ctx), sp.msc(S, context=ctx))
        pin(name + "/msc_raw", ref.spatial.msc(S, context=1, normalize=False),
            sp.msc(S, context=1, normalize=False))
    report["spatial/oracle_vs_ref_maxabs"] = worst
    np.savez_compressed(os.path.join(GOLD, "ref_spatial.npz"), **out)


def fixed_cases(ref, report):
    """
    Geometry-based beamformers of libs/beamformer.py (106-212, 323-512) run by the REFERENCE:
    weights of the DS / SD beamformers for linear and circular arrays, a beam pattern, and the
    enhanced STFT of run(doa, obs) / FixedBeamformer.run(obs) on a seeded 4-channel mixture.
    """
    rng = np.random.default_rng(20240928)
    bf = ref.beamformer
    out = {}
    mix, _, _ = synth_case(rng, 4, 7000)
    kw = dict(frame_len=256, frame_hop=128, window="hann", center=True, transpose=False)
    obs = ref_multichannel_stft(ref, mix, round_power_of_two=True, **kw)            # c64 4 x F x T
    F = obs.shape[1]
    out["mix"] = mix
    topo = [0.0, 0.05, 0.1, 0.15]
    for name, obj, doa in (("lin_ds", bf.LinearDSBeamformer(topo), 60.0),
                           ("lin_sd", bf.LinearSDBeamformer(topo), 110.0),
                           ("cir_ds", bf.CircularDSBeamformer(0.05, 4), 45.0),
                           ("cir_sd", bf.CircularSDBeamformer(0.05, 3, center=True), 200.0)):
        out[name + "/weight"] = obj.weight(doa, F)
        out[name + "/enh"] = obj.run(doa, obs)
        out[name + "/doa"] = np.array(doa)
    out["cir_sd/distance_mat"] = bf.CircularSDBeamformer(0.05, 3, center=True).distance_mat
    out["fixed/enh"] = bf.FixedBeamformer(out["lin_sd/weight"]).run(obs)
    sv = np.stack([bf.linear_steer_vector(np.array(topo), d, F) for d in (0.0, 45.0, 90.0, 135.0)], axis=1)
    out["pattern/sv"] = sv                                                           # F x D x N
    out["pattern/single"] = bf.beam_pattern(out["lin_ds/weight"], sv)
    out["pattern/multi"] = np.stack(bf.beam_pattern(np.stack([out["lin_ds/weight"], out["lin_sd/weight"]]), sv))
    out["diffuse"] = bf.diffuse_covar(F, np.abs(np.subtract.outer(topo, topo)), diag_eps=0.01)
    report["fixed/cases"] = sorted(out)
    np.savez_compressed(os.path.join(GOLD, "ref_fixed_bf.npz"), **out)


def wpd_cases(ref, report):
    """
    libs/wpe.py facted_wpd() run by the REFERENCE (complex64 observations, as apply_wpd.py feeds
    it) on small mixtures: the final 2-class mask and the enhanced spectrum.
    """
    from oracle import wpe_oracle as wo
    rng = np.random.default_rng(20240929)
    out = {}
    for name, C, N, fl, hop, taps, delay, ctx, ci, wi in (("c3", 3, 6000, 256, 64, 3, 2, 1, 4, 2),
                                                        ("c4", 4, 9000, 256, 128, 4, 3, 1, 3, 3)):
        mix, _, _ = synth_case(rng, C, N)
        kw = dict(frame_len=fl, frame_hop=hop, window="hann", center=True, transpose=True)
        obs = ref_multichannel_stft(ref, mix, round_power_of_two=True, **kw)        # c64 C x T x F
        tf_mask, enh = ref.wpe.facted_wpd(obs, cgmm_iters=ci, wpd_iters=wi, taps=taps, delay=delay,
                                          context=ctx)
        out[name + "/mix"] = mix
        out[name + "/cfg"] = np.array([fl, hop, taps, delay, ctx, ci, wi], dtype=np.int64)
        out[name + "/tf_mask"] = tf_mask.astype(np.float32)                          # T x F x 2
        out[name + "/enh"] = enh.astype(np.complex64)                                # T x F
        for tag, dt in (("c64", np.complex64), ("c128", np.complex128)):
            m, e = wo.facted_wpd(obs, cgmm_iters=ci, wpd_iters=wi, taps=taps, delay=delay, context=ctx, dtype=dt)
            ea, _ = bo.align_phase(e.T, enh.T)                                       # per bin
            report[f"wpd/{name}/oracle_{tag}_enh_vs_ref_relinf"] = bo.rel_inf(ea, enh.T)
            report[f"wpd/{name}/oracle_{tag}_mask_vs_ref_maxabs"] = float(np.max(np.abs(m - tf_mask)))
    np.savez_compressed(os.path.join(GOLD, "ref_wpd.npz"), **out)


def restatement_cases(ref, report):
    """
    The reference's forward_stft and its Mvdr / Gevd / Pmwf(beta=0) Beamformer.run on a seeded
    3-channel signal and a uniform random mask (complex128 observations), for the CPU test that
    cross-checks the restatement against the reference's code.  The inputs are regenerated from
    the same seed by the test; the outputs are stored at a seeded sample of 64 frequency bins (DC
    and Nyquist included) to keep the fixture small: bins are independent in all of them.
    """
    rng = np.random.default_rng(3)
    C, N = 3, 5000
    x = (rng.standard_normal((C, N)) * 0.1).astype(np.float32)
    kw = dict(frame_len=512, frame_hop=256, center=True, window="hann", transpose=False)
    S = ref_multichannel_stft(ref, x, round_power_of_two=True, **kw)                 # c64 C x F x T
    T, F = S.shape[2], S.shape[1]
    mask = rng.uniform(0, 1, (T, F))
    obs = S.astype(np.complex128)
    bins = np.unique(np.concatenate([[0, F - 1], np.random.default_rng(4).choice(np.arange(1, F - 1), 62,
                                                                                  replace=False)]))
    out = {"bins": bins, "stft": S[:, bins]}
    for kind, bf in (("mvdr", ref.beamformer.MvdrBeamformer(F)),
                     ("gevd", ref.beamformer.GevdBeamformer(F)),
                     ("pmwf", ref.beamformer.PmwfBeamformer(F, beta=0))):
        out["enh_" + kind] = bf.run(mask, obs, ban=(kind == "gevd"))[bins]
    np.savez_compressed(os.path.join(GOLD, "ref_restatement.npz"), **out)


def kaldi_cases(ref, report):
    """
    The reference's Kaldi reader (libs/kaldi_io.py read_float_mat_vec) on CompressedMatrix blobs:
    hand-built CM / CM2 / CM3 bytes (the same seeded bytes the CPU test builds) and a mask through
    this repo's compress_kaldi_cm.  Stores each blob with what the reference decodes from it.
    """
    import importlib
    import io
    import struct
    from setk_b200.libs.data_handler import compress_kaldi_cm
    kio = importlib.import_module("libs.kaldi_io")
    rng = np.random.default_rng(5)
    rows, cols = 7, 5
    blobs = {}
    pch = np.sort(rng.integers(0, 65535, size=(cols, 4)), axis=1).astype("<u2")
    u8 = rng.integers(0, 256, size=(cols, rows)).astype(np.uint8)
    u8[0, :3] = (64, 65, 193)
    blobs["CM"] = b"\0BCM " + struct.pack("<ffii", -3.0, 9.5, rows, cols) + pch.tobytes() + u8.tobytes()
    u16 = rng.integers(0, 65536, size=(rows, cols)).astype("<u2")
    blobs["CM2"] = b"\0BCM2 " + struct.pack("<ffii", 0.25, 4.0, rows, cols) + u16.tobytes()
    u8b = rng.integers(0, 256, size=(rows, cols)).astype(np.uint8)
    blobs["CM3"] = b"\0BCM3 " + struct.pack("<ffii", -1.0, 2.0, rows, cols) + u8b.tobytes()
    m = (rng.random((37, 19)) ** 2).astype(np.float32)
    blobs["mask_cm"] = b"\0BCM " + compress_kaldi_cm(m)
    out = {}
    for key, blob in blobs.items():
        out[key + "/blob"] = np.frombuffer(blob, dtype=np.uint8)
        out[key + "/ref"] = kio.read_float_mat_vec(io.BufferedReader(io.BytesIO(blob)), direct_access=True)
    np.savez_compressed(os.path.join(GOLD, "ref_kaldi_io.npz"), **out)


def main():
    if len(sys.argv) > 1 and sys.argv[1] in ("cgmm", "wpe", "spatial", "fixed", "wpd", "restatement",
                                             "kaldi"):   # add one fixture only
        ref = ref_shim.load_reference()
        report = {}
        {"cgmm": cgmm_cases, "wpe": wpe_cases, "spatial": spatial_cases, "fixed": fixed_cases,
         "wpd": wpd_cases, "restatement": restatement_cases, "kaldi": kaldi_cases}[sys.argv[1]](ref, report)
        path = os.path.join(GOLD, "PINNING.json")
        with open(path) as f:
            full = json.load(f)
        full.update(report)
        with open(path, "w") as f:
            json.dump(full, f, indent=1, sort_keys=True)
        print(json.dumps(report, indent=1, sort_keys=True))
        return 0
    if not ref_shim.reference_available():
        print("reference tree absent; nothing generated", file=sys.stderr)
        return 1
    os.makedirs(GOLD, exist_ok=True)
    ref = ref_shim.load_reference()
    report = {
        "generated_by": "oracle/make_golden.py",
        "reference": "/root/reference (funcwj/setk @ 50e4da0) under oracle/ref_shim.py",
        "numpy": np.__version__,
    }
    doc_example(ref, report)
    small_cases(ref, report)
    config_cases(ref, report)
    cgmm_cases(ref, report)
    wpe_cases(ref, report)
    spatial_cases(ref, report)
    fixed_cases(ref, report)
    wpd_cases(ref, report)
    restatement_cases(ref, report)
    kaldi_cases(ref, report)
    with open(os.path.join(GOLD, "PINNING.json"), "w") as f:
        json.dump(report, f, indent=1, sort_keys=True)
    print(json.dumps(report, indent=1, sort_keys=True))
    return 0


if __name__ == "__main__":
    sys.exit(main())
