"""
CPU tier: the oracle (oracle/*.py, the CPU restatement of the reference) against
the golden vectors generated from the reference's own code and against the
reference's shipped doc vectors (tests/golden/, oracle/make_golden.py).
"""
import json
import os

import numpy as np

from oracle import beamformer_oracle as bo
from oracle import stft_oracle as so

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_pinning_report_records_reference_agreement():
    with open(os.path.join(GOLD, "PINNING.json")) as f:
        rep = json.load(f)
    # reference replay (its own code, imported under the shim) vs its shipped vectors
    for name in ("doc/pmwf-0", "doc/pmwf-0-eig", "doc/pmwf-0-gev"):
        assert rep[name]["ref_replay_vs_shipped_max_lsb"] <= 1
        assert rep[name]["oracle_vs_ref64_relinf_aligned"] <= 1e-12
    assert rep["doc/pmwf-0"]["oracle_e2e_vs_shipped_max_lsb"] <= 1
    assert rep["doc/stft_oracle_vs_refshim_maxabs"] == 0.0
    for name in ("small/c4_512", "small/c5_400", "small/c2_256nc", "small/c8_1024"):
        assert rep[name]["covar_relinf"] <= 1e-12
        assert rep[name]["mvdr_w_relinf_aligned"] <= 1e-12
        assert rep[name]["gev_w_relinf_aligned"] <= 1e-12
        assert rep[name]["istft_relinf"] <= 1e-12


def test_oracle_reproduces_reference_small_cases():
    g = np.load(os.path.join(GOLD, "ref_small.npz"))
    for name in ("c4_512", "c5_400", "c2_256nc", "c8_1024"):
        C, N, fl, hop, center = [int(v) for v in g[name + "/cfg"]]
        window = str(g[name + "/window"])
        kw = dict(frame_len=fl, frame_hop=hop, center=bool(center), window=window, transpose=False)
        mix, mask = g[name + "/mix"], g[name + "/mask"].astype(np.float64)
        obs = so.multichannel_stft(mix, round_power_of_two=True, out_dtype=np.complex64,
                                   **kw).astype(np.complex128)
        Rs = bo.compute_covar(obs, mask)
        Rn = bo.compute_covar(obs, 1 - mask)
        # the fixture keeps the mask as float32 (the covariances were made with float64)
        assert bo.rel_inf(Rs, g[name + "/Rs"]) <= 1e-6
        assert bo.rel_inf(Rn, g[name + "/Rn"]) <= 1e-6     # 1 - mask near 0 amplifies it
        Rs, Rn = g[name + "/Rs"], g[name + "/Rn"]       # the weights are pinned on the reference's own
        w = bo.align_phase(bo.mvdr_weight(Rs, Rn), g[name + "/w_mvdr"])[0]
        assert bo.rel_inf(w, g[name + "/w_mvdr"]) <= 1e-10
        w = bo.align_phase(bo.gevd_weight(Rs, Rn), g[name + "/w_gev"])[0]
        assert bo.rel_inf(w, g[name + "/w_gev"]) <= 1e-10
        w, _ = bo.pmwf_weight(Rs, Rn, beta=1, ref_channel=0)
        assert bo.rel_inf(w, g[name + "/w_pmwf1_ref0"]) <= 1e-10
        enh = bo.beamform(g[name + "/w_mvdr"], obs)
        assert bo.rel_inf(enh, g[name + "/enh_mvdr"]) <= 1e-12
        y = so.inverse_stft(enh, norm=float(np.max(np.abs(mix))), **kw)
        assert y.shape == g[name + "/y_mvdr"].shape
        assert bo.rel_inf(y, g[name + "/y_mvdr"]) <= 1e-12


def test_oracle_end_to_end_matches_shipped_doc_vector():
    """PMWF is phase invariant: the shipped PCM-16 file pins the whole chain (<= 1 LSB)."""
    g = np.load(os.path.join(GOLD, "doc_adaptive_beamformer.npz"))
    samps = so.float_from_pcm16(g["egs_pcm16"])
    for name, r1 in (("pmwf-0", ""), ("pmwf-0-eig", "eig")):
        y, _, _ = bo.enhance_utterance(samps, g["mask"], kind="pmwf", beta=0, rank1_appro=r1,
                                       stft_dtype=np.complex64)
        d = np.abs(so.pcm16_from_float(y).astype(np.int64) - g["shipped/" + name].astype(np.int64))
        assert d.max() <= 1
        assert np.mean(d > 0) <= 0.05


def test_oracle_reproduces_reference_config_cases():
    """configs 3 / 4: reference CGMM mask -> GEV, reference WPE -> MVDR (ref_configs.npz)."""
    g = np.load(os.path.join(GOLD, "ref_configs.npz"))
    kw = dict(frame_len=1024, frame_hop=256, center=True, window="hann", transpose=False)
    obs = so.multichannel_stft(g["cfg3/mix"], round_power_of_two=True, out_dtype=np.complex64,
                               **kw).astype(np.complex128)
    m = np.minimum(g["cfg3/mask_cgmm"], 1).astype(np.float64)
    enh = bo.run_supervised("gevd", m, obs)
    ref = g["cfg3/enh_gevd"].astype(np.complex128)
    assert bo.rel_inf(bo.align_phase(enh, ref)[0], ref) <= 1e-6      # fixture stored as complex64
    enh4 = bo.run_supervised("mvdr", g["cfg4/mask"].astype(np.float64),
                             g["cfg4/stft_wpe"].astype(np.complex128))
    ref4 = g["cfg4/enh_mvdr"].astype(np.complex128)
    assert bo.rel_inf(bo.align_phase(enh4, ref4)[0], ref4) <= 1e-6


def test_cgmm_oracle_pinned_to_reference_masks():
    """
    cluster.py CgmmTrainer run by the reference (make_golden.py): the documented
    command on egs.wav, the config-3 mixture, and the given-posteriors / 3-class /
    prior-update paths.  With the reference's complex64 start the restatement agrees
    to the float32 rounding of the stored masks.
    """
    from oracle import cgmm_oracle as co
    g = np.load(os.path.join(GOLD, "doc_adaptive_beamformer.npz"))
    kw = dict(frame_len=512, frame_hop=256, center=True, window="hann", transpose=False)
    obs = so.multichannel_stft(so.float_from_pcm16(g["egs_pcm16"]), round_power_of_two=True,
                               out_dtype=np.complex64, **kw)
    m = co.cgmm_masks(obs, 2, 20, start_dtype=np.complex64)
    assert np.max(np.abs(m - g["mask"])) <= 1e-7
    g3 = np.load(os.path.join(GOLD, "ref_configs.npz"))
    kw["frame_len"] = 1024
    obs = so.multichannel_stft(g3["cfg3/mix"], round_power_of_two=True, out_dtype=np.complex64, **kw)
    m = co.cgmm_masks(obs, 2, 20, start_dtype=np.complex64)
    assert np.max(np.abs(m - g3["cfg3/mask_cgmm"])) <= 1e-7
    # the float64 start moves a few cells: the reference's own sensitivity (see the oracle header)
    d = np.abs(co.cgmm_masks(obs, 2, 20) - g3["cfg3/mask_cgmm"])
    assert d.mean() <= 5e-6 and d.max() <= 1e-2
    gc = np.load(os.path.join(GOLD, "ref_cgmm.npz"))
    kw["frame_len"] = 512
    for name in ("k3_alpha", "k2_init"):
        K, iters, upd = (int(v) for v in gc[name + "/cfg"])
        obs = so.multichannel_stft(gc[name + "/mix"], round_power_of_two=True, out_dtype=np.complex64, **kw)
        m = co.cgmm_masks(obs, K, iters, init_gamma=gc[name + "/init_gamma"].astype(np.float64),
                          update_alpha=bool(upd))
        m = m[None] if K == 2 else m
        assert np.max(np.abs(m - gc[name + "/masks"][:m.shape[0]])) <= 1e-7


def test_wpe_oracle_pinned_to_reference():
    """libs/wpe.py wpe() run by the reference on complex64 STFTs (ref_wpe.npz)."""
    from oracle import wpe_oracle as wo
    g = np.load(os.path.join(GOLD, "ref_wpe.npz"))
    for name in ("c3_t4", "c4_t10", "c2_t6_ctx0"):
        fl, hop, taps, delay, ctx, iters = (int(v) for v in g[name + "/cfg"])
        obs = so.multichannel_stft(g[name + "/mix"], frame_len=fl, frame_hop=hop, center=True,
                                   window="hann", round_power_of_two=True, transpose=False,
                                   out_dtype=np.complex64)
        x = np.einsum("nft->fnt", obs)
        ref = np.einsum("nft->fnt", g[name + "/derev"])
        assert bo.rel_inf(wo.wpe(x, taps, delay, ctx, iters, dtype=np.complex64), ref) <= 1e-6
        assert bo.rel_inf(wo.wpe(x, taps, delay, ctx, iters), ref) <= 1e-6      # float64 arithmetic


def test_bookkeeping_table():
    """SURVEY.md Appendix A: frame counts and iSTFT lengths at N = 160000, hop 256."""
    rows = [(512, True, 512, 257, 626, 160000), (1024, True, 1024, 513, 626, 160000),
            (400, True, 512, 257, 626, 160000), (512, False, 512, 257, 624, 160000),
            (1024, False, 1024, 513, 622, 160000)]
    for fl, center, n_fft, F, T, n_out in rows:
        assert so.nextpow2(fl) == n_fft
        assert so.num_frames(160000, n_fft, 256, center) == T
        if center:
            assert so.istft_length(T, n_fft, 256, center) == 256 * (T - 1)
    assert so.num_frames(94010, 512, 256, True) == 368
    assert so.istft_length(368, 512, 256, True) == 93952


def test_stft_istft_round_trip():
    rng = np.random.default_rng(0)
    x = rng.standard_normal(16000).astype(np.float32)
    for fl, hop in ((512, 256), (1024, 256), (400, 160)):
        S = so.forward_stft(x, fl, hop, center=True, transpose=False)
        y = so.inverse_stft(S, fl, hop, center=True, transpose=False)
        n = min(len(x), len(y))
        assert bo.rel_inf(y[:n], x[:n].astype(np.float64)) <= 1e-6


def test_restatement_against_reference_outputs():
    """The reference's forward_stft and Mvdr / Gevd / Pmwf Beamformer.run on the same seeded input
    (ref_restatement.npz, at a sample of frequency bins)."""
    g = np.load(os.path.join(GOLD, "ref_restatement.npz"))
    bins = g["bins"]
    rng = np.random.default_rng(3)
    C, N = 3, 5000
    x = (rng.standard_normal((C, N)) * 0.1).astype(np.float32)
    kw = dict(frame_len=512, frame_hop=256, center=True, window="hann", transpose=False)
    S_or = so.multichannel_stft(x, round_power_of_two=True, out_dtype=np.complex64, **kw)
    assert np.array_equal(S_or[:, bins], g["stft"])
    T, F = S_or.shape[2], S_or.shape[1]
    mask = rng.uniform(0, 1, (T, F))
    obs = S_or.astype(np.complex128)
    for kind in ("mvdr", "gevd", "pmwf"):
        e_ref = g["enh_" + kind]
        e_or = bo.run_supervised(kind, mask, obs, ban=(kind == "gevd"))[bins]
        assert bo.rel_inf(bo.align_phase(e_or, e_ref)[0], e_ref) <= 1e-10


def test_spatial_oracle_pinned_to_reference():
    """libs/spatial.py run by the reference on complex64 STFTs (ref_spatial.npz): bit for bit."""
    from oracle import spatial_oracle as sp
    from oracle import stft_oracle as so
    g = np.load(os.path.join(GOLD, "ref_spatial.npz"))
    for name in ("c4_512", "c3_256", "c2_1024"):
        fl, hop = (int(v) for v in g[name + "/cfg"])
        mix = g[name + "/mix"]
        obs = np.stack([so.stft(mix[c], fl, hop, fl, window="hann", center=True, out_dtype=np.complex64)
                        for c in range(mix.shape[0])])
        S = np.ascontiguousarray(np.transpose(obs, (0, 2, 1)))
        C, _, F = S.shape
        steer = g[name + "/steer"]
        pairs = [tuple(int(v) for v in p) for p in g[name + "/df_pairs"]]
        gk = dict(num_bins=F, num_doa=37)
        got = {
            "ipd": sp.ipd(S[0], S[1]), "ipd_cos": sp.ipd(S[0], S[1], cos=True),
            "ipd_cos_sin": sp.ipd(S[0], S[C - 1], cos=True, sin=True),
            "df": sp.directional_feats(obs, steer),
            "df_given_pairs": sp.directional_feats(obs, steer, df_pair=pairs),
            "gcc": sp.gcc_phat_linear(S[0], S[1], 0.07, **gk),
            "gcc_tdoa_raw": sp.gcc_phat_linear(S[0], S[1], -0.05, normalize=False, apply_floor=False,
                                               samp_doa=False, **gk),
            "gcc_diag": sp.gcc_phat_diag(S[0], S[1], 0.3, 0.1, num_doas=25, num_bins=F),
            "srp": sp.srp_phat_linear(S, list(g[name + "/topo"]), **gk),
            "msc_ctx0": sp.msc(S, context=0), "msc_ctx1": sp.msc(S, context=1),
            "msc_ctx2": sp.msc(S, context=2), "msc_raw": sp.msc(S, context=1, normalize=False),
        }
        for k, v in got.items():
            ref = g[name + "/" + k]
            assert v.shape == ref.shape and v.dtype == ref.dtype, (name, k, v.dtype, ref.dtype)
            assert np.array_equal(v, ref), (name, k, float(np.max(np.abs(v - ref))))


def test_wpd_oracle_pinned_to_reference():
    """libs/wpe.py facted_wpd() run by the reference on complex64 STFTs (ref_wpd.npz)."""
    from oracle import stft_oracle as so
    from oracle import wpe_oracle as wo
    g = np.load(os.path.join(GOLD, "ref_wpd.npz"))
    for name in ("c3", "c4"):
        fl, hop, taps, delay, ctx, ci, wi = (int(v) for v in g[name + "/cfg"])
        mix = g[name + "/mix"]
        obs = np.stack([so.stft(mix[c], fl, hop, fl, window="hann", center=True, out_dtype=np.complex64)
                        for c in range(mix.shape[0])])
        x = np.ascontiguousarray(np.transpose(obs, (0, 2, 1)))                       # C x T x F
        for dt in (np.complex64, np.complex128):
            m, e = wo.facted_wpd(x, cgmm_iters=ci, wpd_iters=wi, taps=taps, delay=delay, context=ctx, dtype=dt)
            ea, _ = bo.align_phase(e.T, g[name + "/enh"].T)
            assert bo.rel_inf(ea, g[name + "/enh"].T) <= 5e-6, (name, dt)
            assert np.max(np.abs(m - g[name + "/tf_mask"])) <= 2e-5, (name, dt)
