"""
setk_b200.plan -- Python handle on a libsetk_b200 STFT plan plus the plan-free
entry points, operating on torch tensors (device memory, streams) and calling
the CUDA kernels through the C-ABI.  PyTorch is plumbing here: it owns the
buffers and the stream; every arithmetic step is a kernel of libsetk_b200.

Layouts are the reference's (scripts/sptk/libs): audio (B,C,N) f32, mask
(B,T,F) f32, stft (B,C,F,T) c64, R (B,F,C,C), weight (B,F,C), enhanced
(B,F,T) c64, wave (B,N_out) f32.
"""
import ctypes
import math

import numpy as np
import scipy.signal
import torch

from . import _lib

EPSILON = float(np.finfo(np.float32).eps)  # libs/utils.py:16


def nextpow2(window_size):
    """libs/utils.py:25-27"""
    return 2**math.ceil(math.log2(window_size))


def make_window(window, frame_len):
    """
    Analysis window, float64, length frame_len: librosa's
    get_window(window, frame_len, fftbins=True); "sqrthann" as in
    libs/utils.py:116-117.
    """
    if isinstance(window, str):
        if window == "sqrthann":
            return scipy.signal.get_window("hann", frame_len, fftbins=True)**0.5
        return scipy.signal.get_window(window, frame_len, fftbins=True)
    if isinstance(window, torch.Tensor):
        window = window.detach().cpu().numpy()
    window = np.ascontiguousarray(window, dtype=np.float64)
    if window.shape != (frame_len,):
        raise ValueError(f"Window size mismatch: {window.shape} vs {frame_len}")
    return window


def _dtype_code(t):
    if t.dtype == torch.complex64:
        return _lib.C64
    if t.dtype == torch.complex128:
        return _lib.C128
    raise TypeError(f"expected a complex64/complex128 tensor, got {t.dtype}")


def _f32(t, device):
    t = torch.as_tensor(t, device=device)
    if t.dtype != torch.float32:
        t = t.to(torch.float32)
    return t.contiguous()


class StftPlan(object):
    """
    One STFT geometry (mirrors StftParser, libs/opts.py:21-49, and the keyword
    arguments of forward_stft / inverse_stft, libs/utils.py:96-105,142-150).
    """

    def __init__(self, num_channels, frame_len=512, frame_hop=256, center=True,
                 round_power_of_two=True, window="hann", max_batch=1,
                 max_samples=160000, device=None):
        self.device = torch.device(device if device is not None else (
            "cuda" if torch.cuda.is_available() else "cpu"))
        if self.device.type != "cuda" and not _lib.emulated():
            raise RuntimeError("StftPlan needs a CUDA device (setk_b200 has no CPU fallback)")
        self.num_channels = int(num_channels)
        self.frame_len = int(frame_len)
        self.frame_hop = int(frame_hop)
        self.center = bool(center)
        self.n_fft = nextpow2(frame_len) if round_power_of_two else int(frame_len)
        self.num_bins = self.n_fft // 2 + 1
        self.max_batch = int(max_batch)
        self.max_samples = int(max_samples)
        win = make_window(window, self.frame_len)
        self._win = np.ascontiguousarray(win, dtype=np.float64)
        cfg = _lib.SetkConfig(
            num_channels=self.num_channels, frame_len=self.frame_len,
            n_fft=self.n_fft, frame_hop=self.frame_hop, center=int(self.center),
            max_batch=self.max_batch, max_samples=self.max_samples, reserved=0,
            window_host=self._win.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
        handle = ctypes.c_void_p()
        # the handle belongs to the library that made it: close() must not hand it to another one
        # bound later by use_library() (its memory may be device memory the other cannot free)
        self._cdll = _lib.library()
        with self._device_ctx():
            _lib.check(self._cdll.setk_plan_create(ctypes.byref(cfg), ctypes.byref(handle)))
        self._h = handle

    # ------------------------------------------------------------------ misc
    def _device_ctx(self):
        if self.device.type == "cuda":
            return torch.cuda.device(self.device)
        import contextlib
        return contextlib.nullcontext()

    def close(self):
        if getattr(self, "_h", None):
            try:
                with self._device_ctx():
                    self._cdll.setk_plan_destroy(self._h)
            finally:
                self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def num_frames(self, nsamps):
        T = _lib.library().setk_num_frames(self._h, int(nsamps))
        if T < 1:
            raise ValueError(f"{nsamps} samples are too short for n_fft={self.n_fft}")
        return T

    def istft_length(self, num_frames):
        return _lib.library().setk_istft_length(self._h, int(num_frames))

    def _stream(self):
        return _lib.current_stream(self.device)

    def _check_audio(self, audio):
        audio = _f32(audio, self.device)
        if audio.dim() != 3 or audio.shape[1] != self.num_channels:
            raise ValueError(f"audio must be (B, {self.num_channels}, N), got {tuple(audio.shape)}")
        return audio

    def _nsamp(self, n_samples, B):
        if n_samples is None:
            return None
        ns = torch.as_tensor(n_samples, device=self.device).to(torch.int32).contiguous()
        if ns.shape != (B,):
            raise ValueError(f"n_samples must have shape ({B},)")
        return ns

    # --------------------------------------------------------------- kernels
    def stft(self, audio, n_samples=None):
        """audio (B,C,N) -> (B,C,F,T) complex64.  forward_stft per channel."""
        audio = self._check_audio(audio)
        B, C, N = audio.shape
        T = self.num_frames(N)
        ns = self._nsamp(n_samples, B)
        out = torch.empty((B, C, self.num_bins, T), dtype=torch.complex64, device=self.device)
        with self._device_ctx():
            _lib.check(_lib.library().setk_stft(self._h, _lib.ptr(audio), _lib.ptr(ns), B, N,
                                                _lib.ptr(out), self._stream()))
        return out

    def stft_cov(self, audio, mask_s, mask_n=None, n_samples=None, clip_mask=False,
                 mask_ft=False, want_maxabs=True):
        """
        Fused STFT + mask-weighted covariance.  Returns (Rs, Rn, maxabs):
        Rs, Rn (B,F,C,C) complex64; maxabs (B,) float32 or None.
        """
        audio = self._check_audio(audio)
        B, C, N = audio.shape
        T = self.num_frames(N)
        F = self.num_bins
        mshape = (B, F, T) if mask_ft else (B, T, F)
        mask_s = _f32(mask_s, self.device)
        if tuple(mask_s.shape) != mshape:
            raise ValueError(f"mask must be {mshape}, got {tuple(mask_s.shape)}")
        if mask_n is not None:
            mask_n = _f32(mask_n, self.device)
            if tuple(mask_n.shape) != mshape:
                raise ValueError(f"mask_n must be {mshape}, got {tuple(mask_n.shape)}")
        ns = self._nsamp(n_samples, B)
        Rs = torch.empty((B, F, C, C), dtype=torch.complex64, device=self.device)
        Rn = torch.empty_like(Rs)
        maxabs = torch.empty((B,), dtype=torch.float32, device=self.device) if want_maxabs else None
        flags = (_lib.F_CLIP_MASK if clip_mask else 0) | (_lib.F_MASK_FT if mask_ft else 0)
        with self._device_ctx():
            _lib.check(_lib.library().setk_stft_cov(
                self._h, _lib.ptr(audio), _lib.ptr(ns), B, N, _lib.ptr(mask_s), _lib.ptr(mask_n),
                flags, _lib.ptr(Rs), _lib.ptr(Rn), _lib.ptr(maxabs), self._stream()))
        return Rs, Rn, maxabs

    def cgmm_masks(self, audio, num_classes=2, num_iters=20, init_gamma=None, update_alpha=False,
                   n_samples=None):
        """
        CGMM mask estimation from audio (STFT + CgmmTrainer(...).train(num_iters),
        cluster.py:396-465).  init_gamma (B,K,T,F) or None (2 classes only).
        Returns (masks (B,K,T,F) float32, status (B,) int32).
        """
        audio = self._check_audio(audio)
        B, C, N = audio.shape
        T = self.num_frames(N)
        F = self.num_bins
        K = int(num_classes)
        if init_gamma is not None:
            init_gamma = _f32(init_gamma, self.device)
            if tuple(init_gamma.shape) != (B, K, T, F):
                raise ValueError(f"init_gamma must be {(B, K, T, F)}, got {tuple(init_gamma.shape)}")
        ns = self._nsamp(n_samples, B)
        masks = torch.empty((B, K, T, F), dtype=torch.float32, device=self.device)
        status = torch.zeros((B,), dtype=torch.int32, device=self.device)
        with self._device_ctx():
            _lib.check(_lib.library().setk_cgmm_masks(
                self._h, _lib.ptr(audio), _lib.ptr(ns), B, N, K, int(num_iters), _lib.ptr(init_gamma),
                1 if update_alpha else 0, _lib.ptr(masks), _lib.ptr(status), self._stream()))
        return masks, status

    def istft(self, enh, n_out=None, norm=None):
        """enh (B,F,T) complex64 -> wave (B,n_out) float32 (inverse_stft)."""
        enh = torch.as_tensor(enh, device=self.device)
        if enh.dtype != torch.complex64:
            enh = enh.to(torch.complex64)
        enh = enh.contiguous()
        if enh.dim() != 3 or enh.shape[1] != self.num_bins:
            raise ValueError(f"enh must be (B, {self.num_bins}, T), got {tuple(enh.shape)}")
        B, F, T = enh.shape
        if n_out is None:
            n_out = self.istft_length(T)
        norm_t = None if norm is None else _f32(norm, self.device).reshape(B)
        wave = torch.empty((B, int(n_out)), dtype=torch.float32, device=self.device)
        with self._device_ctx():
            _lib.check(_lib.library().setk_istft(self._h, _lib.ptr(enh), B, T, int(n_out),
                                                 _lib.ptr(norm_t), _lib.ptr(wave), self._stream()))
        return wave

    def apply_istft(self, audio, weight, post_mask=None, n_out=None, norm=None, n_samples=None,
                    pcm16=False):
        """Fused beamform + iSTFT from audio.  weight (B,F,C) complex.
        pcm16=True: the `norm` rescale pass writes what WaveWriter would put in the wav file
        (int16 = floor(y * 32768) clipped, utils.py:45-62) instead of float32."""
        audio = self._check_audio(audio)
        B, C, N = audio.shape
        T = self.num_frames(N)
        weight = torch.as_tensor(weight, device=self.device).contiguous()
        if tuple(weight.shape) != (B, self.num_bins, C):
            raise ValueError(f"weight must be {(B, self.num_bins, C)}, got {tuple(weight.shape)}")
        if post_mask is not None:
            post_mask = _f32(post_mask, self.device)
            if tuple(post_mask.shape) != (B, T, self.num_bins):
                raise ValueError("post_mask must be (B, T, F)")
        if n_out is None:
            n_out = self.istft_length(T)
        norm_t = None if norm is None else _f32(norm, self.device).reshape(B)
        ns = self._nsamp(n_samples, B)
        wave = torch.empty((B, int(n_out)), dtype=torch.int16 if pcm16 else torch.float32,
                           device=self.device)
        fn = _lib.library().setk_apply_istft_pcm16 if pcm16 else _lib.library().setk_apply_istft
        with self._device_ctx():
            _lib.check(fn(
                self._h, _lib.ptr(audio), _lib.ptr(ns), B, N, _lib.ptr(weight), _dtype_code(weight),
                _lib.ptr(post_mask), int(n_out), _lib.ptr(norm_t), _lib.ptr(wave), self._stream()))
        return wave


# ---------------------------------------------------------------- plan-free ---
def _ctx(device):
    if device.type == "cuda":
        return torch.cuda.device(device)
    import contextlib
    return contextlib.nullcontext()


def cgmm_from_stft(stft, num_classes=2, num_iters=20, init_gamma=None, update_alpha=False):
    """
    CgmmTrainer(obs, K, gamma, update_alpha).train(num_iters) batched (cluster.py:396-465).
    stft (B,C,F,T) complex64; init_gamma (B,K,T,F) or None (2 classes only).
    Returns (masks (B,K,T,F) float32, status (B,) int32).
    """
    stft = stft.contiguous()
    if stft.dtype != torch.complex64:
        stft = stft.to(torch.complex64)
    if stft.dim() != 4:
        raise ValueError(f"stft must be (B, C, F, T), got {tuple(stft.shape)}")
    B, C, F, T = stft.shape
    K = int(num_classes)
    if init_gamma is not None:
        init_gamma = _f32(init_gamma, stft.device)
        if tuple(init_gamma.shape) != (B, K, T, F):
            raise ValueError(f"init_gamma must be {(B, K, T, F)}, got {tuple(init_gamma.shape)}")
    masks = torch.empty((B, K, T, F), dtype=torch.float32, device=stft.device)
    status = torch.zeros((B,), dtype=torch.int32, device=stft.device)
    with _ctx(stft.device):
        _lib.check(_lib.library().setk_cgmm_stft(
            _lib.ptr(stft), B, C, F, T, K, int(num_iters), _lib.ptr(init_gamma), 1 if update_alpha else 0,
            _lib.ptr(masks), _lib.ptr(status), _lib.current_stream(stft.device)))
    return masks, status


def wpe_from_stft(stft, taps=10, delay=3, context=1, num_iters=3):
    """
    wpe(reverb, taps, delay, context, num_iters) batched (libs/wpe.py:82-110).
    stft (B,C,F,T) complex64 -> (dereverberated (B,C,F,T) complex64, status (B,) int32).
    """
    stft = stft.contiguous()
    if stft.dtype != torch.complex64:
        stft = stft.to(torch.complex64)
    if stft.dim() != 4:
        raise ValueError(f"stft must be (B, C, F, T), got {tuple(stft.shape)}")
    B, C, F, T = stft.shape
    out = torch.empty_like(stft)
    status = torch.zeros((B,), dtype=torch.int32, device=stft.device)
    with _ctx(stft.device):
        _lib.check(_lib.library().setk_wpe_stft(
            _lib.ptr(stft), B, C, F, T, int(taps), int(delay), int(context), int(num_iters),
            _lib.ptr(out), _lib.ptr(status), _lib.current_stream(stft.device)))
    return out, status


def wpe_step(stft, lambda_enh=None, taps=10, delay=3, context=1, want_inv_lambda=True):
    """
    One WPE step with the variance of facted_wpd (libs/wpe.py:147-155): stft (B,C,F,T) complex64,
    lambda_enh (B,F,T) complex64 or None (first iteration: compute_lambda of the observations).
    Returns (dereverberated (B,C,F,T) complex64, 1/lambda (B,T,F) float32 or None, status (B,) int32).
    """
    stft = stft.contiguous()
    if stft.dtype != torch.complex64:
        stft = stft.to(torch.complex64)
    if stft.dim() != 4:
        raise ValueError(f"stft must be (B, C, F, T), got {tuple(stft.shape)}")
    B, C, F, T = stft.shape
    if lambda_enh is not None:
        lambda_enh = torch.as_tensor(lambda_enh, device=stft.device).to(torch.complex64).contiguous()
        if tuple(lambda_enh.shape) != (B, F, T):
            raise ValueError(f"lambda_enh must be {(B, F, T)}, got {tuple(lambda_enh.shape)}")
    out = torch.empty_like(stft)
    inv = torch.empty((B, T, F), dtype=torch.float32, device=stft.device) if want_inv_lambda else None
    status = torch.zeros((B,), dtype=torch.int32, device=stft.device)
    with _ctx(stft.device):
        _lib.check(_lib.library().setk_wpe_step(
            _lib.ptr(stft), _lib.ptr(lambda_enh), B, C, F, T, int(taps), int(delay), int(context),
            _lib.ptr(out), _lib.ptr(inv), _lib.ptr(status), _lib.current_stream(stft.device)))
    return out, inv, status


def covariance(stft, mask, clip_mask=False, mask_ft=False):
    """compute_covar batched: stft (B,C,F,T) c64, mask (B,T,F) -> (B,F,C,C) c64."""
    stft = stft.contiguous()
    if stft.dtype != torch.complex64:
        stft = stft.to(torch.complex64)
    B, C, F, T = stft.shape
    mask = _f32(mask, stft.device)
    R = torch.empty((B, F, C, C), dtype=torch.complex64, device=stft.device)
    flags = (_lib.F_CLIP_MASK if clip_mask else 0) | (_lib.F_MASK_FT if mask_ft else 0)
    with _ctx(stft.device):
        _lib.check(_lib.library().setk_cov(_lib.ptr(stft), _lib.ptr(mask), flags, B, C, F, T,
                                           _lib.ptr(R), _lib.current_stream(stft.device)))
    return R


def weights(kind, Rs, Rn=None, Ry=None, beta=0.0, ref_channel=-1, rank1=_lib.RANK1_NONE,
            ban=False, out_dtype=None):
    """
    Per-bin weight solve.  Rs/Rn/Ry (B,F,C,C) complex64|complex128 (same dtype).
    Returns (w (B,F,C), status (B,) int32 tensor, ref_used (B,) int32 tensor).
    """
    Rs = Rs.contiguous()
    B, F, C, _ = Rs.shape
    dt = _dtype_code(Rs)
    for m in (Rn, Ry):
        if m is not None and (m.dtype != Rs.dtype or m.shape != Rs.shape):
            raise ValueError("Rs / Rn / Ry must share dtype and shape")
    Rn = None if Rn is None else Rn.contiguous()
    Ry = None if Ry is None else Ry.contiguous()
    out_dtype = Rs.dtype if out_dtype is None else out_dtype
    w = torch.empty((B, F, C), dtype=out_dtype, device=Rs.device)
    status = torch.zeros((B,), dtype=torch.int32, device=Rs.device)
    ref_used = torch.full((B,), -1, dtype=torch.int32, device=Rs.device)
    with _ctx(Rs.device):
        _lib.check(_lib.library().setk_weights(
            int(kind), float(beta), int(ref_channel), int(rank1), int(bool(ban)), _lib.ptr(Rs),
            _lib.ptr(Rn), _lib.ptr(Ry), dt, B, F, C, _lib.ptr(w), _dtype_code(w), _lib.ptr(status),
            _lib.ptr(ref_used), _lib.current_stream(Rs.device)))
    return w, status, ref_used


def ban(weight, Rn):
    """do_ban batched: weight (B,F,C), Rn (B,F,C,C), same complex dtype."""
    Rn = Rn.contiguous()
    weight = weight.to(Rn.dtype).contiguous()
    B, F, C = weight.shape
    out = torch.empty_like(weight)
    with _ctx(Rn.device):
        _lib.check(_lib.library().setk_ban(_lib.ptr(weight), _lib.ptr(Rn), _dtype_code(Rn), B, F, C,
                                           _lib.ptr(out), _lib.current_stream(Rn.device)))
    return out


def rank1(Rs, Rn=None):
    """rank1_constraint batched.  Returns (R1 (B,F,C,C), status (B,))."""
    Rs = Rs.contiguous()
    B, F, C, _ = Rs.shape
    Rn = None if Rn is None else Rn.to(Rs.dtype).contiguous()
    out = torch.empty_like(Rs)
    status = torch.zeros((B,), dtype=torch.int32, device=Rs.device)
    with _ctx(Rs.device):
        _lib.check(_lib.library().setk_rank1(_lib.ptr(Rs), _lib.ptr(Rn), _dtype_code(Rs), B, F, C,
                                             _lib.ptr(out), _lib.ptr(status),
                                             _lib.current_stream(Rs.device)))
    return out, status


def apply_weights(stft, weight, post_mask=None):
    """Beamformer.beamform batched: (B,C,F,T) x (B,F,C) -> (B,F,T) complex64."""
    stft = stft.contiguous()
    if stft.dtype != torch.complex64:
        stft = stft.to(torch.complex64)
    B, C, F, T = stft.shape
    weight = weight.contiguous()
    if post_mask is not None:
        post_mask = _f32(post_mask, stft.device)
    enh = torch.empty((B, F, T), dtype=torch.complex64, device=stft.device)
    with _ctx(stft.device):
        _lib.check(_lib.library().setk_apply(_lib.ptr(stft), _lib.ptr(weight), _dtype_code(weight),
                                             _lib.ptr(post_mask), B, C, F, T, _lib.ptr(enh),
                                             _lib.current_stream(stft.device)))
    return enh


def float_to_pcm16(wave):
    wave = wave.contiguous()
    pcm = torch.empty(wave.shape, dtype=torch.int16, device=wave.device)
    with _ctx(wave.device):
        _lib.check(_lib.library().setk_float_to_pcm16(_lib.ptr(wave), wave.numel(), _lib.ptr(pcm),
                                                      _lib.current_stream(wave.device)))
    return pcm


def pcm16_to_float(pcm):
    pcm = pcm.contiguous()
    wave = torch.empty(pcm.shape, dtype=torch.float32, device=pcm.device)
    with _ctx(pcm.device):
        _lib.check(_lib.library().setk_pcm16_to_float(_lib.ptr(pcm), pcm.numel(), _lib.ptr(wave),
                                                      _lib.current_stream(pcm.device)))
    return wave


def cm_masks(blobs, T, F, out=None):
    """
    Kaldi "CM" compressed matrices -> float32 masks [B][T][F] on the device (kaldi_io.py:248-281).
    blobs: uint8 [B][slot_bytes] device tensor, one matrix per slot as it lies in the archive behind
    the "CM " token (slot_bytes a multiple of 16).  Returns (masks, status int32 [B]).
    """
    if blobs.dtype != torch.uint8 or blobs.dim() != 2:
        raise ValueError("cm_masks: blobs must be uint8 [B][slot_bytes]")
    blobs = blobs.contiguous()
    B = blobs.shape[0]
    if out is None:
        out = torch.empty((B, T, F), dtype=torch.float32, device=blobs.device)
    status = torch.zeros((B,), dtype=torch.int32, device=blobs.device)
    with _ctx(blobs.device):
        _lib.check(_lib.library().setk_cm_masks(_lib.ptr(blobs), blobs.shape[1], B, T, F, _lib.ptr(out),
                                                _lib.ptr(status), _lib.current_stream(blobs.device)))
    return out, status


# ---------------------------------------------------------------------------
# spatial features on explicit STFTs (libs/spatial.py of the reference; csrc/spatial.cu)
# ---------------------------------------------------------------------------
def _c64(t, device=None):
    t = torch.as_tensor(t) if device is None else torch.as_tensor(t, device=device)
    if t.dtype != torch.complex64:
        t = t.to(torch.complex64)
    return t.contiguous()


def ipd(si, sj, mode=0):
    """spatial.ipd: si, sj (..., T, F) complex64 -> float32 (..., T, F) (mode 0/1) or (..., T, 2F)."""
    si, sj = _c64(si), _c64(sj, si.device if torch.is_tensor(si) else None)
    if si.shape != sj.shape or si.dim() < 2:
        raise ValueError(f"ipd: shapes {tuple(si.shape)} / {tuple(sj.shape)}")
    F = si.shape[-1]
    rows = si.numel() // F
    shape = list(si.shape)
    if mode == 2:
        shape[-1] = 2 * F
    out = torch.empty(shape, dtype=torch.float32, device=si.device)
    with _ctx(si.device):
        _lib.check(_lib.library().setk_ipd(_lib.ptr(si), _lib.ptr(sj), rows, F, int(mode),
                                           _lib.ptr(out), _lib.current_stream(si.device)))
    return out


def directional_feats(stft, steer, pairs=None):
    """
    spatial.directional_feats batched: stft (B,M,F,T) complex64, steer (M,F) or (B,M,F)
    complex -> (B,T,F) float64.  pairs: list of (i, j) or None (all i < j).
    """
    stft = _c64(stft)
    if stft.dim() != 4:
        raise ValueError(f"stft must be (B, M, F, T), got {tuple(stft.shape)}")
    B, M, F, T = stft.shape
    steer = torch.as_tensor(steer, device=stft.device).to(torch.complex128).contiguous()
    batched = steer.dim() == 3
    if tuple(steer.shape[-2:]) != (M, F) or (batched and steer.shape[0] != B):
        raise ValueError(f"steer vector must be ({M}, {F}) or ({B}, {M}, {F}), got {tuple(steer.shape)}")
    p_t, n_pairs = None, 0
    if pairs is not None:
        p_t = torch.as_tensor(pairs, dtype=torch.int32, device=stft.device).reshape(-1, 2).contiguous()
        n_pairs = p_t.shape[0]
        if n_pairs == 0 or int(p_t.min()) < 0 or int(p_t.max()) >= M:
            raise ValueError(f"df_pair entries must lie in [0, {M})")
    out = torch.empty((B, T, F), dtype=torch.float64, device=stft.device)
    with _ctx(stft.device):
        _lib.check(_lib.library().setk_directional_feats(
            _lib.ptr(stft), _lib.ptr(steer), int(batched), _lib.ptr(p_t), n_pairs, B, M, F, T,
            _lib.ptr(out), _lib.current_stream(stft.device)))
    return out


def gcc_phat(si, sj, omega, tau, normalize=True, apply_floor=True, out=None):
    """
    One microphone pair of gcc_phat_linear / gcc_phat_diag: si, sj (T,F) complex64, omega (F,)
    and tau (D,) float64 -> (T,D) float64.  With `out` given the pair is ADDED to it
    (srp_phat_linear).
    """
    si = _c64(si)
    sj = _c64(sj, si.device)
    if si.dim() != 2 or si.shape != sj.shape:
        raise ValueError(f"gcc_phat: si/sj must be (T, F), got {tuple(si.shape)} / {tuple(sj.shape)}")
    T, F = si.shape
    omega = torch.as_tensor(omega, dtype=torch.float64, device=si.device).contiguous()
    tau = torch.as_tensor(tau, dtype=torch.float64, device=si.device).contiguous()
    if omega.numel() != F:
        raise ValueError(f"gcc_phat: {omega.numel()} frequencies for {F} bins")
    D = tau.numel()
    lib = _lib.library()
    work = torch.empty((int(lib.setk_gcc_phat_work_doubles(T, F, D)),), dtype=torch.float64,
                       device=si.device)
    accumulate = out is not None
    if out is None:
        out = torch.empty((T, D), dtype=torch.float64, device=si.device)
    with _ctx(si.device):
        _lib.check(lib.setk_gcc_phat(_lib.ptr(si), _lib.ptr(sj), T, F, _lib.ptr(omega), _lib.ptr(tau), D,
                                     int(bool(normalize)), int(bool(apply_floor)), int(accumulate),
                                     _lib.ptr(work), _lib.ptr(out), _lib.current_stream(si.device)))
    return out


def msc(spec, context=1, normalize=True):
    """spatial.msc: spec (N,T,F) complex64 -> (T,F) float64."""
    spec = _c64(spec)
    if spec.dim() != 3:
        raise ValueError(f"msc: spectrogram must be (N, T, F), got {tuple(spec.shape)}")
    N, T, F = spec.shape
    lib = _lib.library()
    work = torch.empty((int(lib.setk_msc_work_doubles(T, F)),), dtype=torch.float64, device=spec.device)
    out = torch.empty((T, F), dtype=torch.float64, device=spec.device)
    with _ctx(spec.device):
        _lib.check(lib.setk_msc(_lib.ptr(spec), N, T, F, int(context), int(bool(normalize)),
                                _lib.ptr(work), _lib.ptr(out), _lib.current_stream(spec.device)))
    return out
