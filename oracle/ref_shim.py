"""
oracle/ref_shim.py -- import the reference's OWN Python modules
(/root/reference/scripts/sptk/libs/{utils,beamformer,cluster,wpe}.py) in
this container, unmodified, under a small compatibility shim.

TEST INFRASTRUCTURE, BUILD-CONTAINER ONLY.  /root/reference does not exist on
the GPU box; nothing in tests marked gpu, smoke() or bench.py calls this.
It is used by oracle/make_golden.py (to generate tests/golden/*.npz and to
validate the restatement); the tests read only what that stored.

Why a shim is needed (SURVEY.md section 0 finding 2, Appendix C):
  * librosa / soundfile are not installed -> stub modules; librosa.stft/istft
    are served by oracle/stft_oracle.py (librosa 0.8.1 semantics), soundfile
    by scipy.io.wavfile with int16/32768 read and floor(y*32768) write;
  * numpy >= 1.24 removed np.complex / np.int (beamformer.py:49,297);
  * numpy >= 2 changed np.linalg.solve(a(F,N,N), b(F,N)) (beamformer.py:536);
  * scipy >= 1.13 removed scipy.signal.hann (utils.py:117,157).
The shim patches those names process-wide; call it only from test tooling.
"""
import importlib
import os
import sys
import types

import numpy as np

REFERENCE_SPTK = "/root/reference/scripts/sptk"


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_SPTK, "libs"))


def _install_stubs():
    from . import stft_oracle as so

    if "librosa" not in sys.modules:
        librosa = types.ModuleType("librosa")

        def _stft(y, n_fft=2048, hop_length=None, win_length=None,
                  window="hann", center=True, dtype=None, pad_mode="reflect"):
            win_length = n_fft if win_length is None else win_length
            hop_length = win_length // 4 if hop_length is None else hop_length
            out = np.complex64 if np.asarray(y).dtype == np.float32 \
                else np.complex128
            return so.stft(y, n_fft, hop_length, win_length, window=window,
                           center=center, out_dtype=out)

        def _istft(stft_matrix, hop_length=None, win_length=None,
                   window="hann", center=True, dtype=None, length=None):
            n_fft = 2 * (stft_matrix.shape[0] - 1)
            win_length = n_fft if win_length is None else win_length
            hop_length = win_length // 4 if hop_length is None else hop_length
            out = np.float32 if stft_matrix.dtype == np.complex64 \
                else np.float64
            return so.istft(stft_matrix, hop_length, win_length, window=window,
                            center=center, length=length, out_dtype=out)

        librosa.stft = _stft
        librosa.istft = _istft
        sys.modules["librosa"] = librosa

    if "soundfile" not in sys.modules:
        import scipy.io.wavfile as wavfile
        sf = types.ModuleType("soundfile")

        def _read(fname, start=0, stop=None, dtype="float32"):
            sr, data = wavfile.read(fname)
            data = data[start:stop]
            if dtype == "float32":
                data = so.float_from_pcm16(data)
            else:
                data = data.astype(dtype)
            return data, sr

        def _write(fname, samps, sr):
            samps = np.asarray(samps)
            if samps.dtype != np.int16:
                samps = so.pcm16_from_float(samps)
            wavfile.write(str(fname), sr, samps)

        sf.read = _read
        sf.write = _write
        sys.modules["soundfile"] = sf


_patched = False


def _patch_numpy_scipy():
    global _patched
    if _patched:
        return
    import scipy.signal
    if not hasattr(np, "complex"):
        np.complex = complex
    if not hasattr(np, "int"):
        np.int = int
    if not hasattr(np, "float"):
        np.float = float
    if not hasattr(scipy.signal, "hann"):
        scipy.signal.hann = scipy.signal.windows.hann
    _orig_solve = np.linalg.solve

    def _solve(a, b):
        a_ = np.asarray(a)
        b_ = np.asarray(b)
        if b_.ndim == a_.ndim - 1 and a_.ndim > 2:
            return _orig_solve(a_, b_[..., None])[..., 0]
        return _orig_solve(a, b)

    np.linalg.solve = _solve
    _patched = True


def load_reference():
    """
    Returns a namespace with the reference's modules:
      .utils .beamformer .cluster .wpe .spatial (and .data_handler if importable)
    """
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_SPTK}")
    _install_stubs()
    _patch_numpy_scipy()
    if REFERENCE_SPTK not in sys.path:
        sys.path.insert(0, REFERENCE_SPTK)
    ns = types.SimpleNamespace()
    ns.utils = importlib.import_module("libs.utils")
    ns.beamformer = importlib.import_module("libs.beamformer")
    ns.cluster = importlib.import_module("libs.cluster")
    try:
        ns.wpe = importlib.import_module("libs.wpe")
    except Exception:  # nara_wpe-free file, but keep optional
        ns.wpe = None
    try:
        ns.spatial = importlib.import_module("libs.spatial")
    except Exception:
        ns.spatial = None
    try:
        ns.data_handler = importlib.import_module("libs.data_handler")
    except Exception:
        ns.data_handler = None
    return ns
