"""Log-mel front-end on the B200: drop-in for ``nemo.collections.asr.modules.AudioToMelSpectrogramPreprocessor``
(modules/audio_preprocessing.py:100-280 -> parts/preprocessing/features.py:196-453) in inference.

Same constructor arguments, same buffers / ``state_dict`` keys (``featurizer.window`` (win_length),
``featurizer.fb`` (1, features, n_fft / 2 + 1)), same call
``preprocessor(input_signal=(B, L) float, length=(B,) int) -> (processed_signal (B, features, T), processed_length)``.
The arithmetic runs in two CUDA kernels of libcfb.so (csrc/frontend.cu, C ABI ``cfb_op_logmel``; ``cfb_op_logmel_raw``
for ``normalize=None`` / ``"None"``, the front end buffered inference builds); there is no CPU fallback.
Configurations no Conformer recipe uses are rejected at construction.
"""
from __future__ import annotations

import ctypes
import math
from collections import OrderedDict

import numpy as np
import torch
from torch import nn

from . import _lib


def slaney_mel_filters(sr: int, n_fft: int, n_mels: int, fmin: float = 0.0, fmax=None) -> np.ndarray:
    """What the reference obtains from ``librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax)`` (features.py:306-309;
    defaults htk=False, norm="slaney"): triangular filters on the Slaney mel scale, unit area, float32
    (n_mels, n_fft / 2 + 1).  A checkpoint's ``featurizer.fb`` buffer replaces it on ``load_state_dict``."""
    def hz_to_mel(f):
        f = np.asanyarray(f, dtype=np.float64)
        f_sp, min_log_hz, logstep = 200.0 / 3, 1000.0, math.log(6.4) / 27.0
        return np.where(f >= min_log_hz, min_log_hz / f_sp + np.log(np.maximum(f, 1e-30) / min_log_hz) / logstep, f / f_sp)

    def mel_to_hz(m):
        m = np.asanyarray(m, dtype=np.float64)
        f_sp, min_log_hz, logstep = 200.0 / 3, 1000.0, math.log(6.4) / 27.0
        return np.where(m >= min_log_hz / f_sp, min_log_hz * np.exp(logstep * (m - min_log_hz / f_sp)), f_sp * m)

    fmax = float(sr) / 2 if fmax is None else float(fmax)
    fftfreqs = np.linspace(0, float(sr) / 2, 1 + n_fft // 2)
    mel_f = mel_to_hz(np.linspace(hz_to_mel(fmin), hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = mel_f[:, None] - fftfreqs[None, :]
    w = np.zeros((n_mels, 1 + n_fft // 2), dtype=np.float32)
    for i in range(n_mels):
        w[i] = np.maximum(0, np.minimum(-ramps[i] / fdiff[i], ramps[i + 2] / fdiff[i + 1]))
    w *= (2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels]))[:, None]
    return w.astype(np.float32)


class _Featurizer(nn.Module):
    """Holds the two buffers under the reference's names (``featurizer.window``, ``featurizer.fb``)."""

    def __init__(self, window: torch.Tensor, fb: torch.Tensor):
        super().__init__()
        self.register_buffer("window", window)
        self.register_buffer("fb", fb)


class AudioToMelSpectrogramPreprocessor(nn.Module):
    _WINDOWS = {"hann": torch.hann_window, "hamming": torch.hamming_window, "blackman": torch.blackman_window,
                "bartlett": torch.bartlett_window}

    def __init__(self, sample_rate=16000, window_size=0.02, window_stride=0.01, n_window_size=None, n_window_stride=None,
                 window="hann", normalize="per_feature", n_fft=None, preemph=0.97, features=64, lowfreq=0, highfreq=None,
                 log=True, log_zero_guard_type="add", log_zero_guard_value=2 ** -24, dither=1e-5, pad_to=16,
                 frame_splicing=1, exact_pad=False, stft_exact_pad=False, stft_conv=False, pad_value=0, mag_power=2.0,
                 rng=None, nb_augmentation_prob=0.0, nb_max_freq=4000):
        super().__init__()
        self._sample_rate = sample_rate
        if window_size and n_window_size:  # audio_preprocessing.py:238-243
            raise ValueError(f"{self} received both window_size and n_window_size. Only one should be specified.")
        if window_stride and n_window_stride:
            raise ValueError(f"{self} received both window_stride and n_window_stride. Only one should be specified.")
        if window_size:
            n_window_size = int(window_size * sample_rate)
        if window_stride:
            n_window_stride = int(window_stride * sample_rate)
        if (n_window_size is None or n_window_stride is None or not isinstance(n_window_size, int)
                or not isinstance(n_window_stride, int) or n_window_size <= 0 or n_window_stride <= 0):
            raise ValueError(f"{self} got an invalid value for either n_window_size or n_window_stride. "  # features.py:246-258
                             "Both must be positive ints.")
        if log_zero_guard_type not in ["add", "clamp"]:  # features.py:320-325
            raise ValueError(f"{self} received {log_zero_guard_type} for the log_zero_guard_type parameter. "
                             "It must be either 'add' or 'clamp'.")
        self.win_length, self.hop_length = n_window_size, n_window_stride
        self.n_fft = n_fft or 2 ** math.ceil(math.log2(n_window_size))
        unsupported = []
        if self.n_fft != 512 or n_window_size > 512:
            unsupported.append(f"n_fft={self.n_fft} (the kernel is built for n_fft = 512)")
        if window not in self._WINDOWS:
            unsupported.append(f"window={window!r}")
        if normalize not in ("per_feature", None, "None"):
            unsupported.append(f"normalize={normalize!r}")
        if not log or log_zero_guard_type != "add" or isinstance(log_zero_guard_value, str):
            unsupported.append("log / log_zero_guard settings other than log(x + number)")
        if frame_splicing != 1 or exact_pad or stft_exact_pad or stft_conv or pad_value != 0 or mag_power != 2.0:
            unsupported.append("frame_splicing, exact_pad, stft_conv, pad_value != 0 or mag_power != 2")
        if features > 96:
            unsupported.append(f"features={features} > 96")
        if isinstance(pad_to, str):
            unsupported.append(f"pad_to={pad_to!r}")
        if unsupported:
            raise NotImplementedError("AudioToMelSpectrogramPreprocessor (B200) does not support: " + "; ".join(unsupported))
        self.normalize = None if normalize == "None" else normalize
        self.preemph = preemph
        self.log_zero_guard_value = float(log_zero_guard_value)
        self.dither = dither  # training-time noise only (features.py:367-368): inference ignores it
        self.pad_to = int(pad_to)
        self.nfilt = features
        fb = torch.from_numpy(slaney_mel_filters(sample_rate, self.n_fft, features, lowfreq, highfreq or sample_rate / 2))
        self.featurizer = _Featurizer(self._WINDOWS[window](n_window_size, periodic=False).float(), fb.unsqueeze(0))
        self._fb_km = None
        self._flag = None
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate())
        self.eval()

    # ---- reference surface
    @property
    def input_types(self):
        return OrderedDict({"input_signal": ("B", "T"), "length": ("B",)})

    @property
    def output_types(self):
        return OrderedDict({"processed_signal": ("B", "D", "T"), "processed_length": ("B",)})

    @property
    def filter_banks(self):
        return self.featurizer.fb

    def get_seq_len(self, seq_len: torch.Tensor) -> torch.Tensor:
        """features.py:347-353 (center = True)."""
        pad_amount = self.n_fft // 2 * 2
        return (torch.floor((seq_len.float() + pad_amount - self.n_fft) / self.hop_length) + 1).to(torch.long)

    def _invalidate(self):
        self._fb_km = None

    def _apply(self, fn, *a, **k):
        self._invalidate()
        return super()._apply(fn, *a, **k)

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("AudioToMelSpectrogramPreprocessor (B200) is inference-only (no dither / augmentation)")
        return super().train(False)

    @torch.no_grad()
    def forward(self, input_signal: torch.Tensor, length: torch.Tensor, check_lengths: bool = True):
        return self.get_features(input_signal, length, check_lengths)

    def get_features(self, input_signal, length, check_lengths: bool = True):
        if not input_signal.is_cuda:
            raise RuntimeError("AudioToMelSpectrogramPreprocessor (B200): input_signal must be a CUDA tensor (no CPU fallback)")
        if input_signal.dim() != 2:
            raise ValueError("input_signal must be (B, T)")
        lib = _lib.load_library()
        dev = input_signal.device
        x = input_signal.float().contiguous()
        lens = length.to(device=dev, dtype=torch.int64).contiguous()
        B, L = x.shape
        if self._fb_km is None or self._fb_km.device != dev:
            fb = self.featurizer.fb.detach().float().cpu().reshape(self.featurizer.fb.shape[-2], self.featurizer.fb.shape[-1])
            nz = fb != 0  # every filter is summed over its own span of FFT bins only
            first = torch.where(nz.any(1), nz.float().argmax(1), torch.zeros(fb.shape[0], dtype=torch.long))
            last = torch.where(nz.any(1), fb.shape[1] - 1 - nz.flip(1).float().argmax(1), -torch.ones(fb.shape[0], dtype=torch.long))
            self._fb_span = torch.stack([first, last - first + 1], 1).to(torch.int32).contiguous().to(dev)
            self._fb_km = fb.contiguous().to(dev)
            self._window = self.featurizer.window.to(dev, torch.float32).contiguous()
            self._flag = torch.zeros(1, dtype=torch.int32, device=dev)
        T = 1 + L // self.hop_length
        T_out = T if self.pad_to <= 0 or T % self.pad_to == 0 else T + self.pad_to - T % self.pad_to  # features.py:447-451
        out = torch.empty(B, self.nfilt, T_out, dtype=torch.float32, device=dev)
        seq_len = torch.empty(B, dtype=torch.int64, device=dev)
        vp = ctypes.c_void_p
        head = (vp(x.data_ptr()), vp(lens.data_ptr()), B, L, vp(self._window.data_ptr()), self.win_length, self.n_fft,
                self.hop_length, vp(self._fb_km.data_ptr()), vp(self._fb_span.data_ptr()), self.nfilt,
                float(self.preemph if self.preemph is not None else 0.0), self.log_zero_guard_value)
        stream = vp(torch.cuda.current_stream(dev).cuda_stream)
        if self.normalize is None:  # normalize_batch returns x unchanged: no statistics, nothing to check
            _lib.check(lib.cfb_op_logmel_raw(*head, vp(out.data_ptr()), T_out, vp(seq_len.data_ptr()), stream), None,
                       "cfb_op_logmel_raw")
            return out, seq_len
        rc = lib.cfb_op_logmel(*head, 1e-5, vp(out.data_ptr()), T_out, vp(seq_len.data_ptr()), vp(self._flag.data_ptr()), stream)
        _lib.check(rc, None, "cfb_op_logmel")
        if check_lengths and int(self._flag.item()):  # one device read-back; pass check_lengths=False to stay asynchronous
            raise ValueError("normalize_batch with `per_feature` normalize_type received a tensor of length 1. This will "
                             "result in torch.std() returning nan")  # features.py:58-62
        return out, seq_len
