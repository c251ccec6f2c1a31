"""Thin torch-tensor front of the C ABI: one :class:`Engine` per GPU.

PyTorch is plumbing here (device memory, the current CUDA stream); every
computation is a kernel of ``libtaco_b200.so``.  Methods mirror the stage-level
entry points of ``include/taco_b200.h`` and are what the parity tests call.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _abi
from .hparams import HParams
from .weights import canonicalize


def pad_inputs(seqs, pad: int = 0) -> np.ndarray:
    """Batch of id sequences padded with ``pad`` to the longest one: the layout the reference feeder hands to
    ``Tacotron.initialize`` (reference ``datasets/datafeeder_npy.py:174-176,184-185``)."""
    n = max(len(x) for x in seqs)
    return np.stack([np.pad(np.asarray(x), (0, n - len(x)), mode="constant", constant_values=pad) for x in seqs])


def pad_targets(targets, outputs_per_step: int, pad: float = 0.0) -> np.ndarray:
    """Teacher-forcing targets ``[T_i, C]`` padded with ``pad`` to ``max(T_i) + 1`` rounded up to a multiple of
    ``outputs_per_step`` (reference ``datasets/datafeeder_npy.py:179-181,188-195``)."""
    n = max(len(t) for t in targets) + 1
    n = -(-n // outputs_per_step) * outputs_per_step
    return np.stack([np.pad(np.asarray(t), [(0, n - len(t)), (0, 0)], mode="constant", constant_values=pad)
                     for t in targets])


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class Engine:
    """Owns a ``taco_handle`` on one CUDA device."""

    def __init__(self, hp: HParams, id_num: int = 0, device: int | torch.device | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("tacotron_multispeaker_b200 needs a CUDA device (B200, sm_100a); "
                               "there is no CPU fallback")
        self.lib = _abi.load()
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        self.hp = hp.copy()
        self.id_num = int(id_num)
        chp = _abi.TacoHParams(hp.num_mels, hp.num_freq, hp.outputs_per_step, hp.max_iters,
                               hp.embedding_text_channels, hp.embedding_id_channels,
                               hp.num_symbols, self.id_num)
        self._h = C.c_void_p()
        rc = self.lib.taco_create(C.byref(chp), self.device.index or 0, C.byref(self._h))
        if rc != _abi.TACO_OK:
            raise _abi.TacoError(rc, "taco_create failed (not an sm_100 GPU, or bad hparams)")
        self._finalized = False

    # ---- lifetime ----
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.taco_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self) -> int:
        """The ``taco_handle*`` as an integer (first argument of the ``torch.ops.taco_b200`` operators)."""
        return int(self._h.value or 0)

    def _ck(self, rc):
        _abi.check(self.lib, self._h, rc)

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- weights ----
    def weight_names(self):
        n = self.lib.taco_num_weights(self._h)
        return [self.lib.taco_weight_name(self._h, i).decode() for i in range(n)]

    def load_weights(self, weights: Dict[str, np.ndarray]):
        """Variables keyed by TF checkpoint names (see weights.py)."""
        canon = canonicalize(weights, self.hp, self.id_num)
        for name, arr in canon.items():
            a = np.ascontiguousarray(arr, dtype=np.float32)
            shape = (C.c_int64 * a.ndim)(*a.shape)
            self._ck(self.lib.taco_set_weight(self._h, name.encode(), a.ctypes.data_as(C.c_void_p),
                                              shape, a.ndim))
        with torch.cuda.device(self.device):
            self._ck(self.lib.taco_finalize_weights(self._h))
        self._finalized = True

    # ---- helpers ----
    def _i32(self, x) -> Optional[torch.Tensor]:
        if x is None:
            return None
        t = torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x)
        return t.to(device=self.device, dtype=torch.int32).contiguous()

    def _f32(self, x) -> Optional[torch.Tensor]:
        if x is None:
            return None
        t = torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x)
        return t.to(device=self.device, dtype=torch.float32).contiguous()

    def max_steps(self, teacher_force: bool, T_tgt: int = 0) -> int:
        return int(self.lib.taco_max_steps(self._h, int(teacher_force), int(T_tgt)))

    def decoder_geometry(self, N: int):
        cs, s, nc = C.c_int(), C.c_int(), C.c_int()
        self._ck(self.lib.taco_decoder_geometry(self._h, N, C.byref(cs), C.byref(s), C.byref(nc)))
        return dict(cluster_size=cs.value, samples_per_cluster=s.value, num_clusters=nc.value)

    def launch_count(self) -> int:
        return int(self.lib.taco_launch_count(self._h))

    def set_gemm_mode(self, mode: int):
        """1 = bf16x3 tcgen05 (default, fp32-class), 2 = plain bf16 tcgen05; any other mode raises TacoError."""
        self._ck(self.lib.taco_set_gemm_mode(self._h, int(mode)))

    def set_decoder_clusters(self, n: int):
        """0 = default geometry (fewest clusters within 20 % of the shortest decode: batch 32 -> 4 clusters of 8);
        n > 0 = n clusters of <= 8 utterances."""
        self._ck(self.lib.taco_set_decoder_clusters(self._h, int(n)))

    def set_cuda_graphs(self, on: bool):
        """``taco_set_cuda_graphs``: capture / replay of the forward's launches (default on; needs a non-default stream)."""
        self._ck(self.lib.taco_set_cuda_graphs(self._h, int(on)))

    def set_profiling(self, on: bool):
        self._ck(self.lib.taco_set_profiling(self._h, int(on)))

    def last_stage_ms(self):
        buf = (C.c_float * 4)()
        self._ck(self.lib.taco_last_stage_ms(self._h, buf))
        return dict(encoder=buf[0], decoder=buf[1], postnet=buf[2], decoder_kernel=buf[3])

    def check_ids(self):
        self._ck(self.lib.taco_check_ids(self._h, self.stream))

    # ---- stages ----
    def embed(self, ids, spk=None):
        ids = self._i32(ids)
        spk = self._i32(spk) if (spk is not None and self.id_num > 1) else None
        N, T = ids.shape
        width = self.hp.embedding_text_channels + (self.hp.embedding_id_channels if spk is not None else 0)
        out = torch.empty(N, T, width, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_embed(self._h, _ptr(ids), _ptr(spk), N, T, _ptr(out), self.stream))
        return out

    def encoder(self, ids, lengths, spk=None, bn_mode=_abi.BN_MOVING):
        ids, lengths = self._i32(ids), self._i32(lengths)
        spk = self._i32(spk) if (spk is not None and self.id_num > 1) else None
        N, T = ids.shape
        out = torch.empty(N, T, 256, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_encoder(self._h, _ptr(ids), _ptr(lengths), _ptr(spk), N, T, bn_mode,
                                       _ptr(out), self.stream))
        return out

    def decode(self, memory, mel_targets=None, teacher_force=False, want_alignments=True):
        memory = self._f32(memory)
        N, T_in, _ = memory.shape
        tg = self._f32(mel_targets) if teacher_force else None
        T_tgt = tg.shape[1] if tg is not None else 0
        ms = self.max_steps(teacher_force, T_tgt)
        D = self.hp.num_mels * self.hp.outputs_per_step
        dec = torch.zeros(N, ms, D, device=self.device, dtype=torch.float32)
        al = torch.zeros(N, T_in, ms, device=self.device, dtype=torch.float32) if want_alignments else None
        steps = C.c_int32(0)
        self._ck(self.lib.taco_decode(self._h, _ptr(memory), N, T_in, _ptr(tg), T_tgt, int(teacher_force),
                                      _ptr(dec), _ptr(al), C.byref(steps), self.stream))
        s = steps.value
        return dec[:, :s], (al[:, :, :s] if al is not None else None), s

    def cbhg(self, which, x, lengths=None, bn_mode=_abi.BN_MOVING):
        x = self._f32(x)
        lengths = self._i32(lengths)
        N, T, _ = x.shape
        out = torch.empty(N, T, 256, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_cbhg(self._h, which, _ptr(x), _ptr(lengths), N, T, bn_mode, 0, _ptr(out),
                                    self.stream))
        return out

    def postnet(self, mel, bn_mode=_abi.BN_MOVING):
        mel = self._f32(mel)
        N, T, _ = mel.shape
        out = torch.empty(N, T, self.hp.num_freq, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_postnet(self._h, _ptr(mel), N, T, bn_mode, 0, _ptr(out), 0, self.stream))
        return out

    def bigru(self, which, x, lengths=None):
        x = self._f32(x)
        lengths = self._i32(lengths)
        N, T, _ = x.shape
        out = torch.empty(N, T, 256, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_bigru(self._h, which, _ptr(x), _ptr(lengths), N, T, _ptr(out), self.stream))
        return out

    def conv1d(self, x, kernel, bias=None, act=_abi.ACT_NONE):
        x, kernel, bias = self._f32(x), self._f32(kernel), self._f32(bias)
        N, T, Cin = x.shape
        k, _, Cout = kernel.shape
        out = torch.empty(N, T, Cout, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_conv1d(self._h, _ptr(x), N, T, Cin, _ptr(kernel), _ptr(bias), k, Cout, act,
                                      _ptr(out), self.stream))
        return out

    def maxpool_affine(self, x, scale=None, shift=None):
        """``taco_maxpool_affine``: max_pooling1d(2, 1, 'same') of ``scale * x + shift`` (reference modules.py:45-49)."""
        x = self._f32(x)
        N, T, Cc = x.shape
        sc = self._f32(scale) if scale is not None else None
        sh = self._f32(shift) if shift is not None else None
        out = torch.empty_like(x)
        self._ck(self.lib.taco_maxpool_affine(self._h, _ptr(x), N, T, Cc, _ptr(sc), _ptr(sh), _ptr(out), self.stream))
        return out

    def bn_batch_stats(self, x, gamma, beta):
        """``taco_bn_batch_stats``: (scale, shift) with BN_training(x) = scale * x + shift (reference modules.py:101)."""
        x, gamma, beta = self._f32(x), self._f32(gamma), self._f32(beta)
        N, T, Cc = x.shape
        scale = torch.empty(Cc, device=self.device, dtype=torch.float32)
        shift = torch.empty(Cc, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_bn_batch_stats(self._h, _ptr(x), N, T, Cc, _ptr(gamma), _ptr(beta), _ptr(scale), _ptr(shift), self.stream))
        return scale, shift

    def gemm_unit(self, N, T, Cin, Cout, w, *, x=None, x_bs=None, ldx=None, x_split=None, taps=1, bank=1, bias=None,
                  scale=None, shift=None, res=None, res_bs=None, ldres=None, act=_abi.ACT_NONE, out=None, out_bs=None,
                  ldo=None, col_off=0, out_split=None, out_cp=0):
        """``taco_gemm_unit`` in the current gemm mode.  ``x`` / ``res`` / ``out`` are device tensors addressed through the
        given strides (defaults: dense [N, T, C]); ``x_split`` / ``out_split`` are (hi, lo) bf16 operand tensors.  Weights
        and per-channel parameters are host arrays in the reference layouts.  Returns the plan the launch used (a dict)."""
        keep = []

        def host(a):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.float32)
            keep.append(a)
            return a.ctypes.data

        def dev(t):
            return None if t is None else t.data_ptr()

        d = _abi.TacoGemmDesc()
        d.x, d.x_bs, d.ldx = dev(x), T * Cin if x_bs is None else x_bs, Cin if ldx is None else ldx
        d.x_hi, d.x_lo = (dev(x_split[0]), dev(x_split[1])) if x_split is not None else (None, None)
        d.N, d.T, d.Cin, d.taps, d.bank, d.Cout = N, T, Cin, taps, bank, Cout
        d.w_host, d.bias_host = host(w), host(bias)
        d.scale_host, d.shift_host = host(scale), host(shift)
        d.res, d.res_bs, d.ldres = dev(res), T * Cout if res_bs is None else res_bs, Cout if ldres is None else ldres
        d.act = act
        width = Cout * max(bank, 1)
        d.out, d.out_bs, d.ldo, d.col_off = dev(out), T * width if out_bs is None else out_bs, width if ldo is None else ldo, col_off
        d.out_hi, d.out_lo = (dev(out_split[0]), dev(out_split[1])) if out_split is not None else (None, None)
        d.out_cp = out_cp
        plan = _abi.TacoGemmPlan()
        self._ck(self.lib.taco_gemm_unit(self._h, C.byref(d), C.byref(plan), self.stream))
        return plan.as_dict()

    def highway4_unit(self, x, w_h, b_h, w_t, b_t, out=None, out_split=None):
        """``taco_highway4_unit``: len(w_h) highway layers on x [rows, 128] (device) with host weights [layers, 128, 128] and
        biases [layers, 128]; writes ``out`` [rows, 128] and / or the bf16 (hi, lo) copy ``out_split``."""
        w_h, b_h, w_t, b_t = (np.ascontiguousarray(a, dtype=np.float32) for a in (w_h, b_h, w_t, b_t))
        hi, lo = out_split if out_split is not None else (None, None)
        self._ck(self.lib.taco_highway4_unit(self._h, _ptr(x), x.shape[0], w_h.shape[0], w_h.ctypes.data, b_h.ctypes.data,
                                             w_t.ctypes.data, b_t.ctypes.data, _ptr(out), _ptr(hi), _ptr(lo), self.stream))

    def bigru_unit(self, xproj, ug, uc, lengths=None, impl=0, out=None):
        """``taco_bigru_unit``: the BiGRU recurrence alone on hoisted projections xproj [N, T, 768] (device, fp32) with host
        recurrent kernels ug [2, 128, 256], uc [2, 128, 128]; impl 0 = fp32 FFMA kernel, 1 = tensor-core kernel.  Writes
        ``out`` [N, T, 256] (device; allocated when None, else any 16-byte aligned dense view) and returns it."""
        ug, uc = (np.ascontiguousarray(a, dtype=np.float32) for a in (ug, uc))
        N, T, _ = xproj.shape
        lengths = self._i32(lengths)
        if out is None:
            out = torch.empty(N, T, 256, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_bigru_unit(self._h, int(impl), _ptr(xproj), _ptr(lengths), N, T, ug.ctypes.data,
                                          uc.ctypes.data, _ptr(out), self.stream))
        return out

    # ---- vocoder (the step after the path) ----
    def audio_params(self, griffin_lim_iters: Optional[int] = None) -> "_abi.TacoAudioParams":
        hp = self.hp
        return _abi.TacoAudioParams(
            int(hp.sample_rate), int(hp.griffin_lim_iters if griffin_lim_iters is None else griffin_lim_iters),
            float(hp.frame_length_ms), float(hp.frame_shift_ms), float(hp.preemphasis),
            float(hp.min_level_db), float(hp.ref_level_db), float(hp.power))

    def griffin_lim(self, linear, griffin_lim_iters: Optional[int] = None, inv_preemphasis: bool = True, out=None):
        """``audio.inv_spectrogram_tensorflow`` + ``audio.inv_preemphasis`` (reference synthesizer.py:27,50) for a
        batch ``linear [N,T,num_freq]`` (or one ``[T,num_freq]``): returns wav ``[N,(T-1)*hop+win]`` on the device."""
        linear = self._f32(linear)
        single = linear.dim() == 2
        if single:
            linear = linear[None]
        N, T, F = linear.shape
        if F != self.hp.num_freq:
            raise ValueError("linear spectrogram has %d bins, hparams.num_freq is %d" % (F, self.hp.num_freq))
        ap = self.audio_params(griffin_lim_iters)
        if not inv_preemphasis:
            ap.preemphasis = 0.0
        L = self.lib.taco_wav_length(C.byref(ap), T)
        if L < 0:
            raise ValueError("bad audio hparams")
        if out is None:
            wav = torch.empty(N, L, device=self.device, dtype=torch.float32)
        else:                                          # caller's buffer (stable pointers let the C ABI replay its CUDA graph)
            wav = out
            if tuple(wav.shape) != (N, L) or wav.dtype != torch.float32 or not wav.is_contiguous() or wav.device != linear.device:
                raise ValueError("out must be a contiguous float32 [%d, %d] tensor on the engine's device" % (N, L))
        self._ck(self.lib.taco_griffin_lim(self._h, C.byref(ap), _ptr(linear), N, T, 0, _ptr(wav), self.stream))
        return wav[0] if single else wav

    def spectrogram_frames(self, num_samples: int) -> int:
        """Frames the analysis gives ``num_samples`` samples: ``1 + num_samples // hop`` (``taco_spectrogram_frames``)."""
        T = int(self.lib.taco_spectrogram_frames(C.byref(self.audio_params()), int(num_samples)))
        if T < 0:
            raise ValueError("bad audio hparams or length")
        return T

    def spectrogram(self, wav, lengths=None, T_out: Optional[int] = None):
        """``audio.spectrogram`` and ``audio.melspectrogram`` of the reference (``taco_spectrogram``) for one waveform
        ``[L]``, a batch ``[N, L]`` (with optional per-utterance ``lengths``) or a list of 1-D waveforms of different
        lengths.  Returns ``(linear, mel)`` CUDA tensors ``[N, T_out, num_freq]`` / ``[N, T_out, num_mels]`` (``[T, F]``
        for one 1-D waveform); ``T_out`` defaults to the longest utterance's frames, and rows past an utterance's own
        frames are 0.0, the padding of the teacher-forcing targets."""
        wav, len_host, single = self._batch(wav, lengths)
        N, L = wav.shape
        longest = int(len_host.max()) if len_host is not None else L
        T = self.spectrogram_frames(longest) if T_out is None else int(T_out)
        hp = self.hp
        lin = torch.empty(N, T, hp.num_freq, device=self.device, dtype=torch.float32)
        mel = torch.empty(N, T, hp.num_mels, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_spectrogram(self._h, C.byref(self.audio_params()), _ptr(wav),
                                           None if len_host is None else len_host.ctypes.data, N, L, T, _ptr(lin),
                                           _ptr(mel), self.stream))
        return (lin[0], mel[0]) if single else (lin, mel)

    def resample_length(self, num_samples: int, orig_sr: int, target_sr: int) -> int:
        """Samples ``librosa.core.resample`` returns for ``num_samples`` inputs: ``ceil(num_samples * target_sr /
        orig_sr)`` (``taco_resample_length``)."""
        n = int(self.lib.taco_resample_length(int(num_samples), int(orig_sr), int(target_sr)))
        if n < 0:
            raise ValueError("bad sample rate or length")
        return n

    def resample(self, wav, orig_sr: int, target_sr: int, lengths=None):
        """``librosa.core.resample(wav, orig_sr, target_sr)`` with resampy's ``kaiser_best`` filter and ``fix=True``
        (``taco_resample``) for one waveform ``[L]``, a batch ``[N, L]`` (with optional per-utterance ``lengths``) or a
        list of 1-D waveforms of different lengths.  Returns a CUDA tensor ``[L_out]`` for one waveform; for a batch
        ``(y [N, L_out], out_lengths)``, where row n holds ``out_lengths[n] = ceil(len_n * target_sr / orig_sr)`` samples
        and 0.0 after them."""
        wav, len_host, single = self._batch(wav, lengths)
        N, L = wav.shape
        lens = len_host if len_host is not None else np.full(N, L, np.int32)
        out_len = np.asarray([self.resample_length(v, orig_sr, target_sr) for v in lens], np.int64)
        L_out = int(out_len.max())
        y = torch.empty(N, L_out, device=self.device, dtype=torch.float32)
        self._ck(self.lib.taco_resample(self._h, int(orig_sr), int(target_sr), _ptr(wav),
                                        None if len_host is None else len_host.ctypes.data, N, L, _ptr(y), L_out,
                                        self.stream))
        return y[0] if single else (y, out_len)

    def durations(self, align, text_lengths, frames):
        """Frames per symbol of a teacher-forced alignment ``[N, T_in, steps]`` (``taco_durations``): Glow-TTS's
        monotonic alignment search in float64 over ``log(max(a, 2^-149))``, ties staying on the same symbol, for
        utterances of ``text_lengths[n]`` symbols and ``frames[n]`` target frames (``ceil(frames / r)`` decoder steps).
        Returns a CUDA int32 tensor ``[N, T_in]``: each symbol's frames (they sum to ``frames[n]``, each >= 1), 0 past
        the text length."""
        align = self._f32(align)
        if align.dim() != 3:
            raise ValueError("align must be [N, T_in, steps]")
        N, T_in, steps = align.shape

        def host_i32(v):
            v = v.cpu() if isinstance(v, torch.Tensor) else v
            v = np.ascontiguousarray(np.asarray(v).reshape(-1), dtype=np.int32)
            if v.shape != (N,):
                raise ValueError("text_lengths and frames must be [N]")
            return v
        lens, fr = host_i32(text_lengths), host_i32(frames)
        out = torch.empty(N, T_in, device=self.device, dtype=torch.int32)
        self._ck(self.lib.taco_durations(self._h, _ptr(align), N, T_in, steps, lens.ctypes.data, fr.ctypes.data, _ptr(out),
                                         self.stream))
        return out

    def _batch(self, wav, lengths):
        """(wav [N, L] float32 on the device, host int32 lengths [N] or None, whether the input was one 1-D waveform) for
        a waveform, a batch with optional lengths or a list of 1-D waveforms."""
        if isinstance(wav, (list, tuple)):
            if lengths is not None:
                raise ValueError("lengths are implied by a list of waveforms")
            seqs = [np.asarray(w.detach().cpu() if isinstance(w, torch.Tensor) else w, dtype=np.float32) for w in wav]
            if not seqs or any(s.ndim != 1 or s.size == 0 for s in seqs):
                raise ValueError("expected a non-empty list of non-empty 1-D waveforms")
            lengths = [s.size for s in seqs]
            batch = np.zeros((len(seqs), max(lengths)), np.float32)
            for i, s in enumerate(seqs):
                batch[i, :s.size] = s
            wav = batch
        wav = self._f32(wav)
        single = False
        if wav.dim() == 1:
            if lengths is not None:
                raise ValueError("lengths need a batch [N, L]")
            single, wav = True, wav[None]
        if wav.dim() != 2 or wav.shape[1] == 0:
            raise ValueError("wav must be [L] or [N, L] with L >= 1")
        len_host = None
        if lengths is not None:
            len_host = np.ascontiguousarray(np.asarray(lengths).reshape(-1), dtype=np.int32)
            if len_host.shape != (wav.shape[0],):
                raise ValueError("lengths must be [N]")
        return wav, len_host, single

    # ---- whole path ----
    def forward(self, ids, lengths, spk=None, mel_targets=None, teacher_force=False,
                bn_mode=_abi.BN_MOVING, want_linear=True, want_alignments=True, out=None):
        """Device-resident call of ``taco_forward``.  Returns (mel [N,steps*r,M],
        linear [N,steps*r,F] | None, alignments [N,T_in,steps] | None, steps)."""
        ids, lengths = self._i32(ids), self._i32(lengths)
        spk = self._i32(spk) if (spk is not None and self.id_num > 1) else None
        tg = self._f32(mel_targets) if teacher_force else None
        N, T_in = ids.shape
        T_tgt = tg.shape[1] if tg is not None else 0
        hp = self.hp
        ms = self.max_steps(teacher_force, T_tgt)
        maxT = ms * hp.outputs_per_step
        if out is None:
            mel = torch.zeros(N, maxT, hp.num_mels, device=self.device, dtype=torch.float32)
            lin = torch.zeros(N, maxT, hp.num_freq, device=self.device, dtype=torch.float32) if want_linear else None
            al = torch.zeros(N, T_in, ms, device=self.device, dtype=torch.float32) if want_alignments else None
        else:
            mel, lin, al = out
        steps = C.c_int32(0)
        self._ck(self.lib.taco_forward(self._h, _ptr(ids), _ptr(lengths), _ptr(spk), _ptr(tg), N, T_in, T_tgt,
                                       bn_mode, int(teacher_force), _ptr(mel), _ptr(lin), _ptr(al),
                                       C.byref(steps), self.stream))
        s = steps.value
        T = s * hp.outputs_per_step
        return (mel[:, :T], lin[:, :T] if lin is not None else None,
                al[:, :, :s] if al is not None else None, s)

    def _check_host_buffers(self, ids, lengths, spk, mel_targets, teacher_force, mel_out, linear_out, align_out):
        """The C ABI reads and writes raw host pointers: refuse anything that is not the dtype / layout it expects instead of
        reinterpreting an int64 id array as int32 or overrunning a short output buffer.  Returns the (possibly converted)
        input arrays; outputs must already be C-contiguous float32 of the full size."""
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        if ids.ndim != 2:
            raise ValueError("ids must be [N, T_in]")
        N, T_in = ids.shape
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        if lengths.shape != (N,):
            raise ValueError("lengths must be [N]")
        if spk is not None:
            spk = np.ascontiguousarray(spk, dtype=np.int32)
            if spk.shape != (N,):
                raise ValueError("speaker ids must be [N]")
        T_tgt = 0
        if teacher_force:
            if mel_targets is None:
                raise ValueError("teacher_force needs mel_targets")
            mel_targets = np.ascontiguousarray(mel_targets, dtype=np.float32)
            if mel_targets.ndim != 3 or mel_targets.shape[0] != N or mel_targets.shape[2] != self.hp.num_mels:
                raise ValueError("mel_targets must be [N, T_tgt, num_mels]")
            T_tgt = mel_targets.shape[1]
        ms = self.max_steps(teacher_force, T_tgt)
        maxT = ms * self.hp.outputs_per_step
        for name, buf, shape in (("mel_out", mel_out, (N, maxT, self.hp.num_mels)),
                                 ("linear_out", linear_out, (N, maxT, self.hp.num_freq)),
                                 ("align_out", align_out, (N, T_in, ms))):
            if buf is None:
                if name == "mel_out":
                    raise ValueError("mel_out is required")
                continue
            if not isinstance(buf, np.ndarray) or buf.dtype != np.float32 or not buf.flags["C_CONTIGUOUS"] or not buf.flags["WRITEABLE"]:
                raise TypeError("%s must be a writeable C-contiguous float32 numpy array" % name)
            if tuple(buf.shape) != shape:
                raise ValueError("%s must have shape %s (max_steps = %d), got %s" % (name, shape, ms, tuple(buf.shape)))
        return ids, lengths, spk, mel_targets

    def forward_host_begin(self, ids: np.ndarray, lengths: np.ndarray, spk: Optional[np.ndarray],
                           mel_targets: Optional[np.ndarray], teacher_force: bool, bn_mode: int,
                           mel_out: np.ndarray, linear_out: Optional[np.ndarray], align_out: Optional[np.ndarray]) -> None:
        """``taco_forward_host_begin``: inputs copied, forward run, output copies ENQUEUED (see ``forward_host_end``).
        The input arrays must stay alive (and unchanged) until ``forward_host_end`` returns."""
        ids, lengths, spk, mel_targets = self._check_host_buffers(ids, lengths, spk, mel_targets, teacher_force,
                                                                  mel_out, linear_out, align_out)
        self._host_keepalive = (ids, lengths, spk, mel_targets)
        N, T_in = ids.shape
        T_tgt = mel_targets.shape[1] if (teacher_force and mel_targets is not None) else 0

        def hp_(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)

        use_spk = spk if (spk is not None and self.id_num > 1) else None
        self._ck(self.lib.taco_forward_host_begin(self._h, hp_(ids), hp_(lengths), hp_(use_spk),
                                                  hp_(mel_targets if teacher_force else None), N, T_in, T_tgt, bn_mode,
                                                  int(teacher_force), hp_(mel_out), hp_(linear_out), hp_(align_out),
                                                  self.stream))

    def forward_host_wait(self, stage: int = 1) -> None:
        """``taco_forward_host_wait``: block until the decoder loop (stage 0) or all kernels (stage 1) of the forward
        begun on this handle are done (its post-net resp. output copies may still be in flight)."""
        self._ck(self.lib.taco_forward_host_wait(self._h, stage))

    def forward_host_end(self) -> int:
        """``taco_forward_host_end``: wait for the output copies of the forward begun on this handle; step count."""
        steps = C.c_int32(0)
        self._ck(self.lib.taco_forward_host_end(self._h, C.byref(steps), self.stream))
        return steps.value

    def forward_host(self, ids: np.ndarray, lengths: np.ndarray, spk: Optional[np.ndarray],
                     mel_targets: Optional[np.ndarray], teacher_force: bool, bn_mode: int,
                     mel_out: np.ndarray, linear_out: Optional[np.ndarray], align_out: Optional[np.ndarray]) -> int:
        """``taco_forward_host``: HOST numpy buffers in and out (H2D/D2H inside)."""
        ids, lengths, spk, mel_targets = self._check_host_buffers(ids, lengths, spk, mel_targets, teacher_force,
                                                                  mel_out, linear_out, align_out)
        N, T_in = ids.shape
        T_tgt = mel_targets.shape[1] if (teacher_force and mel_targets is not None) else 0

        def hp_(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)

        steps = C.c_int32(0)
        use_spk = spk if (spk is not None and self.id_num > 1) else None
        self._ck(self.lib.taco_forward_host(self._h, hp_(ids), hp_(lengths), hp_(use_spk),
                                            hp_(mel_targets if teacher_force else None), N, T_in, T_tgt, bn_mode,
                                            int(teacher_force), hp_(mel_out), hp_(linear_out), hp_(align_out),
                                            C.byref(steps), self.stream))
        return steps.value
