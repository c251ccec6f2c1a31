"""Serving facade with the reference's ``Synthesizer`` surface.

Mirrors reference ``synthesizer.py:13-58``: ``load(checkpoint_path,
model_name='tacotron')`` builds the model for batch-1 inference with
``max_iters = 400`` (``synthesizer.py:21``) and discovers ``id_num`` from the
shape of the checkpoint variable ``model/inference/embedding_id``
(``synthesizer.py:23-25``; a single-speaker checkpoint raises ``KeyError``
exactly like the reference); ``synthesize(text, identity, path, path_align)``
converts text with ``text_to_sequence2(...)[:-1]`` (``synthesizer.py:39``) and
runs the forward path.

``synthesize`` then runs the reference's Griffin-Lim graph (``synthesizer.py:27``,
``util/audio.py:39-46``) and ``inv_preemphasis`` (``synthesizer.py:50``) on the GPU
(``taco_griffin_lim``), writes the waveform with ``save_wav`` to ``path`` (``./1.wav``
when ``path`` is None, as the reference does) and the alignment image to
``path_align``.  It returns the bytes of the WAV file (the reference returns an
empty ``BytesIO`` it never writes to -- ``synthesizer.py:52-58``).
Checkpoints are TensorFlow V2 bundles (``model.ckpt-N.index`` + ``.data-*``, read by
``tf_checkpoint.py`` without TensorFlow) or ``.npz`` archives keyed by TF variable
names; without one, ``load(None, id_num=...)`` uses random-init weights.
"""
from __future__ import annotations

import io
from typing import Optional

import numpy as np
import torch

from . import audio, plot
from .engine import pad_inputs, pad_targets
from .hparams import HParams, hparams as default_hparams
from .tacotron import create_model
from .text import sequence_to_text2, text_to_sequence2
from .tf_checkpoint import load_weights
from .weights import PREFIX, random_init


class Synthesizer:
    def __init__(self, hparams: Optional[HParams] = None, device=None, verbose: bool = False):
        self.hparams = (hparams or default_hparams).copy()
        self._device = device
        self._verbose = verbose
        self.model = None
        self.id_num = 0

    def load(self, checkpoint_path, model_name="tacotron", id_num: Optional[int] = None, seed: int = 1234):
        print("Constructing model: %s" % model_name)
        hp = self.hparams
        hp.chinese_symbol = True          # synthesizer.py:20
        hp.max_iters = 400                # synthesizer.py:21
        self.model = create_model(model_name, hp, device=self._device, verbose=self._verbose)
        if checkpoint_path is None:
            if id_num is None:
                raise ValueError("load(None) needs id_num for the random-init fallback")
            weights = random_init(hp, id_num, seed=seed)
        else:
            print("Loading checkpoint: %s" % checkpoint_path)
            # a TF V2 checkpoint prefix ("model.ckpt-1000"), a log directory with a `checkpoint` state file, or .npz
            weights = load_weights(checkpoint_path)
        var_to_shape_map = {k: tuple(v.shape) for k, v in weights.items()}
        self.id_num = var_to_shape_map[PREFIX + "embedding_id"][0]   # KeyError if single-speaker: synthesizer.py:25
        self.model.load_weights(weights)
        return self

    def synthesize_sequence(self, seq, identity: int):
        """Batch-1 forward on an id sequence.  Returns (linear [T_out,F], alignment [T_in,steps])
        as numpy arrays (the two fetches of synthesizer.py:47 before Griffin-Lim)."""
        seq = np.asarray(seq, dtype=np.int32)[None, :]
        lengths = np.asarray([seq.shape[1]], dtype=np.int32)
        ident = np.asarray([identity], dtype=np.int32)
        self.model.initialize(seq, lengths, identities=ident, id_num=self.id_num)
        return (self.model.linear_outputs[0].cpu().numpy(), self.model.alignments[0].cpu().numpy())

    def synthesize_sequence_wav(self, seq, identity: int):
        """Batch-1 forward + vocoder on an id sequence.  Returns (wav float32 [L], alignment [T_in,steps])."""
        seq = np.asarray(seq, dtype=np.int32)[None, :]
        lengths = np.asarray([seq.shape[1]], dtype=np.int32)
        ident = np.asarray([identity], dtype=np.int32)
        self.model.initialize(seq, lengths, identities=ident, id_num=self.id_num)
        wav = audio.synthesize_wav(self.model.engine, self.model.linear_outputs[0])
        return wav.cpu().numpy(), self.model.alignments[0].cpu().numpy()

    def teacher_forced(self, text, identity, wav, path_align=None, orig_sr=None):
        """Teacher-forced run on a text and its recording: the attention alignment of the two and the ground-truth-aligned
        mel outputs.  ``wav`` is a path (``audio.load``: 16-bit PCM WAV of any sample rate and channel count, mixed down
        and resampled to ``hparams.sample_rate`` as ``librosa.core.load`` does), an array of samples or a CUDA tensor;
        an array or tensor recorded at another rate is resampled from ``orig_sr``.  Its mel spectrogram
        (``audio.melspectrogram`` on the GPU), padded as the feeder pads targets (``pad_targets``), feeds the decoder
        through ``initialize(..., teacher_force=True)``; batch norm keeps its moving statistics.  As in the reference, the
        decoder stops after min(max_iters, T_targets / r) steps, and ``load`` sets max_iters to 400, so a recording longer
        than 400 * r frames is cut there.  Returns ``(mel_outputs [steps*r, num_mels], alignment [T_in, steps])`` as
        numpy arrays and writes the alignment image to ``path_align`` when given."""
        seq = np.asarray(text_to_sequence2(text, [x.strip() for x in self.hparams.cleaners.split(",")])[:-1], np.int32)
        engine = self.model._get_engine(self.id_num if self.id_num > 1 else 0)
        if isinstance(wav, (str, bytes)) or hasattr(wav, "__fspath__"):
            wav = audio.load(engine, wav, self.hparams.sample_rate)
        elif orig_sr is not None:
            wav = audio.resample(engine, torch.as_tensor(wav).reshape(-1), orig_sr, self.hparams.sample_rate)
        if not isinstance(wav, torch.Tensor):
            wav = np.asarray(wav, dtype=np.float32)
        mel = audio.melspectrogram(engine, wav.reshape(-1))
        targets = pad_targets([mel.cpu().numpy()], self.hparams.outputs_per_step)
        self.model.initialize(seq[None, :], np.asarray([seq.size], np.int32), mel_targets=targets,
                              identities=np.asarray([identity], np.int32), id_num=self.id_num, teacher_force=True)
        alignment = self.model.alignments[0].cpu().numpy()
        if path_align is not None:
            plot.plot_alignment(alignment, path_align)
        return self.model.mel_outputs[0].cpu().numpy(), alignment

    def align(self, texts, identities, wavs, orig_sr=None):
        """Batched teacher forcing of texts with their recordings, and per-symbol durations from the attention.
        ``wavs`` are read as ``teacher_forced`` reads one (a path through ``audio.load``; an array or tensor, resampled
        from ``orig_sr`` when given).  The batch's mel targets come from one spectrogram call padded as the feeder pads
        targets (``max T_n + 1`` frames rounded up to r, zero rows) and feed one teacher-forced forward with the moving
        statistics of batch norm.  Durations are the monotonic alignment search of ``Engine.durations`` over utterance n's
        ``len_n`` symbols and ``1 + L_n // hop`` frames.  Returns, in input order, ``(durations int32 [len_n], alignment
        float32 [len_n, Y_n])`` numpy pairs with ``Y_n = ceil(frames_n / r)`` decoder steps.

        Attention is not length-masked (reference ``tacotron.py:68``), so a text padded to the batch's longest one
        attends to the padding too and its alignment differs from a batch of its own -- as in the reference's training
        graph.  ``align`` keeps the given order and does not re-bucket.  Raises ``ValueError`` naming the utterance for a
        text longer than 512 symbols, a recording longer than max_iters * r frames (``load`` sets max_iters = 400), or
        fewer decoder steps than symbols."""
        hp = self.hparams
        r = hp.outputs_per_step
        if not len(texts) == len(identities) == len(wavs) or not texts:
            raise ValueError("align needs as many identities and recordings as texts, and at least one")
        cleaners = [x.strip() for x in hp.cleaners.split(",")]
        seqs = [np.asarray(text_to_sequence2(t, cleaners)[:-1], np.int32) for t in texts]
        for i, s in enumerate(seqs):
            if not 1 <= s.size <= 512:
                raise ValueError("utterance %d: a text of %d symbols (align takes 1 to 512)" % (i, s.size))
        engine = self.model._get_engine(self.id_num if self.id_num > 1 else 0)
        ys = []
        for w in wavs:
            if isinstance(w, (str, bytes)) or hasattr(w, "__fspath__"):
                w = audio.load(engine, w, hp.sample_rate)
            elif orig_sr is not None:
                w = audio.resample(engine, torch.as_tensor(w).reshape(-1), orig_sr, hp.sample_rate)
            ys.append(engine._f32(w).reshape(-1))
        frames = [engine.spectrogram_frames(y.numel()) for y in ys]
        for i, (s, f) in enumerate(zip(seqs, frames)):
            if f > hp.max_iters * r:
                raise ValueError("utterance %d: %d frames, more than max_iters * r = %d (load sets max_iters = 400)"
                                 % (i, f, hp.max_iters * r))
            if -(-f // r) < s.size:
                raise ValueError("utterance %d: %d decoder steps for %d symbols" % (i, -(-f // r), s.size))
        N = len(ys)
        wav = torch.zeros(N, max(y.numel() for y in ys), device=engine.device, dtype=torch.float32)
        for i, y in enumerate(ys):
            wav[i, :y.numel()] = y
        T_out = -(-(max(frames) + 1) // r) * r                     # pad_targets' length
        _, mel = engine.spectrogram(wav, lengths=[y.numel() for y in ys], T_out=T_out)
        lengths = np.asarray([s.size for s in seqs], np.int32)
        _, _, al, _ = engine.forward(pad_inputs(seqs), lengths, np.asarray(identities, np.int32), mel, teacher_force=True,
                                     want_linear=False)
        engine.check_ids()
        dur = engine.durations(al, lengths, frames).cpu().numpy()
        al = al.cpu().numpy()
        return [(dur[i, :s.size], al[i, :s.size, :-(-f // r)]) for i, (s, f) in enumerate(zip(seqs, frames))]

    def synthesize(self, text, identity, path=None, path_align=None):
        seq = text_to_sequence2(text, [x.strip() for x in self.hparams.cleaners.split(",")])[:-1]
        print(seq)
        print(sequence_to_text2(seq))
        wav, alignment = self.synthesize_sequence_wav(seq, identity)
        if path_align is not None:
            plot.plot_alignment(alignment, path_align)
        # wav = wav[:audio.find_endpoint(wav, self.hparams.sample_rate)]   (disabled in the reference too)
        out = io.BytesIO()
        audio.save_wav(wav, out, self.hparams.sample_rate)
        audio.save_wav(wav, path if path is not None else "./1.wav", self.hparams.sample_rate)
        return out.getvalue()
