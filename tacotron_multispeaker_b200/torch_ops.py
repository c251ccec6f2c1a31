"""PyTorch custom operators over the C ABI: ``TORCH_LIBRARY(taco_b200, ...)`` in ``csrc/torch_ops.cpp``.

The reference is pure Python on TensorFlow 1.x (``models/tacotron.py:18``, ``synthesizer.py:47``) and has no operator API
of its own; SURVEY.md §8(b) asks for the path behind the host framework's operator interface, which for a PyTorch host is
``torch.ops``.  ``load()`` loads the in-tree ``libtaco_b200_torch.so`` (built by ``build.build_torch_ops`` /
``__graft_entry__.build``); after that ``torch.ops.taco_b200.forward(engine.handle, ids, lengths, ...)`` and friends are
available.  The operators check dtype / device / contiguity, allocate the outputs and pass raw device pointers and the
current CUDA stream to ``libtaco_b200.so``: no arithmetic is done by torch.  CUDA tensors only (there is no CPU fallback).
"""
from __future__ import annotations

import os

import torch

from . import _abi

_LIB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libtaco_b200_torch.so")
_loaded = False

OPS = ("forward", "encoder", "decode", "postnet", "griffin_lim", "spectrogram", "resample")


def load() -> str:
    """Load the operator library (idempotent).  Raises if it has not been built."""
    global _loaded
    if not _loaded:
        if not os.path.exists(_LIB):
            raise RuntimeError("%s not built: run tacotron_multispeaker_b200/build.py --torch-ops" % _LIB)
        _abi.load()                      # libtaco_b200.so first (the operator library links against it)
        torch.ops.load_library(_LIB)
        _loaded = True
    return _LIB


def forward(engine, ids, lengths, identities=None, mel_targets=None, teacher_force=False, bn_mode=_abi.BN_MOVING,
            want_linear=True, want_alignments=True):
    """``torch.ops.taco_b200.forward`` with the shape hyper-parameters taken from ``engine`` (device int32 / float32 tensors)."""
    load()
    hp = engine.hp
    return torch.ops.taco_b200.forward(engine.handle, ids, lengths, identities, mel_targets, bool(teacher_force), int(bn_mode),
                                       hp.num_mels, hp.num_freq, hp.outputs_per_step, want_linear, want_alignments)
