"""Device time of the spectrogram analysis (taco_spectrogram: linear and mel rows) for a batch of config-3 sized utterances,
against the time the bytes alone need.
usage: python tools/spec_bench.py [N] [L] [reps] [GB/s for the byte floor]

Default workload: 32 utterances of 250 000 samples (12.5 s at 20 kHz, the config-3 output length) = 1001 frames each.
Every call reads the waveforms (32 MB) and writes the linear (131.3 MB) and mel (10.3 MB) rows: 174 MB, more than the
126 MB of L2, so each call streams from HBM.  Prints the median per-call time over `reps` samples of 10 back-to-back calls
(CUDA events, after warm-up), the card's name and power limit read in the same run, and the byte floor at the given
bandwidth."""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tacotron_multispeaker_b200.engine import Engine  # noqa: E402
from tacotron_multispeaker_b200.hparams import HParams  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 32
L = int(sys.argv[2]) if len(sys.argv) > 2 else 250000
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 50
gbps = float(sys.argv[4]) if len(sys.argv) > 4 else 6547.0     # copy bandwidth measured on a B200 (1000 W)

if not torch.cuda.is_available():
    sys.exit("spec_bench needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                       str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
hp = HParams()
eng = Engine(hp, id_num=0)
wav = torch.rand(N, L, device=eng.device) - 0.5
T = eng.spectrogram_frames(L)
lin = torch.empty(N, T, hp.num_freq, device=eng.device)
mel = torch.empty(N, T, hp.num_mels, device=eng.device)
ap = eng.audio_params()


def call():   # the C ABI on preallocated outputs: what is timed is the kernel, not the wrapper's allocations
    eng._ck(eng.lib.taco_spectrogram(eng._h, C.byref(ap), C.c_void_p(wav.data_ptr()), None, N, L, T,
                                     C.c_void_p(lin.data_ptr()), C.c_void_p(mel.data_ptr()), eng.stream))


for _ in range(5):
    call()
torch.cuda.synchronize()
times = []
for _ in range(reps):   # 10 calls back to back per sample, so that the host's enqueue time is hidden
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        call()
    e1.record()
    e1.synchronize()
    times.append(e0.elapsed_time(e1) * 1e3 / 10)
us = float(np.median(times))
bytes_ = N * L * 4 + N * T * (hp.num_freq + hp.num_mels) * 4
floor_us = bytes_ / (gbps * 1e9) * 1e6
print("card: %s" % card)
print("spectrogram N=%d L=%d (T=%d frames): median %.1f us per call (min %.1f, max %.1f over %d), %.1f M frames/s"
      % (N, L, T, us, min(times), max(times), reps, N * T / us))
print("bytes %.1f MB (wav %.1f, linear %.1f, mel %.1f): floor %.1f us at %.0f GB/s -> %.2fx the floor, %.0f GB/s achieved"
      % (bytes_ / 1e6, N * L * 4 / 1e6, N * T * hp.num_freq * 4 / 1e6, N * T * hp.num_mels * 4 / 1e6, floor_us, gbps,
         us / floor_us, bytes_ / us / 1e3))
