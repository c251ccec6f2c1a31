"""Device time of the resampler (taco_resample) for a batch of config-3 sized recordings at the rates of common corpora,
against its FFMA and byte floors.
usage: python tools/resample_bench.py [N] [seconds] [reps] [GB/s for the byte floor]

Default workload: 32 utterances of 12.5 s (the config-3 output length) from 16, 22.05 and 48 kHz to 20 kHz.  Per output
the filter runs (nwin // index_step) taps on each wing with 2 FMA per tap (A.x and D.x), so the FFMA floor is
N * n_out * 2 * taps * 2 / (148 SMs * 128 lanes * the SM clock read in the same run).  The byte floor is the input read
once plus the output written once.  Prints the median per-call time over `reps` samples of 10 back-to-back calls (CUDA
events, after warm-up) and the card's name and power limit read in the same run."""
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
seconds = float(sys.argv[2]) if len(sys.argv) > 2 else 12.5
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 30
gbps = float(sys.argv[4]) if len(sys.argv) > 4 else 6547.0     # copy bandwidth measured on a B200 (1000 W)
SR_NEW = 20000

if not torch.cuda.is_available():
    sys.exit("resample_bench needs a CUDA device")
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                    str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
card = q
try:
    clock_mhz = float(q.split(",")[2])
except (IndexError, ValueError):
    clock_mhz = 1965.0
sms = torch.cuda.get_device_properties(0).multi_processor_count
print("card: %s (name, power limit W, max SM clock MHz); %d SMs" % (card, sms))
eng = Engine(HParams(), id_num=0)
for sr in (16000, 22050, 48000):
    L = int(seconds * sr)
    x = torch.rand(N, L, device=eng.device) - 0.5
    L_out = eng.resample_length(L, sr, SR_NEW)
    y = torch.empty(N, L_out, device=eng.device)

    def call():   # the C ABI on preallocated buffers: what is timed is the kernel, not the wrapper's allocations
        eng._ck(eng.lib.taco_resample(eng._h, sr, SR_NEW, C.c_void_p(x.data_ptr()), None, N, L, C.c_void_p(y.data_ptr()),
                                      L_out, eng.stream))

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
    step = int(min(1.0, SR_NEW / sr) * 512)
    taps = 32769 // step
    fma = N * int(L * SR_NEW / sr) * 2 * taps * 2
    ffma_us = fma / (sms * 128 * clock_mhz * 1e6) * 1e6
    bytes_ = 4 * N * (L + L_out)
    byte_us = bytes_ / (gbps * 1e9) * 1e6
    print("%5d -> %d Hz  N=%d L=%d -> %d: median %.1f us per call (min %.1f, max %.1f over %d); "
          "FFMA floor %.1f us (%.2f G FMA, %d taps per wing) -> %.2fx; byte floor %.1f us (%.1f MB at %.0f GB/s)"
          % (sr, SR_NEW, N, L, L_out, us, min(times), max(times), reps, ffma_us, fma / 1e9, taps, us / ffma_us, byte_us,
             bytes_ / 1e6, gbps))
