"""Device time of the durations kernel (taco_durations) and of the stages of Synthesizer.align.
usage: python tools/durations_bench.py [reps] [GB/s for the byte floor]

Kernel: batch 32, T_in 100 and 512, Y = 200, 400 and 2000 decoder steps (r = 1, frames = Y), text lengths min(T_in, Y),
column-softmax alignments.  The search has Y dependent steps per utterance, so the kernel is bound by its step latency,
not by bytes: it reads each in-band alignment cell once (2.56 MB at config 3: 32 x 100 x 200 floats), which fits in L2
after the first call.  Printed: the median per-call time over `reps` samples of 10 back-to-back calls (CUDA events,
after warm-up), the time per decoder step, and the byte floor (alignment read once at the given bandwidth).

align: batch 32 recordings of 4.98 s at 16 kHz (399 frames at 20 kHz, within load's max_iters = 400 at r = 1) with
texts of 60 to 120 symbols, random-init weights; each stage as align runs it (32 resample calls, one spectrogram, one
teacher-forced forward without the post-net, one durations call), then the whole call by host clock.  The card's name
and power limit are read in the same run."""
import ctypes as C
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tacotron_multispeaker_b200 import audio, text  # noqa: E402
from tacotron_multispeaker_b200.engine import Engine, pad_inputs  # noqa: E402
from tacotron_multispeaker_b200.hparams import HParams  # noqa: E402
from tacotron_multispeaker_b200.synthesizer import Synthesizer  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 30
gbps = float(sys.argv[2]) if len(sys.argv) > 2 else 6547.0     # copy bandwidth measured on a B200 (1000 W)
N = 32

if not torch.cuda.is_available():
    sys.exit("durations_bench needs a CUDA device")
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                    str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
print("card: %s (name, power limit)" % q)


def median_us(fn, reps, inner=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(inner):
            fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3 / inner)
    return float(np.median(times)), min(times), max(times)


eng = Engine(HParams(outputs_per_step=1), id_num=0)
gen = torch.Generator(device=eng.device).manual_seed(0)
for T_in in (100, 512):
    for Y in (200, 400, 2000):
        X = min(T_in, Y)
        a = torch.softmax(3.0 * torch.randn(N, T_in, Y, device=eng.device, generator=gen), dim=1)
        out = torch.empty(N, T_in, dtype=torch.int32, device=eng.device)
        lens, frames = np.full(N, X, np.int32), np.full(N, Y, np.int32)

        def call():   # the C ABI on preallocated buffers: the kernel, not the wrapper's allocations
            eng._ck(eng.lib.taco_durations(eng._h, C.c_void_p(a.data_ptr()), N, T_in, Y, lens.ctypes.data,
                                           frames.ctypes.data, C.c_void_p(out.data_ptr()), eng.stream))

        us, lo, hi = median_us(call, reps)
        mb = 4.0 * N * X * Y / 1e6   # rows < X, columns < Y: what the kernel stages
        print("durations N=%d T_in=%d X=%d Y=%d: median %.1f us per call (min %.1f, max %.1f over %d); %.3f us per step; "
              "byte floor %.2f us (%.2f MB at %.0f GB/s)" % (N, T_in, X, Y, us, lo, hi, reps, us / Y,
                                                                     mb * 1e6 / (gbps * 1e9) * 1e6, mb, gbps))
eng.close()

# ---- the stages of Synthesizer.align ---------------------------------------------------------------------------------
text.load_symbols([chr(0x4E00 + i) for i in range(7350)])
syn = Synthesizer(HParams()).load(None, id_num=4)
rng = np.random.default_rng(1)
L = int(4.98 * 16000)
wavs = [(0.3 * np.sin(2 * np.pi * (200 + 40 * i) * np.arange(L) / 16000) + 0.01 * rng.normal(size=L)).astype(np.float32)
        for i in range(N)]
texts = ["".join(chr(0x4E00 + int(c)) for c in rng.integers(2, 7000, rng.integers(60, 121))) for _ in range(N)]
ids = list(rng.integers(0, 4, N))
engine = syn.model._get_engine(syn.id_num)
hp = syn.hparams
seqs = [np.asarray(text.text_to_sequence2(t)[:-1], np.int32) for t in texts]
lengths = np.asarray([s.size for s in seqs], np.int32)
stage = {}


def timed(name, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    e1.synchronize()
    stage.setdefault(name, []).append(e0.elapsed_time(e1) * 1e3)
    return r


for it in range(reps // 3 + 3):
    ys = timed("resample x32", lambda: [audio.resample(engine, torch.as_tensor(w), 16000, hp.sample_rate) for w in wavs])
    frames = [engine.spectrogram_frames(y.numel()) for y in ys]
    wav = torch.zeros(N, max(y.numel() for y in ys), device=engine.device)
    for i, y in enumerate(ys):
        wav[i, :y.numel()] = y
    mel = timed("spectrogram", lambda: engine.spectrogram(wav, lengths=[y.numel() for y in ys], T_out=max(frames) + 1)[1])
    al = timed("forward (teacher-forced, no post-net)",
               lambda: engine.forward(pad_inputs(seqs), lengths, np.asarray(ids, np.int32), mel, teacher_force=True,
                                      want_linear=False)[2])
    timed("durations", lambda: engine.durations(al, lengths, frames))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    syn.align(texts, ids, wavs, orig_sr=16000)
    torch.cuda.synchronize()
    stage.setdefault("align() whole call, host clock", []).append((time.perf_counter() - t0) * 1e6)
    if it == 2:   # warm-up done
        stage.clear()
print("align: N=%d, %.2f s at 16 kHz -> %d frames, texts %d..%d symbols, T_in %d, %d decoder steps"
      % (N, L / 16000, max(frames), lengths.min(), lengths.max(), lengths.max(), al.shape[2]))
for name, v in stage.items():
    print("  %-40s median %9.1f us (min %.1f, max %.1f over %d)" % (name, np.median(v), min(v), max(v), len(v)))
