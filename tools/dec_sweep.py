"""Developer aid: decoder_cw_kernel time per step over utterances per cluster S = 1..8 and input lengths, with the residency
plan of the attention operands each launch uses (taco_decoder_plan).  Four clusters of S utterances each (N = 4 S), free
running, max_iters steps.  Also checks that S = 5 and S = 8 give bit-identical decoder outputs at config 3 (N = 32, T_in 100).

    python tools/dec_sweep.py [--root TREE] [--t-in 60,100,200] [--iters 200]

--root runs another checkout of the project (for before / after comparisons in one process)."""
import argparse
import os
import sys

os.environ.setdefault("TACO_DEV", "1")   # per-call developer switches of the C ABI (TACO_DEC_S)
ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--t-in", default="60,100,200")
ap.add_argument("--iters", type=int, default=200)
ap.add_argument("--s", default="1,2,3,4,5,6,7,8")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from tacotron_multispeaker_b200 import _abi  # noqa: E402
from tacotron_multispeaker_b200.engine import Engine  # noqa: E402
from tacotron_multispeaker_b200.hparams import HParams  # noqa: E402
from tacotron_multispeaker_b200.weights import random_init  # noqa: E402

RES = {3: "keys+memory in smem", 4: "keys+memory in tmem", 1: "keys in smem", 2: "memory in smem", 0: "nothing resident"}


def decode(eng, mem, S):
    os.environ["TACO_DEC_S"] = str(S)
    try:
        return eng.decode(mem, None, False, True)
    finally:
        os.environ.pop("TACO_DEC_S", None)


def main():
    hp = HParams(outputs_per_step=5, max_iters=args.iters)
    w = random_init(hp, 60, seed=1234)
    eng = Engine(hp, 60)
    eng.load_weights(w)
    rng = np.random.default_rng(5)
    print("tree %s" % os.path.abspath(args.root), flush=True)
    for T_in in (int(x) for x in args.t_in.split(",")):
        for S in (int(x) for x in args.s.split(",")):
            N = 4 * S
            mem = torch.from_numpy((rng.standard_normal((N, T_in, 256)) * 0.5).astype(np.float32)).cuda()
            for _ in range(2):
                decode(eng, mem, S)
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(3):
                decode(eng, mem, S)
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / 3
            plan = _abi.decoder_plan(S, T_in, 1) if hasattr(_abi, "decoder_plan") else None
            pl = ("%s, ring %d KB, smem %d B" % (RES[plan["att_res"]], plan["ring_kb"], plan["smem_bytes"])) if plan else "n/a"
            print("T_in=%3d S=%d (N=%2d, 4 clusters): decode %.3f ms, %.2f us/step  plan: %s" % (T_in, S, N, ms, ms * 1e3 / args.iters, pl),
                  flush=True)
    mem = torch.from_numpy((rng.standard_normal((32, 100, 256)) * 0.5).astype(np.float32)).cuda()
    d5, a5, s5 = decode(eng, mem, 5)
    d8, a8, s8 = decode(eng, mem, 8)
    same = s5 == s8 and torch.equal(d5, d8) and torch.equal(a5, a8)
    print("config 3 decode S=5 vs S=8: steps %d / %d, bit-identical %s, max|d| dec %.3e align %.3e"
          % (s5, s8, same, float((d5 - d8).abs().max()), float((a5 - a8).abs().max())), flush=True)
    eng.close()


if __name__ == "__main__":
    main()
