"""Developer aid: per-phase clock stamps of decoder_cw_kernel (TACO_DEC_TRACE): critical warp 12 stamps 0..22, background
warps stamp 64+w (items before the attention phases done), 80+w (attention phases done), 96+w (items after them done)."""
import os, sys
os.environ.setdefault("TACO_DEV", "1")   # per-call developer switches of the C ABI
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import make_inputs
from tacotron_multispeaker_b200.engine import Engine
from tacotron_multispeaker_b200.hparams import HParams
from tacotron_multispeaker_b200.weights import random_init

NAMES = {1: "P1 sent", 2: "P1 arrived", 3: "P2 sent", 4: "P2 arr", 5: "P3 sent", 6: "P3 arr", 7: "P4 sent", 8: "P4 arr", 9: "P5 sent",
         10: "P5 arr", 11: "P6 computed+sync", 12: "P6 arr", 13: "P7 computed+sync", 14: "P7 sent", 15: "P7 arr", 16: "P9 sent+align",
         17: "P9 arr", 18: "P10 sent", 19: "P10 arr", 20: "P11 sent", 21: "P11 arr", 22: "P12 sent"}


def run(N, T_in, S, tag, iters=40, teacher=False, cta=0):
    hp = HParams(outputs_per_step=5, max_iters=iters)
    w = random_init(hp, 60, seed=1234)
    ids, lengths, spk = make_inputs(N, T_in, 60, 1, min_len=max(1, int(T_in * 0.6)), vocab=(7108, 7325))
    os.environ["TACO_DEC_S"] = str(S)
    os.environ["TACO_DEC_TRACE_CTA"] = str(cta)
    eng = Engine(hp, 60); eng.load_weights(w)
    mem = eng.encoder(ids, lengths, spk, 0)
    tg = torch.rand(N, iters * 5, 80, device="cuda") if teacher else None
    for _ in range(2):
        eng.decode(mem, tg, teacher, True)
    torch.cuda.synchronize()
    path = os.path.join(ROOT, "gpurun_out", "trace_%s.txt" % tag)
    os.environ["TACO_DEC_TRACE"] = path
    eng.decode(mem, tg, teacher, True)
    torch.cuda.synchronize()
    os.environ.pop("TACO_DEC_TRACE")
    st = [int(l.split()[1]) for l in open(path) if not l.startswith("#")]
    t0 = st[0]
    print("%s N=%d S=%d %s cta %d: step (stamp 0 -> 22) %d clk" % (tag, N, S, "teacher" if teacher else "free", cta, st[22] - t0))
    prev = t0
    line = []
    for i in range(1, 23):
        if st[i]:
            line.append("%s:+%d" % (NAMES[i], st[i] - prev)); prev = st[i]
    print("   " + "  ".join(line))
    for b0, nm, nw in ((64, "pre items done", 12), (160, "P6 start (bg)", 12), (112, "P6 computed", 16), (176, "P6 computed x2", 12), (240, "P6 computed x3", 12), (128, "P7 start", 16), (144, "P7 computed", 16), (208, "P7 computed x2", 12), (272, "P7 computed x3", 12),
                       (80, "attention done", 12), (96, "post items done", 12)):
        print("   %-18s rel. stamp 0: %s" % (nm, [st[b0 + w_] - t0 if st[b0 + w_] else None for w_ in range(nw)]))
    for nm, b0 in (("pre", 320), ("post", 360)):
        rows = []
        for it in range(8):
            v = st[b0 + 4 * it: b0 + 4 * it + 4]
            if v[0]:
                rows.append("it%d@%d[A+%d ops+%d post+%d]" % (it, v[0] - t0, v[1] - v[0] if v[1] else -1, v[2] - (v[1] or v[0]), v[3] - v[2]))
        print("   warp %s %s items: %s" % (os.environ.get("TACO_DEC_TRACE_WARP", "8"), nm, " ".join(rows)))
    print("   P7 intra (warp 0, last rep): %s" % [st[300 + i] - st[300] for i in range(4)])
    print("   crit P11 intra (from P10 arr): late %d, sync CRIT %d, H11+reduce+stage %d, send %d, twait %d" % (st[45] - st[19], st[46] - st[45], st[47] - st[46], st[48] - st[47], st[20] - st[48]))
    print("   kernel: prologue %d clk, step 0 %d clk, steps 0..%d %d clk (%.0f per step)" % (st[25] - st[24], st[27] - st[25], iters - 1, st[26] - st[25], (st[26] - st[25]) / iters))
    ds = [st[401 + i] - st[400 + i] for i in range(min(iters, 100) - 1)]
    print("   step durations (clk): first 12 %s, median %d, max %d (step %d), mean %.0f" % (ds[:12], sorted(ds)[len(ds) // 2], max(ds), ds.index(max(ds)), sum(ds) / len(ds)))
    hn = ["H1", "H3", "H4", "H9", "H10", "H11", "H12"]
    print("   crit handoff waits: " + " ".join("%s:%d" % (hn[i], st[51 + 2 * i] - st[50 + 2 * i]) for i in range(7)))
    print("   crit: P5 arr %d, SYNC6 %d, P6 arr %d, SYNC7 %d" % (st[10] - t0, st[11] - t0, st[12] - t0, st[13] - t0))
    eng.close()


if __name__ == "__main__":
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    for S in (int(x) for x in os.environ.get("TRACE_S", "5").split(",")):   # config 3 cut into clusters of S
        for wtr in os.environ.get("TRACE_WARPS", "8,0,4").split(","):
            os.environ["TACO_DEC_TRACE_WARP"] = wtr
            run(32, 100, S, "cw_n32_s%d_w%s" % (S, wtr))
    if os.environ.get("TRACE_N1"):
        run(1, 100, 1, "cw_n1_s1")
