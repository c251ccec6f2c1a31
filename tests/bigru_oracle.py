"""Float64 restatement of the CBHG's BiGRU recurrence (reference models/modules.py:68-74) and a step-local bound for the CUDA
kernels that run it (``bigru_kernel<NS>`` in bigru.cu, ``bigru_mma_kernel`` in bigru_mma.cu).

TEST INFRASTRUCTURE ONLY (numpy).  The kernels take the hoisted input projections

    xproj[n, t] = x[n, t] Wx + b       [fw gates 256 | fw cand 128 | bw gates 256 | bw cand 128]

and the recurrent halves of the TF kernels, ug [2][128][256] and uc [2][128][128] (rows 128..255 of each direction's
``gates/kernel`` / ``candidate/kernel``).  One step of ``GRUCell`` (oracle ``gru_cell``, KATs 1-3) is then

    [r | u] = sigmoid(xg + h Ug)       r: gate columns 0..127, u: 128..255
    cand    = tanh(xc + (r h) Uc)      the reset gate is applied BEFORE the candidate matmul
    h'      = u h + (1 - u) cand

and ``dynamic_rnn`` (KAT 7) zeroes the outputs and freezes the state at t >= length; the backward direction runs over
``reverse_sequence(x, length)``: its step s reads and writes position length - 1 - s.

``local_check`` compares a kernel's output step by step without accumulating error.  Both kernels store exactly the fp32
state they carry, so the state a step started from is the kernel's own output at the neighbouring position (p - 1
forward, p + 1 backward, zero at a direction's first step).  One float64 step from that state is compared with the
kernel's out[p] against the first-order bound

    tol_j = u(1-u) |h_j - cand_j| eg_u,j + (1-u)(1-cand_j^2) (ec_j + sum_k r_k(1-r_k) eg_r,k |h_k| |Uc_kj|) + eps_act
    eg = c A + xerr_g,     A = |xg| + |h| |Ug|          (pre-activation error of the gates)
    ec = c B + xerr_c,     B = |xc| + (r |h|) |Uc|      (pre-activation error of the candidate)

``c`` is the relative error of the kernel's dot products, ``eps_act`` an absolute term for ``ex2.approx`` / ``rcp.approx``
and the final FMA, and xerr an error bound of xproj itself (the GEMM in front of the recurrence).  The derivatives
vanish where the gates saturate, so there the bound tightens to ``eps_act``.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

H = 128


def _mm(a, b):
    """a @ b with at least two rows: OpenBLAS sends a single row down its gemv path, whose sums are ordered differently
    from the gemm ones, and bigru64 / local_check must give the same bits for the same row whatever the batch."""
    if a.shape[0] >= 2:
        return a @ b
    return (np.concatenate([a, np.zeros((2 - a.shape[0], a.shape[1]))]) @ b)[: a.shape[0]]


def sigmoid(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


def split_weights(weights, scope):
    """The reference variables of one CBHG's BiGRU (``{scope}/bidirectional_rnn/{fw,bw}/gru_cell/...``, with or without the
    ``model/inference/`` prefix) as the kernels read them: wx [128, 768], bx [768], ug [2, 128, 256], uc [2, 128, 128]."""
    def get(name):
        for k in ("model/inference/" + name, name):
            if k in weights:
                return np.asarray(weights[k])
        raise KeyError(name)
    wx = np.zeros((H, 768), np.float32)
    bx = np.zeros(768, np.float32)
    ug = np.zeros((2, H, 256), np.float32)
    uc = np.zeros((2, H, H), np.float32)
    for d, dn in enumerate(("fw", "bw")):
        s = f"{scope}/bidirectional_rnn/{dn}/gru_cell"
        wg, bg, wc, bc = get(s + "/gates/kernel"), get(s + "/gates/bias"), get(s + "/candidate/kernel"), get(s + "/candidate/bias")
        wx[:, d * 384: d * 384 + 256], wx[:, d * 384 + 256: d * 384 + 384] = wg[:H], wc[:H]
        bx[d * 384: d * 384 + 256], bx[d * 384 + 256: d * 384 + 384] = bg, bc
        ug[d], uc[d] = wg[H:], wc[H:]
    return wx, bx, ug, uc


def _step(h, xg, xc, Ug, Uc):
    g = sigmoid(xg + _mm(h, Ug))
    r, u = g[:, :H], g[:, H:]
    cand = np.tanh(xc + _mm(r * h, Uc))
    return u * h + (1.0 - u) * cand, r, u, cand


def gru_step64(h_prev, xg, xc, Ug, Uc):
    """One GRUCell step in float64 on rows: h_prev [R, 128], xg [R, 256], xc [R, 128] -> h [R, 128]."""
    f = lambda a: np.asarray(a, np.float64)  # noqa: E731
    return _step(f(h_prev), f(xg), f(xc), f(Ug), f(Uc))[0]


def _lens(lengths, N, T):
    if lengths is None:
        return np.full(N, T, np.int64)
    return np.clip(np.asarray(lengths, np.int64), 0, T)


def bigru64(xproj, lengths, ug, uc):
    """bidirectional_dynamic_rnn(GRUCell(128), GRUCell(128)) on hoisted projections xproj [N, T, 768]: out [N, T, 256]
    float64, zero past each length, the backward half run over reverse_sequence."""
    xproj = np.asarray(xproj, np.float64)
    N, T, _ = xproj.shape
    L = _lens(lengths, N, T)
    out = np.zeros((N, T, 2 * H))
    ar = np.arange(N)
    for d in range(2):
        h = np.zeros((N, H))
        for s in range(T):
            pos = s if d == 0 else L - 1 - s
            live = (s < L)[:, None]
            posc = np.clip(pos, 0, T - 1) if d else np.full(N, s)
            x = xproj[ar, posc, d * 384: (d + 1) * 384]
            hn = gru_step64(h, x[:, :256], x[:, 256:], ug[d], uc[d])
            h = np.where(live, hn, h)
            cur = out[ar, posc, d * H: (d + 1) * H]
            out[ar, posc, d * H: (d + 1) * H] = np.where(live, hn, cur)
    return out


EPS_GRID = (5e-8, 1e-7, 2e-7, 5e-7, 1e-6)


@dataclass
class LocalResult:
    ok: bool
    checked: int           # elements compared
    max_err: float         # largest |out - step64| (inf for a NaN)
    c_ratio: float         # the c this output needs at the given eps_act: max c (|err| - eps_act) / (tol - eps_act)
    eps_excess: float      # the eps_act it needs at the given c: max |err| - (tol - eps_act)
    worst: tuple           # (n, p, dir, j, got, want, tol) of the largest |err| / tol
    c_at_eps: dict         # eps_act -> the c this output needs with that eps_act (no xproj_err only)

    def __str__(self):
        return "checked %d, max err %.3e, needs c >= %.3e, eps_act >= %.3e, worst (n, p, dir, j, got, want, tol) = %s" % (
            self.checked, self.max_err, self.c_ratio, self.eps_excess, self.worst)


def local_check(out_gpu, xproj, lengths, ug, uc, c, eps_act, xproj_err=None, chunk=16):
    """Step-local comparison of a kernel's BiGRU output out_gpu [N, T, 256] (see the module docstring) at every valid
    (utterance, position, direction, column).  xproj_err [N, T, 768] or None: an absolute error bound of each entry of
    xproj, added to eg / ec.  Returns a LocalResult; ``ok`` when every element is within its bound."""
    N, T, _ = xproj.shape
    L = _lens(lengths, N, T)
    Ugs = [np.asarray(u, np.float64) for u in ug]
    Ucs = [np.asarray(u, np.float64) for u in uc]
    res = dict(ok=True, checked=0, max_err=0.0, c_ratio=0.0, eps_excess=0.0, worst=None, c_at_eps={e: 0.0 for e in EPS_GRID})
    worst_q = -1.0
    p_idx = np.arange(T)
    for n0 in range(0, N, chunk):
        n1 = min(N, n0 + chunk)
        valid = p_idx[None, :] < L[n0:n1, None]                          # [n, T]
        if not valid.any():
            continue
        for d in range(2):
            o = np.asarray(out_gpu[n0:n1, :, d * H: (d + 1) * H], np.float64)
            hp = np.zeros_like(o)
            if d == 0:
                hp[:, 1:] = o[:, :-1]
            else:
                hp[:, :-1] = o[:, 1:]
                hp[~np.roll(valid, -1, axis=1) | (p_idx[None, :] == T - 1)] = 0.0   # p + 1 >= length: the first step
            rows = valid.reshape(-1)
            h = hp.reshape(-1, H)[rows]
            got = o.reshape(-1, H)[rows]
            x = np.asarray(xproj[n0:n1, :, d * 384: (d + 1) * 384], np.float64).reshape(-1, 384)[rows]
            xg, xc = x[:, :256], x[:, 256:]
            Ug, Uc = Ugs[d], Ucs[d]
            want, r, u, cand = _step(h, xg, xc, Ug, Uc)
            ah = np.abs(h)
            eg = c * (np.abs(xg) + _mm(ah, np.abs(Ug)))
            ec = c * (np.abs(xc) + _mm(r * ah, np.abs(Uc)))
            if xproj_err is not None:
                xe = np.asarray(xproj_err[n0:n1, :, d * 384: (d + 1) * 384], np.float64).reshape(-1, 384)[rows]
                eg, ec = eg + xe[:, :256], ec + xe[:, 256:]
            s = (u * (1.0 - u) * np.abs(h - cand) * eg[:, H:]
                 + (1.0 - u) * (1.0 - cand * cand) * (ec + _mm(r * (1.0 - r) * eg[:, :H] * ah, np.abs(Uc))))
            tol = s + eps_act
            err = np.abs(got - want)
            bad = ~(err <= tol)                                             # NaN fails too
            res["checked"] += err.size
            res["max_err"] = max(res["max_err"], np.inf if np.isnan(err).any() else float(err.max()))
            if c > 0:
                with np.errstate(divide="ignore", invalid="ignore"):
                    cr = np.where(s > 0, (err - eps_act) / s * c, np.where(err > eps_act, np.inf, 0.0))
                res["c_ratio"] = max(res["c_ratio"], float(np.nanmax(cr)))
            res["eps_excess"] = max(res["eps_excess"], float(np.nanmax(err - s)))
            if c > 0 and xproj_err is None:
                for e in EPS_GRID:
                    with np.errstate(divide="ignore", invalid="ignore"):
                        need = np.where(err > e, (err - e) / s * c, 0.0)
                    res["c_at_eps"][e] = max(res["c_at_eps"][e], float(np.nanmax(need)))
            with np.errstate(divide="ignore", invalid="ignore"):
                q = np.where(tol > 0, err / tol, np.where(err > 0, np.inf, 0.0))
            q = np.where(np.isnan(err), np.inf, q)
            i = int(np.argmax(q))
            if q.flat[i] > worst_q:
                worst_q = float(q.flat[i])
                row, j = divmod(i, H)
                nn, pp = np.argwhere(valid)[row]
                res["worst"] = (int(n0 + nn), int(pp), d, int(j), float(got.flat[i]), float(want.flat[i]), float(tol.flat[i]))
            if bad.any():
                res["ok"] = False
    return LocalResult(**res)
