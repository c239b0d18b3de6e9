"""Replica exchange restated on the CPU oracle's runs (test infrastructure, like oracle/).

`exchange_delta` restates exchange_delta of polymer-stats_b200/csrc/exchange.cuh with the same FP64 operations in the
same order (Python floats are IEEE doubles and are never contracted into FMA), and `draw_exchange_eps` the ε of Philox
stream 7.  `Ladders` holds one oracle Run per chain of a handle and swaps configurations between Runs: a Run that
receives a configuration re-binds its acceptor and α carry to it at its own kT and F (orc_run_set_state), and keeps
its accumulators, step sizes and counters, as a slot of the CUDA handle does.

The oracle numbers the trials of every orc_run_steps call from 1, i.e. each call restarts the Philox stream of the
init, while the library continues it across pmc_run calls.  A run that is continued chunk by chunk between exchange
rounds is therefore fed from a tape (orc_run_new_tape): `philox_tape` writes the draws the library makes for trials
step0+1 … step0+nsteps of the plain driver in the tape's order, so that the oracle makes the library's decisions.
"""
from __future__ import annotations

import math

import numpy as np

import oracle as O

SUB_EXCHANGE = 7
_M32 = 0xFFFFFFFF


def exchange_delta(kTa, kTb, Ua, Ub, ra, rb, Fxa, Fza, Fxb, Fzb):
    """-> (Δ, U_a(x_b), U_b(x_a)); accept iff Δ ≥ 0 or ε < exp(Δ)."""
    dFx, dFz = float(Fxb) - float(Fxa), float(Fzb) - float(Fza)
    wb = float(rb[0]) * dFx + float(rb[2]) * dFz
    wa = float(ra[0]) * dFx + float(ra[2]) * dFz
    Uab = float(Ub) + wb
    Uba = float(Ua) - wa
    ba, bb = 1.0 / float(kTa), 1.0 / float(kTb)
    return ba * (float(Ua) - Uab) + bb * (float(Ub) - Uba), Uab, Uba


def draw_exchange_eps(seed, chain_id, init, rnd):
    """ε of exchange round `rnd` for the pair whose lower slot is global chain `chain_id` at stream tag `init`."""
    w = O.philox([rnd & _M32, (rnd >> 32) & _M32, chain_id & _M32, ((init << 8) | SUB_EXCHANGE) & _M32],
                 [seed & _M32, (seed >> 32) & _M32])
    return float(((w[1] << 32) | w[0]) >> 11) * 2.0 ** -53


def philox(c0, c1, c2, c3, seed):
    """Philox4x32-10 over arrays of counters (oracle/polymc_oracle.c orc_philox4x32_10), key = the 64-bit seed."""
    c = [np.asarray(x, dtype=np.uint64) & _M32 for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(seed & _M32), np.uint64((seed >> 32) & _M32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & np.uint64(_M32), (p0 >> np.uint64(32)) ^ c[3] ^ k1,
             p0 & np.uint64(_M32)]
        k0 = (k0 + np.uint64(0x9E3779B9)) & np.uint64(_M32)
        k1 = (k1 + np.uint64(0xBB67AE85)) & np.uint64(_M32)
    return c


def _u53(lo, hi):
    return (((hi << np.uint64(32)) | lo) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def philox_tape(case, seed, chain_id, init, step0, nsteps):
    """Uniforms in the order a tape-driven oracle Run of the plain driver consumes them (polymc_oracle.h
    orc_run_new_tape): 2n for its initial chain (placeholders; set the state afterwards), then per trial idx, dϕ,
    [flip], dθ, ϵ — the Philox draws of trials step0+1 … step0+nsteps (chain_math.cuh draw_step)."""
    n = int(case.n)
    steps = np.arange(step0 + 1, step0 + nsteps + 1, dtype=np.uint64)
    tag = (init << 8)
    a = philox(steps, steps >> np.uint64(32), np.full_like(steps, chain_id), np.full_like(steps, tag | 0), seed)
    b = philox(steps, steps >> np.uint64(32), np.full_like(steps, chain_id), np.full_like(steps, tag | 1), seed)
    v_hi, v_lo = a[1], a[0]
    idx = (v_hi * np.uint64(n) + ((v_lo * np.uint64(n)) >> np.uint64(32))) >> np.uint64(32)   # umulhi(v, n)
    cols = [(idx.astype(np.float64) + 0.5) / n, _u53(a[2], a[3])]
    if case.do_flips:
        cols.append(np.where((a[2] & np.uint64(1)) != 0, 0.25, 0.75))   # the tape flips iff u < 1/2
    if not case.planar:
        cols.append(_u53(b[0], b[1]))
    cols.append(_u53(b[2], b[3]))
    return np.concatenate([np.full(2 * n, 0.5), np.stack(cols, axis=1).ravel()])


def pair_lists(ladders, replicas):
    """Candidate pairs (a, b, stat, flags) of even and of odd rounds, in the order pmc_set_ladders builds them."""
    pairs = ([], [])
    for lad in ladders:
        m = len(lad)
        for i in range(m - 1):
            for r in range(replicas):
                pairs[i & 1].append((lad[i] * replicas + r, lad[i + 1] * replicas + r, lad[i],
                                     (1 if i == 0 else 0) | (2 if i + 2 == m else 0)))
    return pairs


class Exchange:
    """The bookkeeping of pmc_set_ladders / pmc_exchange: candidate pairs, round counter, pair statistics, walker
    labels and round trips of a handle of `nchains` chains, `ncases` cases × `replicas`."""

    def __init__(self, ncases, replicas, chain_id_base=0):
        self.ncases, self.R, self.base = int(ncases), int(replicas), int(chain_id_base)
        self.nchains = self.ncases * self.R
        self.set_ladders([])

    def set_ladders(self, ladders):
        self.pairs = pair_lists(ladders, self.R)
        self.round = 0
        self.stats = np.zeros((self.ncases, 2), dtype=np.int64)
        self.walker = np.arange(self.nchains, dtype=np.int64) + self.base
        self.wstate = np.zeros(self.nchains, dtype=np.int64)
        for lad in ladders:
            self.wstate[lad[0] * self.R:(lad[0] + 1) * self.R] = 1
        self.trips = np.zeros(self.nchains, dtype=np.int64)

    def _arrive(self, walker, bottom, top):
        w = walker - self.base
        if bottom:
            if self.wstate[w] == 2:
                self.trips[w] += 1
            self.wstate[w] = 1
        elif top and self.wstate[w] == 1:
            self.wstate[w] = 2

    def round_pairs(self):
        return self.pairs[self.round & 1]

    def record(self, a, b, stat, flags, take):
        """Count one attempt of pair (a, b) and, if taken, move the walker labels."""
        self.stats[stat, 0] += 1
        if take:
            self.stats[stat, 1] += 1
            wa, wb = self.walker[a], self.walker[b]
            self.walker[a], self.walker[b] = wb, wa
            self._arrive(wb, flags & 1, False)
            self._arrive(wa, False, flags & 2)


class Ladders(Exchange):
    """One oracle Run per chain of a handle (case c // replicas, global id chain_id_base + c) and the exchange rounds
    of pmc_exchange on them."""

    def __init__(self, cases, replicas, seed, chain_id_base=0, algo=1, tape_steps=0, rng=None):
        """tape_steps > 0: every Run is fed from a tape of that many trials, continued across steps() calls —
        the library's Philox draws (philox_tape, initial chains as the library draws them) or, given a numpy
        Generator `rng`, plain uniforms (a statistically equivalent sampler with its own random numbers)."""
        self.cases, self.seed = list(cases), int(seed)
        super().__init__(len(self.cases), replicas, chain_id_base)
        self.runs = []
        for c in range(self.nchains):
            case, cid = self.cases[c // self.R], self.base + c
            if not tape_steps:
                self.runs.append(O.Run(case, self.seed, cid, algo))
                continue
            per = 3 + bool(case.do_flips) + (not case.planar)
            tape = (rng.random(2 * int(case.n) + per * tape_steps) if rng is not None
                    else philox_tape(case, self.seed, cid, 0, 0, tape_steps))
            run = O.Run(case, self.seed, cid, algo, tape=tape)
            if rng is None:
                run.set_state(*O.draw_init(self.seed, cid, 0, int(case.n)))
            self.runs.append(run)
        self.kT = [float(self.cases[c // self.R].kT) for c in range(self.nchains)]
        self.init = [0] * self.nchains

    def begin_stage(self, kT_scale):
        for c, run in enumerate(self.runs):
            self.kT[c] = float(self.cases[c // self.R].kT) * kT_scale
            run.begin_stage(self.kT[c])
            self.init[c] += 1

    def exchange(self):
        """One round; -> accepted [chains] (1 at the lower slot of every accepted pair)."""
        acc = np.zeros(self.nchains, dtype=np.int32)
        for a, b, stat, flags in self.round_pairs():
            ra, rb = self.runs[a], self.runs[b]
            ca, cb = self.cases[a // self.R], self.cases[b // self.R]
            delta, _, _ = exchange_delta(self.kT[a], self.kT[b], ra.diag()["U"], rb.diag()["U"], ra.chain().r(),
                                         rb.chain().r(), ca.Fx, ca.Fz, cb.Fx, cb.Fz)
            take = delta >= 0.0 or draw_exchange_eps(self.seed, self.base + a, self.init[a], self.round) < math.exp(delta)
            self.record(a, b, stat, flags, take)
            if take:
                acc[a] = 1
                xa, xb = ra.chain().state(), rb.chain().state()
                ra.set_state(*xb)
                rb.set_state(*xa)
        self.round += 1
        return acc
