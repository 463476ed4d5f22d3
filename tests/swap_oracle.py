"""Population MCMC for the tests (TEST INFRASTRUCTURE ONLY, not part of the product).

* `swap_round`: the numpy statement of the swap contract shared with csrc/phf_swap.cu (phf_am_single_swap; not in the
  reference -- Calderhead & Girolami 2009, Friel & Pettitt 2008):
    ladder   T chain slots of one dataset, temperatures t_0 < t_1 < ... (each slot keeps its temperature);
    schedule the round after iteration t = sK (K = swap interval, s = 1, 2, ...) tries the disjoint pairs (k, k+1)
             with k = s (mod 2) -- `parity`;
    accept   iff ln u < (t_k - t_k+1) (l1(x_k+1) - l1(x_k)) with the temperature-1 log-likelihoods stored in the two
             state rows (the prior cancels); a non-finite l1 on either side rejects.  u = uniform53 of words 0, 1 of
             philox_call(seed, ladder_id, t, SWAP_CALL0 + k), ladder_id a global id of the ladder;
    accepted theta moves between the slots, and each slot's (log_target, l1) is re-evaluated for its new theta at its
             own temperature.  Adaptation state (mean, cov, loga), the l1 sum and the accept count stay with the slot.
* `c_swap_round` / `c_ladder_run`: ctypes binding of the C statement, tests/native/swap_oracle.c, which runs whole
  ladders on top of the C oracle of the sampler (oracle/hill_oracle.c: phf_oracle_am_single per slot, then the round).
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np

from c_oracle import classify, state_size
from hill_oracle import philox_call, uniform53

SWAP_CALL0 = 0x80000000

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "native", "swap_oracle.c")
_SO = os.path.join(_HERE, "native", "libswap_oracle.so")
_lib = None


def swap_round(states, temps, ladder, d, seed, ladder_id, t, parity, target, counts=None):
    """One swap round of one ladder.  states: [n, >= d+2] rows (theta[d], log_target, l1, ...), changed in place;
    temps [n]; ladder: the T row indices; target(theta, temperature) -> (log_target, l1); counts: [T-1, 2]
    (attempted, accepted), accumulated, or None."""
    for k in range(parity, len(ladder) - 1, 2):
        a, b = ladder[k], ladder[k + 1]
        w = philox_call(seed, ladder_id, t, SWAP_CALL0 + k)
        la, lb = states[a, d + 1], states[b, d + 1]
        accepted = bool(np.isfinite(la) and np.isfinite(lb)
                        and math.log(uniform53(w[0], w[1])) < (temps[a] - temps[b]) * (lb - la))
        if counts is not None:
            counts[k, 0] += 1
            counts[k, 1] += accepted
        if accepted:
            tha, thb = states[b, :d].copy(), states[a, :d].copy()
            states[a, :d], states[b, :d] = tha, thb
            states[a, d], states[a, d + 1] = target(tha, temps[a])
            states[b, d], states[b, d + 1] = target(thb, temps[b])




def build():
    """tests/native/libswap_oracle.so with the flags of oracle/Makefile (no fast-math, no FMA contraction)"""
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=gnu11", "-fno-fast-math", "-ffp-contract=off", "-shared", "-o",
                           _SO, _SRC, "-lm", "-lpthread"])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        _dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
        _u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
        _i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
        L.phf_oracle_swap_round.restype = None
        L.phf_oracle_swap_round.argtypes = [C.c_int, C.c_int, _dp, _dp, _u8p, C.c_double, C.c_int, _i64p, _dp, _dp,
                                            C.c_int, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_void_p]
        L.phf_oracle_ladder_run.restype = C.c_int
        L.phf_oracle_ladder_run.argtypes = [C.c_int, C.c_int, _dp, _dp, _u8p, C.c_double, C.c_int, _dp, _dp, C.c_uint32,
                                            C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint64,
                                            np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS"), C.c_uint64,
                                            C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int64, C.c_void_p]
        _lib = L
    return _lib


def c_swap_round(model, concs, responses, pi_bit, slots, temps, states, seed, ladder_id, t, parity, counts=None,
                 cls=None):
    """One swap round of the ladder `slots` (chain indices into the rows of `states`, changed in place; `temps` per
    row).  counts: int64 [T-1, 2] (attempted, accepted), accumulated, or None."""
    concs = np.ascontiguousarray(concs, dtype=np.float64)
    responses = np.ascontiguousarray(responses, dtype=np.float64)
    cls = classify(responses) if cls is None else cls
    slots = np.ascontiguousarray(slots, dtype=np.int64)
    assert states.flags.c_contiguous and states.dtype == np.float64
    lib().phf_oracle_swap_round(model, len(concs), concs, responses, cls, float(pi_bit), len(slots), slots,
                                np.ascontiguousarray(temps, dtype=np.float64), states, states.shape[1], seed, ladder_id,
                                t, parity, None if counts is None else counts.ctypes.data)


def c_ladder_run(model, concs, responses, pi_bit, temps, states, t0, iters, thinning, adapt_when, reset_mean, seed,
                 chain_ids, ladder_id, swap_every, burn=0xFFFFFFFF, want_chain=True, counts=None, cls=None):
    """T slots of one dataset (oracle state rows `states` [T, state_size(d)], changed in place) run with swaps every
    `swap_every` iterations.  Returns the rows saved by the call, [T, rows, d+1] (or None)."""
    concs = np.ascontiguousarray(concs, dtype=np.float64)
    responses = np.ascontiguousarray(responses, dtype=np.float64)
    cls = classify(responses) if cls is None else cls
    d = 2 if model == 1 else 3
    T = len(temps)
    row0 = t0 // thinning + 1
    nrows = (t0 + iters) // thinning - t0 // thinning
    chain = np.zeros((T, nrows, d + 1)) if want_chain else None
    assert states.shape == (T, state_size(d)) and states.flags.c_contiguous
    rc = lib().phf_oracle_ladder_run(model, len(concs), concs, responses, cls, float(pi_bit), T,
                                     np.ascontiguousarray(temps, dtype=np.float64), states, t0, iters, thinning,
                                     adapt_when, int(reset_mean), seed, np.ascontiguousarray(chain_ids, dtype=np.uint64),
                                     ladder_id, swap_every, row0, burn, chain.ctypes.data if want_chain else None, nrows,
                                     None if counts is None else counts.ctypes.data)
    if rc:
        raise RuntimeError("oracle ladder run failed (%d)" % rc)
    return chain
