"""The Kimura two-parameter distance (--model K2P) on the CPU: the definition the device is checked against.

An extension of the oracle (oracle/apples_oracle.py), which stays as it is.  A K2P run is the oracle's own
observed_alignment(..., dist_fn=k2p, ...) followed by place_from_observed: the representatives, the two-phase rule, the
tie order (distance, index), the own-name removal, the zero-distance shortcut and the `<= 2` rule are upstream's, with
K2P in place of JC69.  With P and Q the fractions of transitions (A<->G, C<->T) and transversions among the valid sites
(neither row has '-'), the overlap gate of jc69, and

    d = -0.5 ln(1 - 2P - Q) - 0.25 ln(1 - 2Q),   missing (-1) when 1 - 2P - Q <= 0 or 1 - 2Q <= 0,   0 without differences.
"""
import numpy as np

PURINES = [b'A', b'G']


def k2p(a, b, overlap_frac):
    """a, b: 'S1' rows over A,C,G,T,- (same shape as oracle.jc69)"""
    both = np.logical_and(a != b'-', b != b'-')
    valid = np.count_nonzero(both)
    if not valid or valid / len(both) < overlap_frac:
        return -1.0
    diff = np.logical_and(a != b, both)
    pur_a, pur_b = np.isin(a, PURINES), np.isin(b, PURINES)
    ts = np.count_nonzero(diff & (pur_a == pur_b))        # A<->G or C<->T
    tv = np.count_nonzero(diff) - ts
    if ts + tv == 0:
        return 0.0
    P = ts * 1.0 / valid
    Q = tv * 1.0 / valid
    w1 = 1 - 2 * P - Q
    w2 = 1 - 2 * Q
    if 0 >= w1 or 0 >= w2:
        return -1.0                                       # missing, as jc69 does for loc <= 0
    return -0.5 * np.log(w1) - 0.25 * np.log(w2)


def k2p_counts(a, b):
    """(transitions, transversions, valid) site counts of two 'S1' rows"""
    both = np.logical_and(a != b'-', b != b'-')
    diff = np.logical_and(a != b, both)
    ts = int(np.count_nonzero(diff & (np.isin(a, PURINES) == np.isin(b, PURINES))))
    return ts, int(np.count_nonzero(diff)) - ts, int(np.count_nonzero(both))


def k2p_from_counts(ts, tv, valid, L, overlap_frac):
    """k2p evaluated from the integer counts (the same fp64 operations)"""
    if not valid or valid / L < overlap_frac:
        return -1.0
    if ts + tv == 0:
        return 0.0
    P = ts * 1.0 / valid
    Q = tv * 1.0 / valid
    w1 = 1 - 2 * P - Q
    w2 = 1 - 2 * Q
    if 0 >= w1 or 0 >= w2:
        return -1.0
    return -0.5 * np.log(w1) - 0.25 * np.log(w2)


def oracle_context(ci):
    """tests.util.CaseInputs.oracle_context with K2P as the distance: its runquery is a K2P run"""
    octx = ci.oracle_context()
    octx.dist_fn = k2p
    return octx

