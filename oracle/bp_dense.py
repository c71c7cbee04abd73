"""Independent dense transliteration of the reference decode! (TEST INFRASTRUCTURE ONLY).

A second, deliberately naive restatement used to cross-check oracle/bp_oracle.c on small
cases: dense s x n float64 matrices, 1:1 with
/root/reference/src/decoders/belief_propagation.jl:121-188 (same loop nests, same operand order).
Pure-Python loops -> small cases only.
"""
import numpy as np


def decode_dense(H, per, max_iters, syndrome):
    """Returns (err float64[n] of 0.0/1.0, converged bool, ratio float64[n], iters int)."""
    H = np.asarray(H).astype(np.int64)
    s, n = H.shape
    f = np.float64
    one, two = f(1.0), f(2.0)
    per = f(per)
    rows_of_col = [np.nonzero(H[:, j])[0] for j in range(n)]   # rowvals/nzrange of sparse_H
    cols_of_row = [np.nonzero(H[i, :])[0] for i in range(s)]   # rowvals/nzrange of sparse_HT
    # reset! (:83-91)
    log_ratio = np.ones(n, dtype=f)
    channel = np.full(n, per, dtype=f)
    b2c = np.zeros((s, n), dtype=f)
    c2b = np.zeros((s, n), dtype=f)
    err = np.zeros(n, dtype=f)
    with np.errstate(all="ignore"):
        for j in range(n):                                       # :127-131
            for i in rows_of_col[j]:
                b2c[i, j] = channel[j] / (one - channel[j])
        converged = False
        iters = 0
        for it in range(1, max_iters + 1):                       # :134
            iters = it
            for i in range(s):                                   # :135-150
                temp = f(-1.0) if int(syndrome[i]) % 2 else one  # (-1)^syndrome[i]
                for j in cols_of_row[i]:
                    c2b[i, j] = temp
                    temp = temp * (two / (one + b2c[i, j]) - one)
                temp = one
                for j in cols_of_row[i][::-1]:
                    c2b[i, j] = c2b[i, j] * temp
                    c2b[i, j] = (one - c2b[i, j]) / (one + c2b[i, j])
                    temp = temp * (two / (one + b2c[i, j]) - one)
            for j in range(n):                                   # :152-178
                temp = channel[j] / (one - channel[j])
                for i in rows_of_col[j]:
                    b2c[i, j] = temp
                    temp = temp * c2b[i, j]
                    if np.isnan(temp):
                        temp = one
                log_ratio[j] = temp                              # reference keeps log(1/temp)
                err[j] = 1.0 if temp >= 1 else 0.0
                temp = one
                for i in rows_of_col[j][::-1]:
                    b2c[i, j] = b2c[i, j] * temp
                    temp = temp * c2b[i, j]
                    if np.isnan(temp):
                        temp = one
            decoded = (H @ err.astype(np.int64)) % 2             # :180
            if np.all(decoded == np.asarray(syndrome).astype(np.int64)):   # :181
                converged = True
                break
    return err, converged, log_ratio, iters


def brute_force_ratio(H, per, syndrome):
    """Exact posterior ratios P(e_j=1|s)/P(e_j=0|s) by enumeration (n <= ~20).
    BP is exact on cycle-free Tanner graphs, so this is a known-answer test there."""
    H = np.asarray(H).astype(np.int64)
    s, n = H.shape
    syndrome = np.asarray(syndrome).astype(np.int64)
    p1 = np.zeros(n)
    p0 = np.zeros(n)
    for m in range(1 << n):
        e = np.array([(m >> j) & 1 for j in range(n)], dtype=np.int64)
        if np.any((H @ e) % 2 != syndrome):
            continue
        w = int(e.sum())
        pr = per ** w * (1 - per) ** (n - w)
        p1 += pr * e
        p0 += pr * (1 - e)
    with np.errstate(all="ignore"):
        return p1 / p0


def osd0_dense(H, syndrome, bp_err, ratio, return_pivots=False):
    """Dense transliteration of decode!(::BeliefPropagationOSDDecoder) after the BP call
    (belief_propagation_osd.jl:52-60) and of osd(..., Val(0)) (:63-125), numpy bool matrices, physical
    row swaps, same loop order.  r = 1/R replaces exp(log(1/R)) exactly as in bp_oracle.c.
    With return_pivots: (result, number of pivots used)."""
    H = np.asarray(H).astype(bool)
    m, n = H.shape
    with np.errstate(all="ignore"):
        r = np.float64(1.0) / np.asarray(ratio, dtype=np.float64)
        key = np.maximum(r, np.float64(1.0) - r)
    order = sorted(range(n), key=lambda j: (-key[j], j))          # stable sortperm(..., rev=true)
    Hs = H[:, order].copy()
    e = np.asarray(bp_err).astype(np.int64)[order]
    t = np.asarray(syndrome).astype(bool).copy()                  # :66
    for j in range(n):
        if e[j] == 1:
            t ^= Hs[:, j]
    rows, cols = [], []
    if not t.any():
        corr = e.astype(bool)
    else:
        Hw = Hs.copy()
        rows, cols = [], []
        i = 0
        for j in range(n):
            if i >= m or not t[i:].any():
                break
            nz = np.nonzero(Hw[i:, j])[0]
            if nz.size:
                k = int(nz[0])
                if e[j] == 1:
                    t ^= Hw[:, j]
                if k > 0:
                    ii = i + k
                    Hw[[i, ii], :] = Hw[[ii, i], :]
                    t[i], t[ii] = t[ii], t[i]
                for ii in range(i + 1, m):
                    if Hw[ii, j]:
                        Hw[ii, :] ^= Hw[i, :]
                        t[ii] ^= t[i]
                rows.append(i)
                cols.append(j)
                i += 1
        corr = e.astype(bool).copy()
        for rr, c in zip(rows[::-1], cols[::-1]):
            corr[c] = t[rr]
            if corr[c]:
                for ii in range(rr):
                    if Hw[ii, c]:
                        t[ii] ^= True
    out = np.zeros(n, dtype=np.uint8)
    out[np.asarray(order)] = corr.astype(np.uint8)
    return (out, len(rows)) if return_pivots else out


def osdk_dense(H, syndrome, bp_err, ratio, osd_order):
    """Dense transliteration of osd(H_sorted, syndrome, bp_err_sorted, Val{O}) for O > 0
    (belief_propagation_osd.jl:127-209) behind the sort of :53-57 and the un-permutation of :60."""
    H = np.asarray(H).astype(bool)
    m, n = H.shape
    with np.errstate(all="ignore"):
        r = np.float64(1.0) / np.asarray(ratio, dtype=np.float64)
        key = np.maximum(r, np.float64(1.0) - r)
    order = sorted(range(n), key=lambda j: (-key[j], j))
    Hs = H[:, order].copy()
    e = np.asarray(bp_err).astype(np.int64)[order]
    s = np.asarray(syndrome).astype(bool).copy()
    rows, cols = [], []
    i = j = 0
    while i < m and j < n:
        nz = np.nonzero(Hs[i:, j])[0]
        if nz.size == 0:
            j += 1
            continue
        k = int(nz[0])
        if k > 0:
            ii = i + k
            Hs[[i, ii], :] = Hs[[ii, i], :]
            s[i], s[ii] = s[ii], s[i]
        for ii in range(i + 1, m):
            if Hs[ii, j]:
                Hs[ii, :] ^= Hs[i, :]
                s[ii] ^= s[i]
        rows.append(i)
        cols.append(j)
        i += 1
        j += 1
    for pi, pj in zip(rows[::-1], cols[::-1]):
        for ii in range(pi):
            if Hs[ii, pj]:
                Hs[ii, :] ^= Hs[pi, :]
                s[ii] ^= s[pi]
    rk = len(rows)
    osd_order = min(osd_order, n - rk)
    err = e.astype(bool).copy()
    best = err.copy()
    mrc = [c for c in range(n) if c not in set(cols)]
    min_w = n + 1
    for x in range(1 << osd_order):
        if x != 0:
            for b in range(osd_order):
                err[mrc[b]] = bool((x >> b) & 1)
        for pi, pj in zip(rows, cols):
            v = bool(s[pi])
            for c in mrc:
                v ^= bool(Hs[pi, c]) and bool(err[c])
            err[pj] = v
        w = int(err.sum())
        if w < min_w:
            min_w = w
            best = err.copy()
    out = np.zeros(n, dtype=np.uint8)
    out[np.asarray(order)] = best.astype(np.uint8)
    return out
