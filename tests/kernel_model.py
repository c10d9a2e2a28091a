"""Executable model (numpy) of the ALGORITHM the CUDA kernels run for one frame.

It follows `csrc/sot_kernels.cuh` stage by stage -- merge-path partition per chunk, the sequential
walk with tie-group tracking, the one-slot peek across the chunk boundary, the look-back carry
for a tie group inherited from earlier chunks, the scatter of dL/dCDF to the source entries, the
two suffix scans and the normalisation chain rule -- so the algorithm can be checked against the
oracle on the CPU (tests/test_kernel_model.py) before and independently of any GPU run.
Differences in arithmetic detail that the GPU tests (not this model) pin down: the kernel forms
the CDF as fl32(prefix64 / mass) instead of cumsum64(fl32(a / mass)), forms the mass term
sum(gw * w) per thread as S_t * P_t + sum(ls * w) (P_t = the CDF-stage prefix of the thread), and cuts the
slots into odd-length chunks.  (The peek across the chunk boundary is the thread's own state after its
last advance -- the kernel needs no mailbox between chunks either.)  Test infrastructure only.
"""
import numpy as np

F32 = np.float32
PASS = F32(-1.0)  # carry marker: "my whole range belongs to a group opened before me"
EPS = F32(1e-7)


def merge_path(A, B, k):
    """Number of A entries among the first k outputs of the stable merge (A first on ties)."""
    n, m = len(A), len(B)
    lo, hi = max(0, k - m), min(k, n)
    while lo < hi:
        mid = (lo + hi) // 2
        if A[mid] <= B[k - 1 - mid]:
            lo = mid + 1
        else:
            hi = mid
    return lo


def cost(pa, pb, p):
    d = F32(pa) - F32(pb)
    if p == 2:
        return F32(d * d)
    if p == 1:
        return F32(abs(d))
    return F32(np.power(F32(abs(d)), F32(p)))


def walk_frame(cu, cv, pu, pv, p, limit, T, L, with_grad=True):
    """cu, cv: float32 CDF rows (non-decreasing). Returns loss (float64 sum of float32 partials),
    g_cu, g_cv (float32)."""
    n, m = len(cu), len(cv)
    K = n + m
    assert T * L >= K
    INF = F32(np.inf)
    A = np.concatenate((cu, [INF])).astype(F32)
    B = np.concatenate((cv, [INF])).astype(F32)
    PA = np.concatenate((pu, [pu[-1]])).astype(F32)  # clamp to last bin (losses.py:220)
    PB = np.concatenate((pv, [pv[-1]])).astype(F32)
    g = np.zeros(n + m, F32)  # scatter target: [0,n) -> u entries, [n, n+m) -> v entries
    carry_out = np.full(T, PASS, F32)
    fix_addr = np.full(T, -1, np.int64)
    partial = np.zeros(T, F32)

    for t in range(T):
        k0, k1 = min(t * L, K), min((t + 1) * L, K)
        if k0 >= K:
            continue
        i = merge_path(A[:n], B[:m], k0)
        j = k0 - i
        a, b = A[i], B[j]
        if k0 == 0:
            qprev = F32(0)
            md_prev = cost(PA[0], PB[0], p)  # virtual slot -1: value 0, counters (0, 0), never masked
            inherited = False
        else:
            qprev = max(A[i - 1] if i > 0 else F32(-np.inf), B[j - 1] if j > 0 else F32(-np.inf))
            md_prev = F32(0)   # unknown yet: resolved by look-back if the group closes in my range
            inherited = True
        acc = F32(0)
        src_prev = -1
        k = k0
        while True:
            if k < K:
                q = min(a, b)
                take_v = b < a
                same = (q == qprev)
                fresh = cost(PA[i], PB[j], p)
                masked = limit and (q > F32(1))
                md_k = md_prev if same else (F32(0) if masked else fresh)
            else:  # virtual slot K: always a new group with m*d = 0
                same, md_k = False, F32(0)
            if with_grad and k > k0:  # G of slot k-1 (the slot before k0 belongs to thread t-1)
                if same:
                    g[src_prev] = F32(0)
                else:
                    g[src_prev] = F32(md_prev - md_k)
                    if inherited:  # md_prev is still the placeholder 0: patch after look-back
                        fix_addr[t] = src_prev
            if not same:
                inherited = False  # the open group is now one that started in my range
            if k == k1:
                break
            dq = F32(q - qprev)
            if masked:
                dq = F32(0)
            acc = F32(acc + F32(dq * fresh))
            src_prev = (n + j) if take_v else i
            if take_v:
                j += 1
                b = B[j]
            else:
                i += 1
                a = A[i]
            qprev, md_prev = q, md_k
            k += 1
        carry_out[t] = PASS if inherited else md_prev
        partial[t] = acc

    # look-back: a thread whose inherited group closed inside its range adds the group's m*d
    if with_grad:
        for t in range(T):
            if fix_addr[t] >= 0:
                s = t - 1
                while carry_out[s] == PASS:
                    s -= 1
                g[fix_addr[t]] = F32(g[fix_addr[t]] + carry_out[s])
    return float(np.sum(partial.astype(np.float64))), g[:n].copy(), g[n:].copy()


def normalise(x, y, square, cut_scale):
    """Prologue as the kernel does it: squares in fp32, masses accumulated in fp64 and rounded to
    fp32, true fp32 division, CDF accumulated in fp64 and rounded per element."""
    a = (x * x).astype(F32) if square else x.astype(F32)
    b = (y * y).astype(F32) if square else y.astype(F32)
    Ma = F32(np.sum(a.astype(np.float64)))
    Mb = F32(np.sum(b.astype(np.float64)))
    Ma_c = EPS if Ma <= EPS else Ma
    Mb_c = EPS if Mb <= EPS else Mb
    den_v = Ma_c if cut_scale else Mb_c
    wu = (a / Ma_c).astype(F32)
    wv = (b / den_v).astype(F32)
    cu = np.cumsum(wu.astype(np.float64)).astype(F32)
    cv = np.cumsum(wv.astype(np.float64)).astype(F32)
    return a, b, Ma, Mb, Ma_c, den_v, wu, wv, cu, cv


def frame_loss_and_grads(x, y, pu, pv, p, square, cut_scale, limit, T, L):
    a, b, Ma, Mb, Ma_c, den_v, wu, wv, cu, cv = normalise(x, y, square, cut_scale)
    loss, g_cu, g_cv = walk_frame(cu, cv, pu, pv, p, limit, T, L)
    # suffix scans, the two weighted sums and the subtraction stay in fp64 (cancellation-prone),
    # one rounding to fp32 at the end
    g_wu = np.cumsum(g_cu[::-1].astype(np.float64))[::-1]
    g_wv = np.cumsum(g_cv[::-1].astype(np.float64))[::-1]
    su = np.sum(g_wu * wu.astype(np.float64))
    sv = np.sum(g_wv * wv.astype(np.float64))
    cu_corr = (su + sv if cut_scale else su) if Ma > EPS else 0.0
    cv_corr = sv if ((not cut_scale) and Mb > EPS) else 0.0
    ga = ((g_wu - cu_corr).astype(F32) / Ma_c).astype(F32)
    gb = ((g_wv - cv_corr).astype(F32) / den_v).astype(F32)
    gx = (F32(2) * x * ga).astype(F32) if square else ga
    gy = (F32(2) * y * gb).astype(F32) if square else gb
    return loss, gx, gy, cu, cv, g_cu, g_cv


def cdf_segments(per_thread):
    """Segment boundaries of a thread's local prefix sums (csrc/sot_device.cuh: cdf_segments, seg_begin)."""
    nseg = 4 if per_thread >= 25 else 1
    return [(per_thread * s) // nseg for s in range(nseg + 1)]


def cdf_stage_model(x, threads, per_thread, mass_floor=EPS, square=True, inv64=None, return_inv=False, tile=None,
                    exact_end=False):
    """Model of the CDF stage of both kernels (csrc/sot_device.cuh: cdf_scale, cdf_entries) for one row `x`
    (float32), vectorised over the threads: thread t owns bins [t*E, t*E+E), cut into segments (one for E < 25, four
    for 33 bins); fp32 prefix sums restart in every segment (x^2 fused into the add); a thread's sum = fp32 sum of its
    segment sums; the per-thread sums are added up in fp64 -> exclusive offsets (with `tile`: a scan within each tile of
    that many threads plus the fp64 carry of the tiles before, as the split-frame kernel does); entry =
    fl32(head + fl32(prefix * inv32 + ride)) where (head, tail) is the fp32 split of offset * inv64 and `ride` is the
    tail in the first segment, afterwards the fl32(prefix * inv32 + ride) of the previous segment's last entry; every
    entry is capped by the next thread's head.  `exact_end`: the row end is fl32(mass * inv64), never below the entry
    before it (the split-frame kernel).  Returns the float32 CDF row.  (fl32(x*x + acc) is formed in float64 and
    rounded once: x*x is exact there.)  `inv64`: 1/mass to scale by (cutoff mode scales the target row by the
    prediction's); default: this row's own (`return_inv`: also return the 1/mass used and the fp64 mass)."""
    n = len(x)
    E = per_thread
    bounds = cdf_segments(E)
    xs = np.zeros(threads * E, np.float64)
    xs[:n] = np.asarray(x, np.float32).astype(np.float64)
    xs = xs.reshape(threads, E)
    local = np.zeros((threads, E), np.float32)
    totals = np.zeros(threads, np.float32)
    for s in range(len(bounds) - 1):
        acc = np.zeros(threads, np.float32)
        for c in range(bounds[s], bounds[s + 1]):
            v = xs[:, c]
            acc = ((v * v if square else v) + acc.astype(np.float64)).astype(np.float32)
            local[:, c] = acc
        totals = acc if len(bounds) == 2 else (totals + acc).astype(np.float32)
    tile = threads if tile is None else tile
    offsets = np.zeros(threads + 1)  # offsets[t] exclusive, offsets[threads] = total
    carry = 0.0
    for t0 in range(0, threads, tile):
        excl = np.concatenate(([0.0], np.cumsum(totals[t0:t0 + tile].astype(np.float64))))
        offsets[t0:t0 + len(excl)] = carry + excl
        carry = carry + excl[-1]
    mass = F32(offsets[-1])
    if inv64 is None:
        inv64 = 1.0 / np.float64(mass if mass > mass_floor else mass_floor)
    inv32 = np.float64(F32(inv64))
    base = offsets[:-1] * inv64
    head = base.astype(np.float32).astype(np.float64)
    ride = (base - head).astype(np.float32)
    cap = (offsets[1:] * inv64).astype(np.float32)
    out = np.zeros((threads, E), np.float32)
    for s in range(len(bounds) - 1):
        inner = ride
        for c in range(bounds[s], bounds[s + 1]):
            inner = (local[:, c].astype(np.float64) * inv32 + ride.astype(np.float64)).astype(np.float32)  # one FFMA
            out[:, c] = np.minimum((head + inner.astype(np.float64)).astype(np.float32), cap)
        ride = inner
    out = out.reshape(-1)[:n].copy()
    if exact_end:
        out[-1] = max(F32(offsets[-1] * inv64), out[-2] if n > 1 else F32(0))
    return (out, inv64, offsets[-1]) if return_inv else out
