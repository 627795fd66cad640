"""Exact references of the two interpolations, in mpmath at 40 significant digits.

IDW restates the per-step weighted mean of oracle/sho_region.hpp:140-168 (core/inverse_distance.h:214-249) from the oracle's float64
neighbour lists and weights.  BTK restates build_covariance_matrices, build_operators and the per-step update of
oracle/sho_region.hpp:261-346 (core/bayesian_kriging.h:93-125,280-402).  Both are evaluated on a sample of cells and steps only
(sample_cells, sample_steps): the point is an answer whose own error is far below a float64 ulp, so that a kernel or the oracle can be
measured against it, not speed.

The BTK restatement solves with K by a Cholesky factorisation (K is a covariance matrix) instead of forming K^-1; the quantities are the
same: K^-1 F, omega = k' K^-1 (K symmetric, so omega[c] = K^-1 k[:, c]), H = (F' K^-1 F)^-1, G = (H^-1 + diag(0, 1/sd^2))^-1,
E_beta_w = H F' K^-1 and BM = (f - F' K^-1 k)' (I - G H^-1).
"""
import numpy as np
from mpmath import mp, mpf

DPS = 40
U = 2.0**-53                 # unit round-off of float64
KINDS = ("temperature", "precipitation", "radiation", "wind_speed", "rel_hum")


def _edges_first(n, limit):
    """cells on either side of the interpolation kernels' tile edges (8-cell groups, 8*NT-cell warp tiles, 32*NT-cell blocks), the
    coarse edges first, then the start of every ragged tail"""
    order = []
    for e in (128, 64, 32, 16, 8):
        order += [k * e for k in range(1, (n - 1) // e + 1)]
        if n % e:
            order.append(n - n % e)
    seen, out = set(), []
    for e in order:
        if 0 < e < n and e not in seen:
            seen.add(e)
            out.append(e)
    return out[:limit]


def sample_cells(n, limit=64):
    """at most `limit` cells: all of them when they fit, else the first and last two and both sides of tile edges"""
    if n <= limit:
        return np.arange(n)
    picks = {0, 1, n - 2, n - 1}
    for e in _edges_first(n, limit):
        if len(picks) + 2 > limit:
            break
        picks.update((e - 1, e))
    return np.array(sorted(picks))


def sample_steps(n_steps, limit=8):
    """at most `limit` steps of a launch of n_steps: first and last, and both sides of the 8-step row groups and of the 32- and
    64-step staging buffers"""
    cand = [0, n_steps - 1, 7, 8, 31, 32, 63, 64, 65, 127, 128, 255, 256, 511, 512, n_steps - 2]
    out = []
    for s in cand:
        if 0 <= s < n_steps and s not in out:
            out.append(s)
    return np.array(sorted(out[:limit]), dtype=np.int64)


# ---- inverse distance weighting ------------------------------------------------------------------------------------------------------
def _solve3_exact(A, b):
    """the gradient of temperature_gradient_scale_computer's 3x3 plane fit, exactly; None when singular"""
    try:
        return mp.lu_solve(mp.matrix(A), mp.matrix(b))
    except ZeroDivisionError:
        return None


def idw_exact(oracle, kind, src_xyz, values, dst_xyz, par, cells, steps, dst_slope=None):
    """-> (exact, magnitude), both [len(steps)][len(cells)].

    exact = sum_j w_j tv_j / sum_j w_j over the finite neighbours of the oracle's list (NaN when none is finite), tv the per-variable
    transform of sho_region.hpp:146-162.  magnitude = sum_j w_j (|v_j f_j| + G |z_c - h_j|) / sum_j w_j, with G the size of the
    temperature gradient (|v_hi| + |v_lo|) / dz when it comes from the span of the neighbours, |gradient| otherwise, 0 for the other
    variables: it bounds sum_s |W_cs v_ts| of the dense operator (sb2_interp.cuh, idw_build_dense_kernel), and float64 evaluation of
    either form is off by a small multiple of U times it."""
    mp.dps = DPS
    src_xyz, dst_xyz, values = np.asarray(src_xyz, float), np.asarray(dst_xyz, float), np.asarray(values, float)
    cells, steps = np.asarray(cells), np.asarray(steps)
    idx, w, cnt = oracle.idw_neighbours(src_xyz, dst_xyz[cells], par)
    default_gradient, by_equation, scale = mpf(par[4]), bool(par[5]), mpf(par[6])
    exact = np.full((len(steps), len(cells)), np.nan)
    mag = np.full_like(exact, np.nan)
    for ci, c in enumerate(cells):
        nb = [(int(idx[ci, j]), mpf(w[ci, j])) for j in range(cnt[ci])]
        zc = mpf(dst_xyz[c, 2])
        factor = {}
        for k, _ in nb:
            if kind == "precipitation":
                factor[k] = mp.power(scale, (zc - mpf(src_xyz[k, 2])) / 100)
            elif kind == "radiation":
                factor[k] = mpf(dst_slope[c])
            else:
                factor[k] = mpf(1)
        for ti, t in enumerate(steps):
            v = values[t]
            fin = [(k, wk) for k, wk in nb if np.isfinite(v[k])]
            if not fin:
                continue
            g = G = mpf(0)
            if kind == "temperature":
                g, G = default_gradient, abs(default_gradient)
                solved = False
                if by_equation and len(fin) > 3:
                    p = [fin[r][0] for r in range(4)]
                    A = [[mpf(src_xyz[p[r + 1], i]) - mpf(src_xyz[p[0], i]) for i in range(3)] for r in range(3)]
                    b = [mpf(v[p[r + 1]]) - mpf(v[p[0]]) for r in range(3)]
                    x = _solve3_exact(A, b)
                    if x is not None:
                        g, G, solved = x[2], abs(x[2]), True
                if not solved and len(fin) > 1:
                    lo = hi = 0   # the first lowest and first highest neighbour in list order, as the reference picks them
                    for j, (k, _) in enumerate(fin):
                        h = src_xyz[k, 2]
                        if h < src_xyz[fin[lo][0], 2]:
                            lo = j
                        elif h > src_xyz[fin[hi][0], 2]:
                            hi = j
                    klo, khi = fin[lo][0], fin[hi][0]
                    dz = mpf(src_xyz[khi, 2]) - mpf(src_xyz[klo, 2])
                    if dz > 50:
                        g = (mpf(v[khi]) - mpf(v[klo])) / dz
                        G = (abs(mpf(v[khi])) + abs(mpf(v[klo]))) / dz
            sw = swv = smag = mpf(0)
            for k, wk in fin:
                vk = mpf(v[k])
                if kind == "temperature":
                    dzk = zc - mpf(src_xyz[k, 2])
                    tv, m = vk + g * dzk, abs(vk) + G * abs(dzk)
                else:
                    tv = vk * factor[k]
                    m = abs(tv)
                sw += wk
                swv += wk * tv
                smag += wk * m
            exact[ti, ci] = float(swv / sw)
            mag[ti, ci] = float(smag / sw)
    return exact, mag


# ---- Bayesian temperature kriging ---------------------------------------------------------------------------------------------------
def _cholesky(A):
    n = len(A)
    L = [[mpf(0)] * n for _ in range(n)]
    for j in range(n):
        Lj = L[j]
        d = mp.sqrt(A[j][j] - mp.fdot(Lj[:j], Lj[:j]))
        Lj[j] = d
        for i in range(j + 1, n):
            Li = L[i]
            Li[j] = (A[i][j] - mp.fdot(Li[:j], Lj[:j])) / d
    return L


def _cho_solve(L, b):
    n = len(L)
    y = [mpf(0)] * n
    for i in range(n):
        y[i] = (b[i] - mp.fdot(L[i][:i], y[:i])) / L[i][i]
    x = [mpf(0)] * n
    for i in reversed(range(n)):
        x[i] = (y[i] - mp.fdot([L[j][i] for j in range(i + 1, n)], x[i + 1:])) / L[i][i]
    return x


def _inv2(M):
    (a, b), (c, d) = M
    det = a * d - b * c
    return [[d / det, -b / det], [-c / det, a / det]]


def _mul2(A, B):
    return [[A[i][0] * B[0][j] + A[i][1] * B[1][j] for j in range(2)] for i in range(2)]


def _cov(p, q, sill_m_nug, range_, zscale):
    d = mp.sqrt((p[0] - q[0]) ** 2 + (p[1] - q[1]) ** 2 + ((p[2] - q[2]) * zscale) ** 2)
    return sill_m_nug * mp.exp(-d / range_)


def btk_exact(oracle, src_xyz, values, dst_xyz, t0_us, dt_us, cells, steps, gradient_sd=0.0025, sill=25.0, nug=0.5, range_=200000.0,
              zscale=20.0):
    """-> exact [len(steps)][len(cells)] of btk_interpolation (sho_region.hpp:309-346) at the given cells and steps.  The S x S
    algebra is done once per valid-station set met among `steps`; the prior gradient of a step is the oracle's."""
    mp.dps = DPS
    src_xyz, dst_xyz, values = np.asarray(src_xyz, float), np.asarray(dst_xyz, float), np.asarray(values, float)
    S = src_xyz.shape[0]
    smn, rng, zs, gsd = mpf(sill) - mpf(nug), mpf(range_), mpf(zscale), mpf(gradient_sd)
    P = [[mpf(x) for x in row] for row in src_xyz]
    C = [[mpf(x) for x in dst_xyz[c]] for c in cells]
    K = [[smn if i == j else None for j in range(S)] for i in range(S)]
    for i in range(S):
        for j in range(i + 1, S):
            K[i][j] = K[j][i] = _cov(P[i], P[j], smn, rng, zs)
    kfull = [[_cov(P[i], C[c], smn, rng, zs) for c in range(len(cells))] for i in range(S)]
    ops = {}

    def operators(valid):
        n = len(valid)
        L = _cholesky([[K[a][b] for b in valid] for a in valid])
        F = [[mpf(1), P[a][2]] for a in valid]
        KiF = list(zip(*[_cho_solve(L, [F[i][col] for i in range(n)]) for col in range(2)]))    # [n][2]
        H_inv = [[mp.fdot([F[i][r] for i in range(n)], [KiF[i][col] for i in range(n)]) for col in range(2)] for r in range(2)]
        H = _inv2(H_inv)
        G = _inv2([[H_inv[0][0], H_inv[0][1]], [H_inv[1][0], H_inv[1][1] + 1 / (gsd * gsd)]])
        GH = _mul2(G, H_inv)
        I_GH = [[(1 if r == col else 0) - GH[r][col] for col in range(2)] for r in range(2)]
        E_beta_w = [[H[r][0] * KiF[i][0] + H[r][1] * KiF[i][1] for i in range(n)] for r in range(2)]     # H F' K^-1
        omega, BM = [], []
        for c in range(len(cells)):
            y = _cho_solve(L, [kfull[a][c] for a in valid])                                      # K^-1 k_c
            d = [mpf(1) - mp.fsum(y), C[c][2] - mp.fdot([F[i][1] for i in range(n)], y)]       # f_c - F' K^-1 k_c
            omega.append(y)
            BM.append([d[0] * I_GH[0][col] + d[1] * I_GH[1][col] for col in range(2)])
        return F, E_beta_w, omega, BM

    out = np.full((len(steps), len(cells)), np.nan)
    for ti, t in enumerate(steps):
        valid = tuple(int(s) for s in np.flatnonzero(np.isfinite(values[t])))
        if not valid:
            raise RuntimeError("bayesian kriging temperature: No valid sources for time period, giving up.")
        if valid not in ops:
            ops[valid] = operators(valid)
        F, E_beta_w, omega, BM = ops[valid]
        T_obs = [mpf(values[t, s]) for s in valid]
        beta = [mp.fdot(E_beta_w[r], T_obs) for r in range(2)]
        resid = [T_obs[i] - (F[i][0] * beta[0] + F[i][1] * beta[1]) for i in range(len(valid))]
        prior = mpf(oracle.btk_prior_gradient(int(t0_us) + int(t) * int(dt_us), int(dt_us)))
        for ci in range(len(cells)):
            t_hat = beta[0] + C[ci][2] * beta[1] + mp.fdot(omega[ci], resid)
            out[ti, ci] = float(t_hat - (BM[ci][0] * beta[0] + BM[ci][1] * (beta[1] - prior)))
    return out


def segments(values):
    """[(first, end)] runs of steps with the same set of finite station values"""
    fin = np.isfinite(np.asarray(values, float))
    out, i = [], 0
    while i < fin.shape[0]:
        j = i + 1
        while j < fin.shape[0] and np.array_equal(fin[j], fin[i]):
            j += 1
        out.append((i, j))
        i = j
    return out


def btk_sample_steps(values, per_segment=8):
    """sample_steps of every segment of constant valid set, in absolute steps: each segment is one launch of the apply kernel"""
    return np.concatenate([a + sample_steps(b - a, per_segment) for a, b in segments(values)])
