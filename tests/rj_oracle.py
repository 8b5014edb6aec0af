"""Float64 NumPy restatement of the reversible-jump moves of multi_gym.run_RHMC (reference sampler_RHMC.py:1009-1198,
1200-1445; drop-in hmc_stellar_toy_model_b200/sampler_RHMC.py _run_RHMC_rj, birth_death_move, split_merge_move), built on
the oracle's rhmc_step, potential, metric and kinetic.  It is the checker of field_kernel MODE_RUN_RJ (csrc/field_rj.cuh)
and of the device draw records (csrc/rj_draws.cuh); tests/golden/rj_chain.npz pins it to the unmodified reference.

The proposals take already-mapped values (indices, share, offsets, normals) and return (table_q, table_p, log_ratio) with
tables of shape (N, 3).  rj_run takes a draw provider: LegacyDraws consumes the global np.random stream in the reference's
order, DeviceDraws maps the device records with the kernel's rules.  Where the reference raises (a death or split with no
star, a merge with fewer than two stars or all pair weights zero, a proposal needing more than n_max stars) rj_run rejects
the jump with the state unchanged, as the kernel does."""
from __future__ import annotations

import numpy as np
from scipy.stats import beta as BETA

import stellar_oracle as so

KERNEL_RECORD = 14  # doubles of one device draw record


def _T(S, q3, p3):
    return so.kinetic(np.asarray(p3, float), so.metric(S, np.asarray(q3, float)))


def _momentum(S, q3, z):
    return np.asarray(z, float) * np.sqrt(so.metric(S, np.asarray(q3, float)))


def rj_birth(S, tq, tp, row, col, flux, z):
    """Newborn (flux, row, col) appended last (sampler_RHMC.py:1200-1240)."""
    new = np.array([flux, row, col])
    mom = _momentum(S, new, z)
    lr = S.alpha * np.log(flux) - 3 / 2. + _T(S, new, mom) + S.prior_const()
    return np.vstack([tq, new]), np.vstack([tp, mom]), lr


def rj_death(S, tq, tp, victim):
    """Row `victim` removed, the others keep their order (sampler_RHMC.py:1241-1273)."""
    lr = -S.alpha * np.log(tq[victim, 0]) + 3 / 2. - _T(S, tq[victim], tp[victim]) - S.prior_const()
    return np.delete(tq, victim, axis=0), np.delete(tp, victim, axis=0), lr


def rj_split(S, tq, tp, parent, off_r, off_c, share, z1, z2, K, a, b):
    """The parent becomes child one in place, child two is appended (sampler_RHMC.py:1276-1360)."""
    tq, tp = np.array(tq, copy=True), np.array(tp, copy=True)
    f, r, c = tq[parent]
    one = np.array([share * f, r + (1 - share) * off_r, c + (1 - share) * off_c])
    two = np.array([(1 - share) * f, r - share * off_r, c - share * off_c])
    m1, m2 = _momentum(S, one, z1), _momentum(S, two, z2)
    T_children = so.kinetic(np.concatenate([m1, m2]), so.metric(S, np.concatenate([one, two])))
    lr = ((-3 / 2.) + np.log(f) - BETA.logpdf(share, a, b) + np.log(2 * np.pi * K ** 2)
          + ((off_r ** 2 + off_c ** 2) / (2 * K ** 2)) + T_children - _T(S, tq[parent], tp[parent]))
    tq[parent], tp[parent] = one, m1
    return np.vstack([tq, two]), np.vstack([tp, m2]), lr


def merge_weights(tq, K, a, b):
    """Unnormalised weight of every ordered pair (i, j): Beta density of f_j / (f_i + f_j), zero within 1e-6 of one half,
    times the Gaussian split kernel at the pair's separation (sampler_RHMC.py:1361-1400)."""
    flux, rows, cols = tq[:, 0], tq[:, 1], tq[:, 2]
    share = flux / (flux.reshape((-1, 1)) + flux)
    w = BETA.pdf(share, a, b)
    w[np.abs(share - 0.5) < 1e-6] = 0.
    sep_sq = (rows.reshape((-1, 1)) - rows) ** 2 + (cols.reshape((-1, 1)) - cols) ** 2
    return w * (np.exp(-sep_sq / (2. * K ** 2)) / (2. * np.pi * K ** 2))


def rj_merge(S, tq, tp, one, two, z, K, a, b):
    """Rows one and two removed, the merged star appended; it takes the share f_one / (f_one + f_two) while the pair's weight
    used f_two / (f_one + f_two) (sampler_RHMC.py:1401-1445)."""
    share = tq[one, 0] / (tq[one, 0] + tq[two, 0])
    gap_sq = (tq[one, 1] - tq[two, 1]) ** 2 + (tq[one, 2] - tq[two, 2]) ** 2
    fm = tq[one, 0] + tq[two, 0]
    merged = np.array([fm, share * tq[one, 1] + (1 - share) * tq[two, 1], share * tq[one, 2] + (1 - share) * tq[two, 2]])
    T_pair = so.kinetic(np.concatenate([tp[one], tp[two]]), so.metric(S, np.concatenate([tq[one], tq[two]])))
    mom = _momentum(S, merged, z)
    lr = ((3 / 2.) - np.log(fm) + BETA.logpdf(share, a, b) - np.log(2 * np.pi * K ** 2) - (gap_sq / (2 * K ** 2))
          - T_pair + _T(S, merged, mom))
    keep = np.ones(len(tq), dtype=bool)
    keep[[one, two]] = False
    return np.vstack([tq[keep], merged]), np.vstack([tp[keep], mom]), lr


# ------------------------------------------------------------------------------------------------ draw providers
class LegacyDraws:
    """The global np.random stream in the reference's order, drawn lazily (randn(3N) and randint(0, N) depend on N)."""

    def __init__(self, S, P_move):
        self.S, self.P_move = S, P_move

    def normals(self, l, n):
        return np.random.randn(3 * n)

    def move(self, l):
        return int(np.random.choice([0, 1, 2], p=self.P_move, size=1)[0])

    def grow(self, l):
        return bool(np.random.choice([True, False], p=[0.5, 0.5]))

    def birth(self, l):
        row = np.random.random() * (self.S.num_rows - 2.) + 1.
        col = np.random.random() * (self.S.num_cols - 2.) + 1.
        flux = so.pow_law_sample(self.S.alpha, self.S.fmin, self.S.fmax, np.random.random(size=1))[0]
        return row, col, flux, np.random.randn(3)

    def victim(self, l, n):
        return int(np.random.randint(0, n, size=1)[0])

    def split(self, l, n, K, a, b):
        parent = int(np.random.randint(0, n, size=1)[0])
        off_r, off_c = np.random.randn(2) * K
        share = BETA.rvs(a, b, size=1)[0]
        return parent, off_r, off_c, share, np.random.randn(3), np.random.randn(3)

    def merge(self, l, w):
        n2 = w.size
        pick = int(np.random.choice(range(n2), p=(w / np.sum(w)).ravel()))
        return pick, np.random.randn(3)

    def lnu(self, l):
        return np.log(np.random.random(1))[0]


class DeviceDraws:
    """Device records [L, 14] (philox_rj_draws) with normals [L, 3 n_max] and lnu [L] (philox_draws), mapped with the
    kernel's rules: np.random.choice's rule for the move, index = min(floor(u n), n - 1), row = u (R - 2) + 1, the
    power-law inverse CDF for the flux, and for a merge the first flat index whose cumulative weight exceeds u W."""

    def __init__(self, S, P_move, records, normals, lnu):
        self.S, self.rec, self.z, self.ln = S, np.asarray(records), np.asarray(normals), np.asarray(lnu)
        p = np.asarray(P_move, dtype=float)
        self.cdf = np.cumsum(p) / np.sum(p)

    def normals(self, l, n):
        return self.z[l, :3 * n]

    def move(self, l):
        u = self.rec[l, 0]
        return 0 if u < self.cdf[0] else (1 if u < self.cdf[1] else 2)

    def grow(self, l):
        return self.rec[l, 1] < 0.5

    def _index(self, l, n):
        return min(int(np.floor(self.rec[l, 2] * n)), n - 1)

    def birth(self, l):
        r = self.rec[l]
        S = self.S
        return (r[2] * (S.num_rows - 2.) + 1., r[3] * (S.num_cols - 2.) + 1., so.pow_law_sample(S.alpha, S.fmin, S.fmax, r[4]),
                r[8:11])

    def victim(self, l, n):
        return self._index(l, n)

    def split(self, l, n, K, a, b):
        r = self.rec[l]
        return self._index(l, n), r[5] * K, r[6] * K, r[7], r[8:11], r[11:14]

    def merge(self, l, w):
        flat = w.ravel()
        cum = np.cumsum(flat)
        hit = np.nonzero(cum > self.rec[l, 2] * cum[-1])[0]
        return int(hit[0] if hit.size else np.nonzero(flat > 0)[0][-1]), self.rec[l, 8:11]

    def lnu(self, l):
        return self.ln[l]


# ------------------------------------------------------------------------------------------------ the chain
def rj_run(S, q0, niter, nsteps, dt, P_move, draws, *, n_max, K_split=1., beta_a=2., beta_b=2., f_pos=True, delta=1e-6,
           counter_max=1000, rad=0):
    """multi_gym.run_RHMC with reversible-jump moves.  Returns a dict of q_chain, p_chain [L, 3 n_max] (zero past 3 N),
    E_chain, V_chain, T_chain, A_chain (bool), move_chain, N_chain, q_final (flat, live stars), overflow (-1 or the first
    iteration whose proposal needed more than n_max stars)."""
    S = S.clone(dt=dt)
    L = niter + 1
    out = dict(q_chain=np.zeros((L, 3 * n_max)), p_chain=np.zeros((L, 3 * n_max)), E_chain=np.zeros(L), V_chain=np.zeros(L),
               T_chain=np.zeros(L), A_chain=np.zeros(L, dtype=bool), move_chain=np.zeros(L, dtype=int),
               N_chain=np.zeros(L, dtype=int), overflow=-1)

    def leg(q, p):
        if q.size == 0:
            return q, p
        for _ in range(nsteps):
            q, p = so.rhmc_step(S, q, p, delta=delta, counter_max=counter_max, rad=rad)
        return q, p

    def energy(q, p):
        return so.potential(S, q, f_pos=f_pos, rad=rad) + (so.kinetic(p, so.metric(S, q)) if q.size else 0.0)

    q = np.array(q0, dtype=float)
    for l in range(L):
        n = q.size // 3
        p = draws.normals(l, n) * np.sqrt(so.metric(S, q)) if n else np.zeros(0)
        V0 = so.potential(S, q, f_pos=f_pos, rad=rad)
        T0 = so.kinetic(p, so.metric(S, q)) if n else 0.0
        E0 = V0 + T0
        out["q_chain"][l, :3 * n], out["p_chain"][l, :3 * n] = q, p
        out["V_chain"][l], out["T_chain"][l], out["E_chain"][l], out["N_chain"][l] = V0, T0, E0, n
        move = draws.move(l)
        if move == 0:
            q1, p1 = leg(q, p)
            dE = energy(q1, p1) - E0
            lnu = draws.lnu(l)
            if (dE < 0) or (lnu < -dE):
                out["A_chain"][l], q = True, q1
            continue
        grow = draws.grow(l)
        code = (1 if grow else 2) if move == 1 else (3 if grow else 4)
        out["move_chain"][l] = code
        if (code in (1, 3) and n + 1 > n_max) or (code in (2, 3) and n == 0) or (code == 4 and n < 2):
            if code in (1, 3) and n + 1 > n_max and out["overflow"] < 0:
                out["overflow"] = l
            continue
        q1, p1 = leg(q, p)
        tq, tp = q1.reshape(-1, 3), -p1.reshape(-1, 3)
        if code == 1:
            row, col, flux, z = draws.birth(l)
            tq, tp, lr = rj_birth(S, tq, tp, row, col, flux, z)
        elif code == 2:
            tq, tp, lr = rj_death(S, tq, tp, draws.victim(l, n))
        elif code == 3:
            par, off_r, off_c, share, z1, z2 = draws.split(l, n, K_split, beta_a, beta_b)
            tq, tp, lr = rj_split(S, tq, tp, par, off_r, off_c, share, z1, z2, K_split, beta_a, beta_b)
        else:
            w = merge_weights(tq, K_split, beta_a, beta_b)
            if not (np.sum(w) > 0 and np.isfinite(np.sum(w))):
                continue
            pick, z = draws.merge(l, w)
            tq, tp, lr = rj_merge(S, tq, tp, pick // n, pick % n, z, K_split, beta_a, beta_b)
        q2, p2 = leg(tq.ravel(), tp.ravel())
        p2 = -p2
        ln_alpha = -(energy(q2, p2) - E0) + lr
        lnu = draws.lnu(l)
        if (ln_alpha > 0) or (lnu < ln_alpha):
            out["A_chain"][l], q = True, q2
    out["q_final"] = q
    return out


# ------------------------------------------------------------------------------------------------ device Beta sampler
def _box_muller(a, b, c, d, sine=False):
    rad = np.sqrt(-2.0 * np.log(so.philox_u01(a, b)))
    ang = 2.0 * np.pi * so.philox_u01(c, d)
    return rad * (np.sin(ang) if sine else np.cos(ang))


def gamma_philox(shape, seed, fid, l, domain, max_attempts=64):
    """Marsaglia-Tsang Gamma(shape) exactly as rj_draws.cuh draws it, vectorised over the arrays fid, l.  Attempt t takes its
    normal from word 2t and its uniform from word 2t + 1 of `domain`; shape < 1 is boosted with U^(1/shape), U from the last
    two words of word 1.  Returns (values, attempts)."""
    fid, l = np.broadcast_arrays(np.asarray(fid, dtype=np.uint64), np.asarray(l, dtype=np.uint64))
    boost = shape < 1.0
    d = (shape + 1.0 if boost else shape) - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * d)
    out = np.full(fid.shape, d)
    attempts = np.full(fid.shape, max_attempts)
    live = np.ones(fid.shape, dtype=bool)
    for t in range(max_attempts):
        if not live.any():
            break
        idx = np.nonzero(live)
        r = so.philox4x32_10(seed, np.uint64(2 * t), l[idx], fid[idx], np.uint64(domain))
        x = _box_muller(r[0], r[1], r[2], r[3])
        v = 1.0 + c * x
        ok = v > 0.0
        v = np.where(ok, v, 1.0) ** 3
        r = so.philox4x32_10(seed, np.uint64(2 * t + 1), l[idx], fid[idx], np.uint64(domain))
        u = so.philox_u01(r[0], r[1])
        x2 = x * x
        acc = ok & ((u < 1.0 - 0.0331 * (x2 * x2)) | (np.log(u) < 0.5 * x2 + d * (1.0 - v + np.log(v))))
        sel = tuple(a[acc] for a in idx)
        out[sel] = d * v[acc]
        attempts[sel] = t + 1
        live[sel] = False
    if boost:
        r = so.philox4x32_10(seed, np.uint64(1), l, fid, np.uint64(domain))
        out = out * so.philox_u01(r[2], r[3]) ** (1.0 / shape)
    return out, attempts


def beta_philox(a, b, seed, fid, l):
    """The split share of the device record: X / (X + Y), X ~ Gamma(a) (domain 5), Y ~ Gamma(b) (domain 6).  Returns
    (share, attempts of X, attempts of Y)."""
    x, nx = gamma_philox(a, seed, fid, l, 5)
    y, ny = gamma_philox(b, seed, fid, l, 6)
    return x / (x + y), nx, ny


def rj_records(seed, fids, L, a, b):
    """The device draw records [len(fids), L, 14] (csrc/rj_draws.cuh rj_record)."""
    fid = np.asarray(fids, dtype=np.uint64)[:, None] * np.ones((1, L), dtype=np.uint64)
    l = np.arange(L, dtype=np.uint64)[None, :] * np.ones((len(fids), 1), dtype=np.uint64)
    out = np.zeros(fid.shape + (KERNEL_RECORD,))
    for w, slots in ((0, (0, 1)), (1, (2, 3)), (2, (4,))):
        r = so.philox4x32_10(seed, np.uint64(w), l, fid, np.uint64(4))
        out[..., slots[0]] = so.philox_u01(r[0], r[1])
        if len(slots) > 1:
            out[..., slots[1]] = so.philox_u01(r[2], r[3])
    for blk, (s0, s1) in enumerate(((5, 6), (8, 9), (10, 11), (12, 13))):
        r = so.philox4x32_10(seed, np.uint64(3 + blk), l, fid, np.uint64(4))
        out[..., s0] = _box_muller(*r)
        out[..., s1] = _box_muller(*r, sine=True)
    out[..., 7] = beta_philox(a, b, seed, fid, l)[0]
    return out
