"""numpy model of the planned psgd path (sparsepoly_b200/csrc/psgd_plan.cu), driven by the SAME plan arrays
the CUDA kernels read (sparsepoly_b200/psgd_plan.py).  Test infrastructure: it lets the CPU suite check the
plan layout (chunks, split columns, owner tables), the lazy (C, T) frame and the sharded pull / push /
owner protocol against the oracle without a GPU.  G ranks are simulated in one process; "peer memory" is
just the other rank's arrays."""
import numpy as np

CH = 64
SH = 8


def st_true(r, T, invC):
    m = np.abs(r) - T
    return np.where(m > 0, np.sign(r) * m * invC, 0.0)


def to_raw(v, T, Cn):
    return np.where(v == 0.0, 0.0, np.sign(v) * (np.abs(v) * Cn + T))


def dloss(loss, p, y):
    if loss == "squared":
        return p - y
    if loss == "logistic":
        z = p * y
        if z > 18.0:
            return -y * np.exp(-z)
        if z < -18.0:
            return -y
        return -y / (np.exp(z) + 1.0)
    z = 1.0 - p * y
    return (-2.0 * y) * z if z > 0 else 0.0


def lossv(loss, p, y):
    if loss == "squared":
        return 0.5 * (p - y) ** 2
    if loss == "logistic":
        z = p * y
        if z > 18.0:
            return np.exp(-z)
        if z < -18.0:
            return -z
        return np.log(1.0 + np.exp(-z))
    z = 1.0 - p * y
    return z * z if z > 0 else 0.0


def get_eta(lr, eta0, alpha, beta, power_t, it):
    if lr == "constant":
        return eta0, eta0
    if lr == "optimal":
        e = eta0 * it
        return eta0 / (1.0 + e * beta) ** power_t, eta0 / (1.0 + e * alpha) ** power_t
    if lr == "pegasos":
        return 1.0 / (beta * it), 1.0 / (alpha * it)
    e = eta0 / it ** power_t
    return e, e


def michelot(vals, strength):
    """fixed point tau = 2 s S(tau) / (1 + 2 s C(tau)) over {v > tau}, from tau = 0 (psgd_solve_kernel's
    generic path; the band path lands on the same point)."""
    tau, prev = 0.0, -1
    for _ in range(1000):
        act = vals > tau
        n = int(act.sum())
        tau = 2.0 * strength * float(vals[act].sum()) / (1.0 + 2.0 * strength * n)
        if n == prev:
            return tau
        prev = n
    raise RuntimeError("no fixed point")


def band_exact_sum(vals, E):
    """psgd_solve_kernel's order-independent band sum: every member lies in (2^(E-2), 2^E), so v * 2^(54-E) is an
    integer below 2^54; three 18-bit limbs are added in (32-bit) integers and the total is rounded once."""
    vals = np.asarray(vals, dtype=np.float64)
    I = np.ldexp(vals, 54 - E)
    assert np.all(I == np.floor(I)) and np.all(I < 2.0 ** 54)
    I = I.astype(np.uint64)
    l0 = int(np.sum(I & np.uint64(0x3ffff), dtype=np.uint64))
    l1 = int(np.sum((I >> np.uint64(18)) & np.uint64(0x3ffff), dtype=np.uint64))
    l2 = int(np.sum(I >> np.uint64(36), dtype=np.uint64))
    assert max(l0, l1, l2) < 2 ** 32 or len(vals) > 2048
    return float(np.ldexp(float(l2) * 68719476736.0 + float((l1 << 18) + l0), E - 54))


def band_solve(band, sumA, cntA, strength, b_lo, b_hi, max_iter=64):
    """psgd_solve_kernel's band path for one column: (sumA, cntA) = sum / number of the values above the band,
    `band` = the values inside (b_lo, b_hi] in ANY order.  Returns tau, or None where the kernel falls back to
    the generic passes."""
    band = np.asarray(band, dtype=np.float64)
    E = int(np.floor(np.log2(b_hi))) + 1
    if band.size and not (np.all(band > 2.0 ** (E - 2)) and np.all(band < 2.0 ** E)):
        return None
    tau, prev_n = b_lo, -1
    for _ in range(max_iter):
        act = band > tau
        n = int(act.sum())
        if n == prev_n:
            return tau if b_lo < tau <= b_hi else None
        prev_n = n
        s = band_exact_sum(band[act], E) if n else 0.0
        tau = 2.0 * strength * (sumA + s) / (1.0 + 2.0 * strength * (cntA + n))
    return None



class RankState:
    def __init__(self, plan, csr, y, idx, n_orders, k, degree):
        t = lambda a: None if a is None else a.cpu().numpy()      # noqa: E731
        self.plan = plan
        self.e_pos, self.e_x = t(plan.e_pos), t(plan.e_x)
        self.u_feat, self.u_ptr = t(plan.u_feat), t(plan.u_ptr)
        self.lc_u, self.lc_e0 = t(plan.lc_u), t(plan.lc_e0)
        self.sc_ptr, self.sc_u, self.sc_feat, self.sc_pos, self.sc_x = (t(plan.sc_ptr), t(plan.sc_u), t(plan.sc_feat),
                                                                        t(plan.sc_pos), t(plan.sc_x))
        self.sg_u, self.sg_feat, self.sg_pos, self.sg_x = t(plan.sg_u), t(plan.sg_feat), t(plan.sg_pos), t(plan.sg_x)
        self.ml_u, self.ml_c0 = t(plan.ml_u), t(plan.ml_c0)
        self.csr_slot = t(plan.csr_slot)
        self.own_q, self.own_src = t(plan.own_q), t(plan.own_src)
        self.indptr, self.indices, self.data = (np.asarray(a) for a in csr)
        self.y, self.idx = y, idx
        self.d_rows = plan.d_rows
        self.P = np.zeros((n_orders, plan.d_rows, k))
        self.w = np.zeros(plan.d_rows)
        self.sloss = np.zeros(plan.n_local)


FRAME_MAX = 1e100


def frame_in_range(C, Cw):
    """sp_psgd_plan_run folds the frame into the storage after a minibatch that takes C or Cw out of this range."""
    return 1.0 / FRAME_MAX < C < FRAME_MAX and 1.0 / FRAME_MAX < Cw < FRAME_MAX


def run_model(ranks, d, n_orders, k, degree, reg, loss, fit_linear, lams, alpha, beta, gamma, eta0, lr, power_t, it,
              P_odk, w, epochs=1, folds=None):
    """`epochs` epochs over the plans of `ranks` (list of RankState, one per simulated rank).  P_odk [o,d,k] / w [d]
    are updated in place; returns (it, sum of losses of the last epoch).  `folds` (a list) receives the `it` of
    every minibatch after which the frame was folded."""
    folds = [] if folds is None else folds
    G = len(ranks)
    ncol = n_orders * k
    for r, R in enumerate(ranks):                       # load_model
        nrow = len(range(r, d, G))
        R.P[:] = 0.0; R.w[:] = 0.0
        R.P[:, :nrow] = P_odk[:, r::G]
        R.w[:nrow] = w[r::G]
    thr = np.zeros((n_orders, k))
    C = Cw = 1.0
    M = ranks[0].plan.n_minibatches
    bL = ranks[0].plan.batch_local
    degs = [degree - o for o in range(n_orders)]
    sum_loss = 0.0
    early = {}                                          # rank -> RAW rows of its next minibatch, pulled before the prox
    for _ in range(epochs):
        for m in range(M):
            eta_P, eta_w = get_eta(lr, eta0, alpha, beta, power_t, it)
            b_glob = sum(min((m + 1) * bL, R.plan.n_local) - m * bL for R in ranks)
            cP, denP = eta_P / b_glob, 1.0 + eta_P * beta
            cw, denw = eta_w / b_glob, 1.0 + eta_w * alpha
            CnP = C * denP
            Cnw = Cw * denw if fit_linear else Cw
            invC, invCw = 1.0 / C, 1.0 / Cw
            strength = gamma * eta_P / (1.0 + eta_P * beta)
            inbox = [[None] * G for _ in range(G)]            # inbox[owner][src] = (gP rows, gw)
            for r, R in enumerate(ranks):
                pl = R.plan
                e0, e1 = pl.mb_eptr[m], pl.mb_eptr[m + 1]
                u0, u1 = pl.mb_uptr[m], pl.mb_uptr[m + 1]
                b0, b1 = m * bL, min((m + 1) * bL, pl.n_local)
                # ---- pull (sharded) / direct reads: RAW rows of the minibatch's columns -- for every minibatch but the
                #      first of an epoch they were fetched right after the owners' update of the previous one, i.e.
                #      BEFORE its prox moved the frame (psgd_pull_kernel on the context's own stream); the readers apply
                #      the frame of THIS minibatch
                feats = R.u_feat[u0:u1]
                if r in early:
                    raw_stage, raw_w = early.pop(r)
                else:
                    raw_stage = np.stack([ranks[j % G].P[:, j // G, :] for j in feats]) if len(feats) else np.zeros((0, n_orders, k))
                    raw_w = np.array([ranks[j % G].w[j // G] for j in feats])
                assert raw_stage.shape[0] == u1 - u0
                stage = st_true(raw_stage, thr, invC)
                stage_w = raw_w * invCw
                slot_of = {int(j): su for su, j in enumerate(feats)}
                # ---- rows pass
                bufA = {}
                bufdL = np.zeros(b1 - b0)
                for b in range(b0, b1):
                    i = R.idx[b]
                    st, en = R.indptr[i], R.indptr[i + 1]
                    A = np.zeros((n_orders, degree + 1, k))
                    A[:, 0, :] = 1.0
                    ypred = 0.0
                    for e in range(st, en):
                        j, x = R.indices[e], R.data[e]
                        su = R.csr_slot[e] if G > 1 else slot_of[int(j)]
                        assert feats[su] == j
                        if fit_linear:
                            ypred += x * stage_w[su]
                        for o in range(n_orders):
                            for t in range(degs[o]):
                                A[o, degs[o] - t] += (A[o, degs[o] - t - 1] * x) * stage[su, o]
                    for o in range(n_orders):
                        ypred += float(np.dot(lams, A[o, degs[o]]))
                    bufA[b - b0] = A
                    bufdL[b - b0] = dloss(loss, ypred, R.y[i])
                    R.sloss[b] = lossv(loss, ypred, R.y[i])
                # ---- column pass exactly like psgd_cols_{short,long,combine}_kernel
                part = {}
                done = {}                                   # column -> (g [o,k], gw)

                def term(pos, x, pold):
                    g = np.zeros((n_orders, k))
                    A = bufA[pos]
                    for o in range(n_orders):
                        dprev = np.full(k, x)
                        for t in range(1, degs[o]):
                            dprev = x * (A[o, t] - pold[o] * dprev)
                        g[o] = (bufdL[pos] * lams) * dprev
                    return g, bufdL[pos] * x

                def sum_entries(ea, eb, pold):
                    g, gw = np.zeros((n_orders, k)), 0.0
                    for e in range(ea, eb):
                        tg, tw = term(int(R.e_pos[e]), R.e_x[e], pold)
                        g = g + tg
                        gw = gw + tw
                    return g, gw

                seen = np.zeros(u1 - u0, dtype=int)
                for q in range(pl.mb_sgptr[m], pl.mb_sgptr[m + 1]):       # single-nonzero columns: self-contained records
                    u = int(R.sg_u[q])
                    assert R.u_ptr[u + 1] - R.u_ptr[u] == 1 and R.u_feat[u] == R.sg_feat[q]
                    assert R.e_pos[R.u_ptr[u]] == R.sg_pos[q] and R.e_x[R.u_ptr[u]] == R.sg_x[q]
                    tg, tw = term(int(R.sg_pos[q]), R.sg_x[q], stage[u - u0])
                    done[(u, )] = (np.zeros((n_orders, k)) + tg, 0.0 + tw)
                    seen[u - u0] += 1
                for q in range(pl.mb_shptr[m], pl.mb_shptr[m + 1]):       # short columns: compact copies of their nonzeros
                    u = int(R.sc_u[q])
                    ea, eb = R.u_ptr[u], R.u_ptr[u + 1]
                    p0, p1 = R.sc_ptr[q], R.sc_ptr[q + 1]
                    assert 2 <= eb - ea <= SH and e0 <= ea and eb <= e1 and p1 - p0 == eb - ea and R.sc_feat[q] == R.u_feat[u]
                    assert np.array_equal(R.sc_pos[p0:p1], R.e_pos[ea:eb]) and np.array_equal(R.sc_x[p0:p1], R.e_x[ea:eb])
                    g, gw = np.zeros((n_orders, k)), 0.0
                    for e in range(p0, p1):
                        tg, tw = term(int(R.sc_pos[e]), R.sc_x[e], stage[u - u0])
                        g = g + tg
                        gw = gw + tw
                    done[(u, )] = (g, gw)
                    seen[u - u0] += 1
                lc0, lc1 = pl.mb_lcptr[m], pl.mb_lcptr[m + 1]
                for c in range(lc0, lc1):
                    u, ce0 = int(R.lc_u[c]), int(R.lc_e0[c])
                    cend = R.u_ptr[u + 1]
                    assert cend - R.u_ptr[u] > SH and R.u_ptr[u] <= ce0 < cend and (ce0 - R.u_ptr[u]) % CH == 0
                    ce1 = min(ce0 + CH, cend)
                    res = sum_entries(ce0, ce1, stage[u - u0])
                    if cend - R.u_ptr[u] <= CH:
                        done[(u, )] = res
                        seen[u - u0] += 1
                    else:
                        part[c - lc0] = res
                for q in range(pl.mb_mlptr[m], pl.mb_mlptr[m + 1]):
                    u, c0 = int(R.ml_u[q]), int(R.ml_c0[q])
                    npc = -(-(R.u_ptr[u + 1] - R.u_ptr[u]) // CH)
                    assert npc > 1
                    GPB = 8                                  # groups of a block add strided pieces, then in group order
                    gs = []
                    for wg in range(min(GPB, npc)):
                        g, gw = np.zeros((n_orders, k)), 0.0
                        for pc in range(wg, npc, GPB):
                            assert R.lc_u[lc0 + c0 + pc] == u
                            pg, pw = part.pop(c0 + pc)
                            g = g + pg
                            gw = gw + pw
                        gs.append((g, gw))
                    g, gw = gs[0]
                    for pg, pw in gs[1:]:
                        g = g + pg
                        gw = gw + pw
                    done[(u, )] = (g, gw)
                    seen[u - u0] += 1
                assert not part, "a partial sum was never consumed"
                assert np.all(seen == 1), "every column finished exactly once"
                # ---- apply (single rank) or push to the owners' inboxes
                if G == 1:
                    for (u, ), (g, gw) in done.items():
                        j = int(R.u_feat[u])
                        pold = stage[u - u0]
                        v = (pold - g * cP) / denP
                        R.P[:, j, :] = to_raw(v, thr, CnP)
                        if fit_linear:
                            R.w[j] = ((stage_w[u - u0] - gw * cw) / denw) * Cnw
                else:
                    ost = pl.mb_owner_start[m]
                    for o in range(G):
                        n_o = ost[o + 1] - ost[o]
                        inbox[o][r] = (np.zeros((n_o, n_orders, k)), np.zeros(n_o))
                    for (u, ), (g, gw) in done.items():
                        su = u - u0
                        owner = int(R.u_feat[u]) % G
                        assert ost[owner] <= su < ost[owner + 1]
                        inbox[owner][r][0][su - ost[owner]] = g
                        inbox[owner][r][1][su - ost[owner]] = gw
            # ---- owner pass (after the cross-rank barrier)
            if G > 1:
                for o, R in enumerate(ranks):
                    pl = R.plan
                    o0, o1 = pl.mb_optr[m], pl.mb_optr[m + 1]
                    for t in range(o0, o1):
                        q = int(R.own_q[t])
                        g, gw = np.zeros((n_orders, k)), 0.0
                        for src in range(G):
                            at = int(R.own_src[t, src])
                            if at >= 0:
                                g = g + inbox[o][src][0][at]
                                gw = gw + inbox[o][src][1][at]
                        pold = st_true(R.P[:, q, :], thr, invC)
                        v = (pold - g * cP) / denP
                        R.P[:, q, :] = to_raw(v, thr, CnP)
                        if fit_linear:
                            R.w[q] = ((R.w[q] * invCw - gw * cw) / denw) * Cnw
            C, Cw = CnP, Cnw
            fold = not frame_in_range(C, Cw)
            # ---- early pull of the next minibatch's raw rows (every owner's rows are final; the prox below only
            #      moves thr); after a fold the rows are read from the folded storage instead
            if m + 1 < M and not fold:
                for r, R in enumerate(ranks):
                    nf = R.u_feat[R.plan.mb_uptr[m + 1]:R.plan.mb_uptr[m + 2]]
                    early[r] = (np.stack([ranks[j % G].P[:, j // G, :].copy() for j in nf]) if len(nf) else np.zeros((0, n_orders, k)),
                                np.array([ranks[j % G].w[j // G] for j in nf]))
            # ---- prox as a lazily applied column threshold
            if reg == "l1":
                thr = thr + C * strength
            else:
                invCn = 1.0 / C
                for o in range(n_orders):
                    for s in range(k):
                        vals = np.concatenate([np.maximum(np.abs(R.P[o, :, s]) - thr[o, s], 0.0) * invCn for R in ranks])
                        thr[o, s] = thr[o, s] + C * michelot(vals[vals > 0], strength)
            if fold:                                    # psgd_materialize_kernel + threshold reset (fold_frame)
                for R in ranks:
                    R.P[:] = st_true(R.P, thr[:, None, :], 1.0 / C)
                    if fit_linear:
                        R.w[:] = R.w * (1.0 / Cw)
                thr = np.zeros((n_orders, k))
                C = Cw = 1.0
                folds.append(it)
            it += 1
        sum_loss = sum(float(R.sloss.sum()) for R in ranks)
    for r, R in enumerate(ranks):                       # materialise + store_model
        nrow = len(range(r, d, G))
        P_odk[:, r::G] = st_true(R.P, thr[:, None, :], 1.0 / C)[:, :nrow]
        w[r::G] = (R.w / Cw)[:nrow]
    return it, sum_loss
