"""Host side of the planned psgd path (csrc/psgd_plan.cu): the "batch CSC" plan of a sample order and
the context (model shard, scratch, peer pointers) a planned fit runs in.

Reference semantics: psgd.psgd_epoch (optimizer/psgd.py:125-199) visits the samples in
`indices_samples` order, cuts them into minibatches of batch_size and, per minibatch, adds every
sample's gradient terms to the rows of grad_P its nonzeros touch.  The plan regroups the nonzeros of
each minibatch by feature (samples ascending inside a feature: the reference's summation order), so
that the CUDA side can sum a row's terms without atomics and update only the touched rows.  It depends
on X, the sample order and the batch size only -- built once per fit (once per epoch with shuffle=True)
by device sorts; PyTorch is the sort / allocator provider here, nothing else.

Sharded over the ranks of a process group (one process per GPU): samples are sharded by rank (every
rank holds n_local rows and contributes batch_local of them to each minibatch), P is sharded by rows
(feature j lives on rank j % world, local row j // world) in peer-visible memory (CUDA IPC), and a
minibatch's columns are ordered by (owner, feature) so that the partial gradient rows for one owner
are contiguous.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

CHUNK = 64            # SP_PSGD_CHUNK
SHORT = 8             # SP_PSGD_SHORT
MAX_RANKS = 8         # SP_MAX_RANKS
CHANNELS = 3          # SP_PSGD_CHANNELS
_GROUP_ENTRIES = 48_000_000     # nonzeros sorted at a time while building (bounds the temporaries)


def _comm_device(group):
    import torch.distributed as dist
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")


def all_gather_var(t, group):
    """all_gather of 1-D tensors of different lengths; returns the list on t's device."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    cdev = _comm_device(group)
    n = torch.tensor([t.numel()], dtype=torch.int64, device=cdev)
    ns = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(ns, n, group=group)
    ns = [int(v.item()) for v in ns]
    cap = max(max(ns), 1)
    buf = torch.zeros(cap, dtype=t.dtype, device=cdev)
    buf[: t.numel()] = t.to(cdev)
    outs = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(outs, buf, group=group)
    return [o[:m].to(t.device) for o, m in zip(outs, ns)]


class PsgdPlan:
    """sp_psgd_plan for samples idx[0:n_local] of a device CSR matrix."""

    def __init__(self, csr, idx, n_features, batch_local, world=1, rank=0, group=None, group_entries=_GROUP_ENTRIES,
                 defer_owner_tables=False):
        indptr, indices, data = csr
        dev = data.device
        self.device = dev
        self.world, self.rank = int(world), int(rank)
        self.n_local = int(idx.numel())
        self.batch_local = max(1, int(batch_local))
        self.n_features = int(n_features)
        bL, G = self.batch_local, self.world
        M = (self.n_local + bL - 1) // bL
        self.n_minibatches = M
        dq = (self.n_features + G - 1) // G
        self.d_rows = dq
        Dkey = G * dq
        nnz_total = int(data.numel())
        i64 = torch.int64
        # per-minibatch entry counts decide the build groups
        rows_all = idx.to(i64)
        cnt_all = (indptr[rows_all + 1] - indptr[rows_all]).to(i64)
        csum = torch.zeros(self.n_local + 1, dtype=i64, device=dev)
        csum[1:] = torch.cumsum(cnt_all, 0)
        mb_bounds = torch.arange(0, M + 1, dtype=i64, device=dev) * bL
        mb_bounds[-1] = self.n_local
        mb_eptr = csum[mb_bounds].cpu().numpy().astype(np.int64)             # [M+1]
        E = int(mb_eptr[-1])
        self.e_pos = torch.empty(E, dtype=torch.int32, device=dev)
        self.e_x = torch.empty(E, dtype=torch.float64, device=dev)
        self.csr_slot = torch.zeros(nnz_total, dtype=torch.int32, device=dev) if G > 1 else None
        u_feat, u_ptr, lc_u, lc_e0, lc_feat, lc_cnt, ml_u, ml_c0 = [], [], [], [], [], [], [], []
        sg_u, sg_feat, sg_pos, sg_x = [], [], [], []
        sc_len, sc_u, sc_feat, sc_pos, sc_x = [], [], [], [], []
        mb_ucnt, mb_sgcnt, mb_shcnt, mb_lccnt, mb_mlcnt, owner_cnt = [], [], [], [], [], []
        u_off = 0
        m0 = 0
        while m0 < M:
            m1 = m0 + 1
            while m1 < M and mb_eptr[m1 + 1] - mb_eptr[m0] <= group_entries:
                m1 += 1
            e0, e1 = int(mb_eptr[m0]), int(mb_eptr[m1])
            b0, b1 = m0 * bL, min(m1 * bL, self.n_local)
            tot = e1 - e0
            Mg = m1 - m0
            if tot == 0:
                for lst in (mb_ucnt, mb_sgcnt, mb_shcnt, mb_lccnt, mb_mlcnt):
                    lst.append(np.zeros(Mg, np.int64))
                owner_cnt.append(np.zeros((Mg, G), np.int64))
                m0 = m1
                continue
            cnt = cnt_all[b0:b1]
            pos = torch.arange(b1 - b0, dtype=i64, device=dev)
            pos_rep = torch.repeat_interleave(pos, cnt, output_size=tot)
            first = csum[b0:b1] - e0
            off = torch.arange(tot, dtype=i64, device=dev) - first[pos_rep]
            src = indptr[rows_all[b0:b1]].to(i64)[pos_rep] + off                 # CSR entry of every plan entry
            del off, first
            feat = indices[src].to(i64)
            mb = pos_rep // bL
            lpos = (pos_rep - mb * bL).to(torch.int32)
            del pos_rep
            key = mb * Dkey + (feat % G) * dq + feat // G
            del feat
            if Mg * Dkey < 2 ** 31:
                key = key.to(torch.int32)                                       # half the radix passes
            key, order = torch.sort(key, stable=True)                           # samples stay ascending inside a column
            key = key.to(i64)
            newcol = torch.ones(tot, dtype=torch.bool, device=dev)
            newcol[1:] = key[1:] != key[:-1]
            self.e_pos[e0:e1] = lpos[order]
            self.e_x[e0:e1] = data[src[order]]
            del lpos
            ucol = torch.cumsum(newcol.to(i64), 0) - 1                          # group-relative column of every entry
            ustart = torch.nonzero(newcol).squeeze(1)                           # group-relative first entry of every column
            ukey = key[ustart]
            umb = ukey // Dkey
            upf = ukey - umb * Dkey
            uowner = upf // dq
            u_feat.append(((upf - uowner * dq) * G + uowner).to(torch.int32))
            u_ptr.append(ustart + e0)
            nU = int(ustart.numel())
            ecnt = torch.from_numpy(np.diff(mb_eptr[m0:m1 + 1])).to(dev)
            eptr_rel = torch.zeros(Mg + 1, dtype=i64, device=dev)
            eptr_rel[1:] = torch.cumsum(ecnt, 0)
            ucnt = torch.bincount(umb, minlength=Mg)
            uptr_rel = torch.zeros(Mg + 1, dtype=i64, device=dev)
            uptr_rel[1:] = torch.cumsum(ucnt, 0)
            mb_ucnt.append(ucnt.cpu().numpy())
            if G > 1:
                mb_sorted = key // Dkey
                self.csr_slot[src[order]] = (ucol - uptr_rel[mb_sorted]).to(torch.int32)
                del mb_sorted
                owner_cnt.append(torch.bincount(umb * G + uowner, minlength=Mg * G).reshape(Mg, G).cpu().numpy())
            del src, order, key
            # columns by length: short ones are summed by one group of lanes, longer ones are cut into chunks
            uend = torch.empty(nU, dtype=i64, device=dev)
            uend[:-1] = ustart[1:]
            uend[-1] = tot
            ulen = uend - ustart
            is_short = ulen <= SHORT
            sg_idx = torch.nonzero(ulen == 1).squeeze(1)                          # single-nonzero columns: kept apart, self-contained
            sg_u.append((sg_idx + u_off).to(torch.int32))
            sg_feat.append(u_feat[-1][sg_idx])
            sg_pos.append(self.e_pos[e0:e1][ustart[sg_idx]])
            sg_x.append(self.e_x[e0:e1][ustart[sg_idx]])
            mb_sgcnt.append(torch.bincount(umb[sg_idx], minlength=Mg).cpu().numpy())
            sh_idx = torch.nonzero(is_short & (ulen > 1)).squeeze(1)              # 2..SHORT nonzeros: compact copies of them
            sh_len = ulen[sh_idx]
            nse = int(sh_len.sum()) if sh_idx.numel() else 0
            sc_len.append(sh_len)
            sc_u.append((sh_idx + u_off).to(torch.int32))
            sc_feat.append(u_feat[-1][sh_idx])
            if nse:
                col = torch.repeat_interleave(torch.arange(sh_idx.numel(), dtype=i64, device=dev), sh_len, output_size=nse)
                within = torch.arange(nse, dtype=i64, device=dev) - (torch.cumsum(sh_len, 0) - sh_len)[col]
                src_e = ustart[sh_idx][col] + within
                sc_pos.append(self.e_pos[e0:e1][src_e])
                sc_x.append(self.e_x[e0:e1][src_e])
            mb_shcnt.append(torch.bincount(umb[sh_idx], minlength=Mg).cpu().numpy())
            lg_idx = torch.nonzero(~is_short).squeeze(1)
            npieces = (ulen[lg_idx] + CHUNK - 1) // CHUNK
            ntc = int(npieces.sum()) if lg_idx.numel() else 0
            first_chunk = torch.cumsum(npieces, 0) - npieces                      # group-relative index of a column's first chunk
            lcnt = torch.zeros(Mg, dtype=i64, device=dev)
            lcnt.index_add_(0, umb[lg_idx], npieces)
            lcptr_rel = torch.zeros(Mg + 1, dtype=i64, device=dev)
            lcptr_rel[1:] = torch.cumsum(lcnt, 0)
            mb_lccnt.append(lcnt.cpu().numpy())
            if ntc:
                col_of_chunk = torch.repeat_interleave(torch.arange(lg_idx.numel(), dtype=i64, device=dev), npieces, output_size=ntc)
                piece = torch.arange(ntc, dtype=i64, device=dev) - first_chunk[col_of_chunk]
                lc_u.append((lg_idx[col_of_chunk] + u_off).to(torch.int32))
                lc_e0.append(ustart[lg_idx[col_of_chunk]] + piece * CHUNK + e0)
                lc_feat.append(u_feat[-1][lg_idx[col_of_chunk]])
                cn = torch.clamp(ulen[lg_idx[col_of_chunk]] - piece * CHUNK, max=CHUNK)
                cn = cn + (npieces[col_of_chunk] == 1).to(i64) * (1 << 30)           # the column's only chunk
                lc_cnt.append(cn.to(torch.int32))
            multi = npieces > 1
            ml_idx = lg_idx[multi]
            ml_u.append((ml_idx + u_off).to(torch.int32))
            ml_c0.append((first_chunk[multi] - lcptr_rel[umb[ml_idx]]).to(torch.int32))   # relative to the minibatch's chunks
            mb_mlcnt.append(torch.bincount(umb[ml_idx], minlength=Mg).cpu().numpy())
            del ucol
            u_off += nU
            m0 = m1
        cat = lambda xs, dt: (torch.cat(xs) if xs else torch.zeros(0, dtype=dt, device=dev))   # noqa: E731
        self.u_feat = cat(u_feat, torch.int32)
        self.u_ptr = torch.cat([cat(u_ptr, i64), torch.tensor([E], dtype=i64, device=dev)])
        self.sg_u, self.sg_feat, self.sg_pos = cat(sg_u, torch.int32), cat(sg_feat, torch.int32), cat(sg_pos, torch.int32)
        self.sg_x = cat(sg_x, torch.float64)
        self.sc_u, self.sc_feat = cat(sc_u, torch.int32), cat(sc_feat, torch.int32)
        self.sc_pos, self.sc_x = cat(sc_pos, torch.int32), cat(sc_x, torch.float64)
        lens_all = cat(sc_len, i64)
        self.sc_ptr = torch.zeros(lens_all.numel() + 1, dtype=i64, device=dev)
        self.sc_ptr[1:] = torch.cumsum(lens_all, 0)
        self.lc_u = cat(lc_u, torch.int32)
        self.lc_e0 = cat(lc_e0, i64)
        self.lc_feat, self.lc_cnt = cat(lc_feat, torch.int32), cat(lc_cnt, torch.int32)
        self.ml_u = cat(ml_u, torch.int32)
        self.ml_c0 = cat(ml_c0, torch.int32)
        acc = lambda parts: np.concatenate([[0], np.cumsum(np.concatenate(parts) if parts else np.zeros(0, np.int64))]).astype(np.int64)  # noqa: E731
        self.mb_eptr = mb_eptr
        self.mb_uptr = acc(mb_ucnt)
        self.mb_sgptr = acc(mb_sgcnt)
        self.mb_shptr = acc(mb_shcnt)
        self.mb_lcptr = acc(mb_lccnt)
        self.mb_mlptr = acc(mb_mlcnt)
        self.max_chunks = int(np.max(np.diff(self.mb_lcptr))) if M else 0
        self.max_cols = int(np.max(np.diff(self.mb_uptr))) if M else 0
        self.n_entries = E
        self.n_cols = int(self.mb_uptr[-1])
        # ---- sharded: owner-side tables
        self.mb_owner_start = self.mb_optr = None
        self.own_q = self.own_src = None
        self.inbox_cap = 0
        if G > 1:
            oc = np.concatenate(owner_cnt, 0) if owner_cnt else np.zeros((0, G), np.int64)       # [M, G]
            ostart = np.zeros((M, G + 1), dtype=np.int64)
            ostart[:, 1:] = np.cumsum(oc, 1)
            self.mb_owner_start = np.ascontiguousarray(ostart.astype(np.int32))
            if defer_owner_tables:                      # (tests: several ranks' plans built in one process)
                return
            self.finish_owner_tables(*self.gather_column_lists(group))
            return
        self._fill_struct()

    def column_lists(self):
        """What the owners need from this rank: its columns, per-minibatch column offsets and owner offsets."""
        dev = self.device
        return (torch.tensor([self.n_local, self.batch_local], dtype=torch.int64, device=dev), self.u_feat,
                torch.from_numpy(self.mb_uptr).to(dev),
                torch.from_numpy(self.mb_owner_start.astype(np.int64).reshape(-1)).to(dev))

    def gather_column_lists(self, group):
        mine = self.column_lists()
        return tuple(all_gather_var(t, group) for t in mine)

    def finish_owner_tables(self, n_all, feats, uptrs, ostarts):
        """Rows of this rank touched by each GLOBAL minibatch and, per source rank, where that rank's partial
        row sits in its inbox region (the source's columns owned by this rank, in feature order).  Inputs:
        every rank's column_lists()."""
        dev, G, me, M = self.device, self.world, self.rank, self.n_minibatches
        dq = self.d_rows
        i64 = torch.int64
        if any(int(t[0]) != self.n_local or int(t[1]) != self.batch_local for t in n_all):
            raise ValueError("sharded psgd needs equal shards: (n_local, batch_local) per rank = "
                             + str([(int(t[0]), int(t[1])) for t in n_all]))
        keys, srcs, ats = [], [], []
        cap = 0
        for r in range(G):
            os_r = ostarts[r].reshape(M, G + 1)
            lo = uptrs[r][:-1] + os_r[:, me]                   # [M] absolute first column of rank r owned by me
            n = os_r[:, me + 1] - os_r[:, me]
            tot = int(n.sum())
            cap = max(cap, int(n.max()) if M else 0)
            if tot == 0:
                continue
            mbi = torch.repeat_interleave(torch.arange(M, dtype=i64, device=dev), n, output_size=tot)
            first = torch.cumsum(n, 0) - n
            at = torch.arange(tot, dtype=i64, device=dev) - first[mbi]
            f = feats[r][lo[mbi] + at].to(i64)
            keys.append(mbi * dq + f // G)
            srcs.append(torch.full((tot,), r, dtype=i64, device=dev))
            ats.append(at)
        # most columns any rank sends to any owner in one minibatch (identical on every rank: same layout)
        capg = 0
        for r in range(G):
            os_r = ostarts[r].reshape(M, G + 1)
            if M:
                capg = max(capg, int((os_r[:, 1:] - os_r[:, :-1]).max()))
        self.inbox_cap = max(capg, cap, 1)
        if keys:
            key = torch.cat(keys); src = torch.cat(srcs); at = torch.cat(ats)
            uniq, inv = torch.unique(key, sorted=True, return_inverse=True)
            own_src = torch.full((uniq.numel(), G), -1, dtype=torch.int32, device=dev)
            own_src[inv, src] = at.to(torch.int32)
            mbo = uniq // dq
            self.own_q = (uniq - mbo * dq).to(torch.int32)
            self.own_src = own_src.contiguous()
            ocnt = torch.bincount(mbo, minlength=M).cpu().numpy()
        else:
            self.own_q = torch.zeros(0, dtype=torch.int32, device=dev)
            self.own_src = torch.zeros((0, G), dtype=torch.int32, device=dev)
            ocnt = np.zeros(M, np.int64)
        self.mb_optr = np.concatenate([[0], np.cumsum(ocnt)]).astype(np.int64)
        self._fill_struct()

    def _fill_struct(self):
        s = _lib.SpPsgdPlan()
        s.n_minibatches, s.batch_local, s.n_local = self.n_minibatches, self.batch_local, self.n_local
        s.chunk, s.short_max = CHUNK, SHORT
        hp = lambda a: a.ctypes.data                         # noqa: E731  (host arrays are kept alive by self)
        s.mb_eptr_host, s.mb_uptr_host = hp(self.mb_eptr), hp(self.mb_uptr)
        s.mb_sgptr_host = hp(self.mb_sgptr)
        s.mb_shptr_host, s.mb_lcptr_host, s.mb_mlptr_host = hp(self.mb_shptr), hp(self.mb_lcptr), hp(self.mb_mlptr)
        s.sg_u, s.sg_feat, s.sg_pos, s.sg_x = (t.data_ptr() for t in (self.sg_u, self.sg_feat, self.sg_pos, self.sg_x))
        s.sc_ptr, s.sc_u, s.sc_feat = self.sc_ptr.data_ptr(), self.sc_u.data_ptr(), self.sc_feat.data_ptr()
        s.sc_pos, s.sc_x = self.sc_pos.data_ptr(), self.sc_x.data_ptr()
        s.e_pos, s.e_x = self.e_pos.data_ptr(), self.e_x.data_ptr()
        s.u_feat, s.u_ptr = self.u_feat.data_ptr(), self.u_ptr.data_ptr()
        s.lc_u, s.lc_e0 = self.lc_u.data_ptr(), self.lc_e0.data_ptr()
        s.lc_feat, s.lc_cnt = self.lc_feat.data_ptr(), self.lc_cnt.data_ptr()
        s.ml_u, s.ml_c0 = self.ml_u.data_ptr(), self.ml_c0.data_ptr()
        s.max_chunks, s.max_cols = self.max_chunks, self.max_cols
        if self.world > 1:
            s.csr_slot = self.csr_slot.data_ptr()
            s.mb_owner_start_host = hp(self.mb_owner_start)
            s.mb_optr_host = hp(self.mb_optr)
            s.own_q, s.own_src = self.own_q.data_ptr(), self.own_src.data_ptr()
        self.struct = s

    def ref(self):
        return C.byref(self.struct)

    def nbytes(self):
        ts = [self.e_pos, self.e_x, self.u_feat, self.u_ptr, self.sg_u, self.sg_feat, self.sg_pos, self.sg_x, self.sc_ptr, self.sc_u, self.sc_feat, self.sc_pos, self.sc_x, self.lc_u, self.lc_feat, self.lc_cnt, self.lc_e0, self.ml_u, self.ml_c0,
              self.csr_slot, self.own_q, self.own_src]
        return sum(t.numel() * t.element_size() for t in ts if t is not None)


class _Raw:
    """__cuda_array_interface__ view of library-allocated device memory (no ownership)."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def _view(ptr, shape, dtype=torch.float64):
    typestr = {torch.float64: "<f8", torch.int32: "<i4", torch.int64: "<i8", torch.uint8: "|u1"}[dtype]
    if int(np.prod(shape)) == 0:
        return torch.zeros(tuple(shape), dtype=dtype, device="cuda")
    return torch.as_tensor(_Raw(ptr, shape, typestr), device=torch.device("cuda", torch.cuda.current_device()))


def arows(degree, n_orders):
    """rows A^1..A^(deg_o-1) kept per sample over all orders (ARows<DEG,NORD> in psgd_plan.cu)."""
    return sum(degree - o - 1 for o in range(n_orders))


class PsgdContext:
    """sp_psgd_ctx + the device memory behind it.  Single rank: P / w are ordinary tensors.  Sharded: the
    peer-visible buffers (model shard, inboxes, statistics boxes, flags) live in one cudaMalloc slab per
    rank whose CUDA IPC handle is exchanged through the process group at construction."""

    def __init__(self, plan, n_orders, k, degree, reg, loss, fit_linear, lams, group=None, inbox_cap=None):
        L = _lib.load()
        dev = plan.device
        self.plan_dims = (plan.max_chunks, plan.max_cols, plan.batch_local)
        self.world, self.rank, self.group = plan.world, plan.rank, group
        self.n_orders, self.k, self.d, self.d_rows = int(n_orders), int(k), plan.n_features, plan.d_rows
        f64 = torch.float64
        ncolk = self.n_orders * self.k
        self.lams = lams
        self.thr = torch.zeros(ncolk, dtype=f64, device=dev)
        ar = arows(degree, n_orders)
        self.bufA = torch.empty(max(plan.batch_local * ar * k, 1), dtype=f64, device=dev)
        self.bufdL = torch.empty(max(plan.batch_local, 1), dtype=f64, device=dev)
        self.sample_loss = torch.zeros(max(plan.n_local, 1), dtype=f64, device=dev)
        self.part_g = torch.empty(max(plan.max_chunks * ncolk, 1), dtype=f64, device=dev)
        self.part_w = torch.empty(max(plan.max_chunks, 1), dtype=f64, device=dev)
        self.work = torch.zeros(int(L.sp_psgd_plan_work_doubles(self.n_orders, self.k)), dtype=f64, device=dev)
        xw = int(L.sp_psgd_plan_xwork_doubles(self.n_orders, self.k, self.world))
        s = _lib.SpPsgdCtx()
        self._slab = None
        self._peer_bases = []
        if self.world == 1:
            self.P = torch.zeros((self.n_orders, self.d_rows, self.k), dtype=f64, device=dev)
            self.w = torch.zeros(self.d_rows, dtype=f64, device=dev)
            self.xwork = torch.zeros(xw, dtype=f64, device=dev)
            s.xwork = self.xwork.data_ptr()
        else:
            import torch.distributed as dist
            cap = max(plan.inbox_cap, int(inbox_cap or 0))        # (shuffle=True: bound for any sample order)
            sizes = [("P", ncolk * self.d_rows), ("w", self.d_rows), ("inbox_g", self.world * cap * ncolk),
                     ("inbox_w", self.world * cap), ("xwork", xw), ("flags", CHANNELS * MAX_RANKS), ("err", 2)]
            offs, at = {}, 0
            for name, n in sizes:
                offs[name] = at
                at += (int(n) + 31) // 32 * 32                      # 256-byte aligned sub-buffers
            base = C.c_void_p()
            _lib.check(L.sp_shm_alloc(C.c_size_t(at * 8), C.byref(base)))
            self._slab = base.value
            handle = (C.c_ubyte * 64)()
            _lib.check(L.sp_ipc_export(C.c_void_p(self._slab), handle))
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle), group=group)
            bases = []
            for r in range(self.world):
                if r == self.rank:
                    bases.append(self._slab)
                    continue
                hb = (C.c_ubyte * 64).from_buffer_copy(handles[r])
                p = C.c_void_p()
                _lib.check(L.sp_ipc_open(hb, C.byref(p)))
                bases.append(p.value)
                self._peer_bases.append(p.value)
            at_ptr = lambda r, name: bases[r] + offs[name] * 8          # noqa: E731
            self.P = _view(at_ptr(self.rank, "P"), (self.n_orders, self.d_rows, self.k))
            self.w = _view(at_ptr(self.rank, "w"), (self.d_rows,))
            self.stage = torch.empty(max(plan.max_cols * ncolk, 1), dtype=f64, device=dev)
            self.stage_w = torch.empty(max(plan.max_cols, 1), dtype=f64, device=dev)
            s.stage, s.stage_w = self.stage.data_ptr(), self.stage_w.data_ptr()
            s.inbox_g, s.inbox_w = at_ptr(self.rank, "inbox_g"), at_ptr(self.rank, "inbox_w")
            s.inbox_cap = cap
            s.err = at_ptr(self.rank, "err")
            s.xwork = at_ptr(self.rank, "xwork")
            self._err = _view(at_ptr(self.rank, "err"), (2,), torch.int32)
            for r in range(self.world):
                s.peer_P[r], s.peer_w[r] = at_ptr(r, "P"), at_ptr(r, "w")
                s.peer_inbox_g[r] = at_ptr(r, "inbox_g") + self.rank * cap * ncolk * 8
                s.peer_inbox_w[r] = at_ptr(r, "inbox_w") + self.rank * cap * 8
                s.peer_xwork[r] = at_ptr(r, "xwork")
                s.peer_flags[r] = at_ptr(r, "flags")
            dist.barrier(group=group)
        s.P, s.w, s.lams, s.thr = self.P.data_ptr(), self.w.data_ptr(), lams.data_ptr(), self.thr.data_ptr()
        s.n_orders, s.k, s.d_rows, s.degree = self.n_orders, self.k, self.d_rows, int(degree)
        s.reg, s.loss, s.fit_linear = _lib.REG_IDS[reg], _lib.LOSS_IDS[loss], int(bool(fit_linear))
        s.world, s.rank = self.world, self.rank
        s.bufA, s.bufdL, s.sample_loss = self.bufA.data_ptr(), self.bufdL.data_ptr(), self.sample_loss.data_ptr()
        s.part_g, s.part_w, s.work = self.part_g.data_ptr(), self.part_w.data_ptr(), self.work.data_ptr()
        s.C, s.Cw, s.seq, s.seq_generic, s.seq_pull = 1.0, 1.0, 0, 0, 0
        s.aux_stream = None
        s.aux_event[0] = s.aux_event[1] = None
        self.struct = s

    def ref(self):
        return C.byref(self.struct)

    # ---- model in / out (feature-major P [n_orders, d, k], w [d] on the device)
    def load_model(self, P_odk, w):
        G, r = self.world, self.rank
        if G == 1:
            self.P.copy_(P_odk)
            self.w.copy_(w)
            return
        nrow = (self.d - r + G - 1) // G if self.d > r else 0
        self.P.zero_()
        self.w.zero_()
        self.P[:, :nrow] = P_odk[:, r::G]
        self.w[:nrow] = w[r::G]

    def store_model(self, P_odk, w):
        """all ranks end up with the full model (sharded: one all-gather of the row shards)."""
        if self.world == 1:
            P_odk.copy_(self.P)
            w.copy_(self.w)
            return
        import torch.distributed as dist
        G = self.world
        cdev = _comm_device(self.group)
        mine = torch.cat([self.P.reshape(-1), self.w]).to(cdev)
        parts = [torch.empty_like(mine) for _ in range(G)]
        dist.all_gather(parts, mine, group=self.group)
        npk = self.n_orders * self.d_rows * self.k
        for r in range(G):
            nrow = (self.d - r + G - 1) // G if self.d > r else 0
            pr = parts[r].to(P_odk.device)
            P_odk[:, r::G] = pr[:npk].reshape(self.n_orders, self.d_rows, self.k)[:, :nrow]
            w[r::G] = pr[npk:][:nrow]

    def check_peers(self):
        if self.world > 1 and int(self._err[0].item()) != 0:
            raise RuntimeError("sharded psgd: a cross-rank wait timed out (a peer rank failed or stalled)")

    def rebind(self, plan):
        """The scratch sized by the plan must cover a rebuilt plan (shuffle=True rebuilds every epoch) and the plan of
        another chunk of rows (partial_fit: any number of rows)."""
        if plan.n_local > self.sample_loss.numel():
            self.sample_loss = torch.zeros(plan.n_local, dtype=torch.float64, device=plan.device)
            self.struct.sample_loss = self.sample_loss.data_ptr()
        if (plan.max_chunks, plan.max_cols, plan.batch_local) != self.plan_dims:
            dev, f64 = plan.device, torch.float64
            ncolk = self.n_orders * self.k
            if plan.max_chunks > self.plan_dims[0]:
                self.part_g = torch.empty(max(plan.max_chunks * ncolk, 1), dtype=f64, device=dev)
                self.part_w = torch.empty(max(plan.max_chunks, 1), dtype=f64, device=dev)
                self.struct.part_g, self.struct.part_w = self.part_g.data_ptr(), self.part_w.data_ptr()
            if self.world > 1 and plan.max_cols > self.plan_dims[1]:
                self.stage = torch.empty(max(plan.max_cols * ncolk, 1), dtype=f64, device=dev)
                self.stage_w = torch.empty(max(plan.max_cols, 1), dtype=f64, device=dev)
                self.struct.stage, self.struct.stage_w = self.stage.data_ptr(), self.stage_w.data_ptr()
            if self.world > 1 and plan.inbox_cap > self.struct.inbox_cap:
                raise RuntimeError("sharded psgd with shuffle=True: inbox capacity exceeded after a reshuffle")
            self.plan_dims = (max(plan.max_chunks, self.plan_dims[0]), max(plan.max_cols, self.plan_dims[1]), plan.batch_local)

    def close(self):
        L = _lib.load()
        if getattr(self, "struct", None) is not None and self.struct.aux_stream:
            torch.cuda.synchronize()
            L.sp_psgd_plan_release(self.ref())
        if self._slab is not None:
            torch.cuda.synchronize()
            if self.group is not None:
                import torch.distributed as dist
                dist.barrier(group=self.group)
            for p in self._peer_bases:
                L.sp_ipc_close(C.c_void_p(p))
            self._peer_bases = []
            self.P = self.w = self._err = None
            L.sp_shm_free(C.c_void_p(self._slab))
            self._slab = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
