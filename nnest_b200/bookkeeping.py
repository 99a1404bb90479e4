"""Evidence bookkeeping of nested sampling, many iterations at a time.

Same arithmetic, in the same order, as the reference's per-iteration loop (nnest/nested.py:272-293,429-439,458-464):
the selection of worst points / usable chains comes from the exact host routine nnb_ns_consume (C ABI), the float64
recurrences are evaluated with NumPy's *sequential* accumulations (np.cumsum, np.logaddexp.accumulate) and a scalar
loop for the information H, so every intermediate equals the reference's bit for bit.  Host-only (no GPU needed).
"""
import ctypes as C

import numpy as np

from . import _lib as L


class NSBook(object):
    """State of the run: evidence, information, prior volume, iteration counter, dead points.  With num_derived > 0 the
    derived parameters of the dead points are kept too (saved_derived, next to saved_v), and the methods that move live
    points take the live set's derived rows as well."""

    def __init__(self, num_live_points, num_derived=0):
        self.nlive = int(num_live_points)
        self.num_derived = int(num_derived)
        self.saved_derived = []
        self.h = 0.0                                                      # nested.py:242-247
        self.logz = -1e300
        self.logvol = np.log(1.0 - np.exp(-1.0 / self.nlive))
        self.fraction_remain = 1.0
        self.it = 0
        self.saved_v, self.saved_logl, self.saved_logwt = [], [], []      # lists of array chunks

    def dead_points(self):
        if not self.saved_v:
            return np.empty((0, 0)), np.empty((0,)), np.empty((0,))
        return np.concatenate(self.saved_v), np.concatenate(self.saved_logl), np.concatenate(self.saved_logwt)

    def samples_with(self, active_v):
        """np.concatenate((dead points, active_v)) built with ONE copy of the dead points (they are kept as chunks), the
        chunks copied by a few host threads: at config-4 size the result is 2.1 GB of freshly faulted pages, and first-touch
        page faults on one core are what a plain concatenate spends its time on."""
        from concurrent.futures import ThreadPoolExecutor
        active_v = np.asarray(active_v, dtype=np.float64)
        sizes = [c.shape[0] for c in self.saved_v]
        offs = np.concatenate(([0], np.cumsum(sizes, dtype=np.int64)))
        m = int(offs[-1])
        out = np.empty((m + active_v.shape[0], active_v.shape[1]), dtype=np.float64)
        nt = 8 if m * active_v.shape[1] >= (1 << 22) else 1

        def work(t):
            for i in range(t, len(sizes), nt):
                if sizes[i]:
                    out[offs[i]:offs[i + 1]] = self.saved_v[i].reshape(sizes[i], -1)
        if nt == 1:
            work(0)
        else:
            with ThreadPoolExecutor(nt) as pool:
                list(pool.map(work, range(nt)))
        out[m:] = active_v
        return out

    def dead_derived(self):
        """derived parameters (num_dead, num_derived) of the dead points, in the order of dead_points()"""
        if not self.saved_derived:
            return np.empty((0, self.num_derived))
        return np.concatenate(self.saved_derived)

    def num_dead(self):
        return int(sum(len(a) for a in self.saved_logl))

    # ---- one iteration, exactly as the reference (used around refills / retrains / checkpoints) ---------------
    def evidence_update(self, active_v, active_logl, worst, active_derived=None):
        """nested.py:273,280-293"""
        logwt = self.logvol + active_logl[worst]
        logz_new = np.logaddexp(self.logz, logwt)
        self.h = (np.exp(logwt - logz_new) * active_logl[worst]
                  + np.exp(self.logz - logz_new) * (self.h + self.logz) - logz_new)
        self.logz = logz_new
        self.saved_v.append(np.array(active_v[worst], copy=True)[None, :])
        self.saved_logwt.append(np.array([logwt]))
        self.saved_logl.append(np.array([active_logl[worst]]))
        if self.num_derived:
            self.saved_derived.append(np.array(active_derived[worst], dtype=np.float64)[None, :])

    def shrink(self, max_logl):
        """nested.py:460-464"""
        self.logvol -= 1.0 / self.nlive
        logz_remain = max_logl - self.it / self.nlive
        self.fraction_remain = np.logaddexp(self.logz, logz_remain) - self.logz
        self.it += 1

    # ---- a run of plain iterations ----------------------------------------------------------------------------
    def bulk(self, active_u, active_v, active_logl, transform, b_first, b_last, b_logl, nb, max_iters, dlogz,
             it_limit, active_derived=None, b_derived=None):
        """Runs up to `max_iters` iterations that all start with accept_point == True (evidence update, scan of the
        batch from `nb`, replacement, shrink).  Mutates the live set and self.  Returns
        (nb, n_done, exhausted, finished): `exhausted` = the last started iteration used up the batch without
        finding a usable chain (its evidence update has been applied, accept_point is now False); `finished` = the
        loop condition `fraction_remain > dlogz and it <= it_limit` (nested.py:269) failed after the last iteration.
        With derived parameters, active_derived (nlive, num_derived) is updated like active_u, from b_derived (the derived
        parameters of the rows of b_last), and the dead points' rows are recorded as for active_v."""
        lib = L.load()
        nlive, n_chains, d = self.nlive, b_first.shape[0], b_first.shape[1]
        worst = np.empty(max_iters + 1, dtype=np.int64)
        chain = np.empty(max_iters + 1, dtype=np.int64)
        prev = np.empty(max_iters + 1, dtype=np.int64)
        lstar = np.empty(max_iters + 1, dtype=np.float64)
        maxl = np.empty(max_iters + 1, dtype=np.float64)
        c_nb, exh = C.c_int64(nb), C.c_int(0)
        ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        assert active_logl.dtype == np.float64 and active_logl.flags.c_contiguous
        k = lib.nnb_ns_consume(dp(active_logl), nlive, fp(b_first), fp(b_last), dp(b_logl), n_chains, d, C.byref(c_nb),
                               max_iters, ip(worst), ip(chain), ip(prev), dp(lstar), dp(maxl), C.byref(exh))
        if k < 0:
            raise RuntimeError('nnb_ns_consume failed (%d)' % k)
        exhausted = bool(exh.value)
        n_ev = k + (1 if exhausted else 0)               # iterations whose evidence update is due
        if n_ev == 0:
            return c_nb.value, 0, False, False
        # prior volume at the start of iteration j: repeated `logvol -= 1/nlive` (sequential, like the reference)
        lv = np.cumsum(np.concatenate(([self.logvol], np.full(k, -1.0 / nlive))))
        logwt = lv[:n_ev] + lstar[:n_ev]
        lz = np.logaddexp.accumulate(np.concatenate(([self.logz], logwt)))
        lz_prev, lz_new = lz[:-1], lz[1:]
        # loop condition after each successful iteration
        finished, n_done, n_evid = False, k, n_ev
        if k > 0:
            its = np.arange(self.it, self.it + k)
            logz_remain = maxl[:k] - its / nlive
            frac = np.logaddexp(lz_new[:k], logz_remain) - lz_new[:k]
            go_on = (frac > dlogz) & (its + 1 <= it_limit)
            stop = np.nonzero(~go_on)[0]
            if len(stop):
                finished = True
                n_done = int(stop[0]) + 1
                n_evid = n_done
                exhausted = False
        a_term = np.exp(logwt[:n_evid] - lz_new[:n_evid]) * lstar[:n_evid]
        b_term = np.exp(lz_prev[:n_evid] - lz_new[:n_evid])
        # h <- (a + b * (h + logz_old)) - logz_new, one iteration after the other (exact host routine of the C ABI)
        zp_c, zn_c = np.ascontiguousarray(lz_prev[:n_evid]), np.ascontiguousarray(lz_new[:n_evid])
        self.h = lib.nnb_ns_information(float(self.h), dp(np.ascontiguousarray(a_term)), dp(np.ascontiguousarray(b_term)),
                                        dp(zp_c), dp(zn_c), n_evid)
        self.logz = lz_new[n_evid - 1]
        # dead points: the physical point sitting in slot `worst` when its iteration started
        # row movements (gather of the end points, dead points, last-write-wins replacement): exact host routines of the C
        # ABI, a few threads each (random-row gathers of a 16 MB live set are cache-miss bound)
        new_u = np.empty((n_done, d), dtype=np.float64)
        chain_c = np.ascontiguousarray(chain[:n_done])
        if n_done:
            rc = lib.nnb_gather_rows_f32(fp(b_last), n_chains, d, ip(chain_c), n_done, dp(new_u))
            assert rc == 0, rc
        new_v = np.ascontiguousarray(np.asarray(transform(new_u), dtype=np.float64).reshape(new_u.shape)) if n_done \
            else new_u
        new_logl = np.ascontiguousarray(b_logl[chain_c], dtype=np.float64)
        w = np.ascontiguousarray(worst[:n_evid])
        pv = np.ascontiguousarray(prev[:n_evid])
        dead = np.empty((n_evid, d), dtype=np.float64)
        assert active_u.flags.c_contiguous and active_v.flags.c_contiguous and active_u.dtype == np.float64 \
            and active_v.dtype == np.float64
        rc = lib.nnb_ns_apply(ip(w), ip(pv), n_evid, n_done, d, dp(new_u), dp(new_v), dp(new_logl), dp(active_u),
                              dp(active_v), dp(active_logl), nlive, dp(dead))
        assert rc == 0, rc
        if self.num_derived:
            # the same rule as nnb_ns_apply's dead_out: the row that sat in slot worst[i] when iteration i started, i.e.
            # the replacement an earlier iteration of this call wrote there (prev[i]) or the live row from before the call
            new_der = b_derived[chain_c]
            dead_der = np.where((pv >= 0)[:, None], new_der[np.maximum(pv, 0)] if n_done else 0.0, active_derived[w])
            if n_done:                                              # the last write to a slot wins
                _, first_rev = np.unique(w[:n_done][::-1], return_index=True)
                keep = n_done - 1 - first_rev
                active_derived[w[keep]] = new_der[keep]
            self.saved_derived.append(dead_der)
        self.saved_v.append(dead)
        self.saved_logwt.append(np.array(logwt[:n_evid], copy=True))
        self.saved_logl.append(np.array(lstar[:n_evid], copy=True))
        self.last_slots = np.array(worst[:n_done], copy=True)       # (slot, chain) pairs of this call, in order: lets the
        self.last_chains = np.array(chain[:n_done], copy=True)      # caller mirror the replacements elsewhere (device)
        if n_done:
            self.logvol = lv[n_done]
            self.fraction_remain = frac[n_done - 1]
            self.it += n_done
        nb_out = c_nb.value
        if finished and n_done < k:
            nb_out = int(chain[n_done - 1]) + 1      # chains after the last used one were not consumed
        return nb_out, n_done, exhausted, finished
