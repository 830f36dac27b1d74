"""Engine: one device handle of libyue_b200.so, numpy in / numpy out.

This is the layer the recommender classes (yue_b200/bpr.py) sit on; it only marshals
arguments.  All compute happens in the CUDA library -- there is no CPU path here.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import (MODE_HOGWILD, MODE_HOGWILD_STORE, MODE_SERIAL, RANK_AUTO, RANK_EXACT,  # noqa: F401
                   RANK_TC, YueError)


def _ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


def _as(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


class PinnedArray:
    """numpy array over cudaHostAlloc'ed memory (DMA target for factor tables / results)."""

    def __init__(self, shape, dtype):
        lib = _lib.load()
        self._lib = lib
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        rc = lib.yue_host_alloc(self.nbytes, C.byref(p))
        if rc:
            raise YueError(rc, "yue_host_alloc(%d) failed" % self.nbytes)
        self._p = p
        buf = (C.c_byte * max(self.nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if self._p is not None:
            self.array = None
            self._lib.yue_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    def __init__(self, device=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.yue_create(int(device), C.byref(h))
        if rc:
            raise YueError(rc, self.lib.yue_last_error(None).decode())
        self.h = h
        self.device = int(device)
        self.m = self.n = self.k = self.T = 0

    # -- plumbing -------------------------------------------------------------------------
    def _ck(self, rc):
        if rc:
            raise YueError(rc, self.lib.yue_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.yue_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._ck(self.lib.yue_sync(self.h))

    # -- data ------------------------------------------------------------------------------
    def set_interactions(self, m, n, ev_indptr, ev_items, uq_indptr, uq_items,
                         user_begin=0, event_base=0):
        ev_indptr, uq_indptr = _as(ev_indptr, np.int64), _as(uq_indptr, np.int64)
        ev_items, uq_items = _as(ev_items, np.int32), _as(uq_items, np.int32)
        if len(ev_indptr) != m + 1 or len(uq_indptr) != m + 1:
            raise ValueError("indptr arrays must have m+1 entries")
        if len(ev_items) != ev_indptr[-1] or len(uq_items) != uq_indptr[-1]:
            raise ValueError("item arrays do not match indptr[-1]")
        self._ck(self.lib.yue_set_interactions_shard(
            self.h, m, n, user_begin, event_base, _ptr(ev_indptr, C.c_int64), _ptr(ev_items, C.c_int32),
            _ptr(uq_indptr, C.c_int64), _ptr(uq_items, C.c_int32)))
        self.m, self.n, self.T = int(m), int(n), int(ev_indptr[-1])

    def ingest_events(self, m, n, ev_user, ev_item, is_test=None):
        """Array form of the log built on the device from events in file order (yue_ingest_events)."""
        ev_user, ev_item = _as(ev_user, np.int32), _as(ev_item, np.int32)
        if len(ev_user) != len(ev_item):
            raise ValueError("ev_user and ev_item differ in length")
        flag = None
        if is_test is not None:
            is_test = _as(is_test, np.uint8)
            if len(is_test) != len(ev_user):
                raise ValueError("is_test length")
            flag = _ptr(is_test, C.c_uint8)
        self._ck(self.lib.yue_ingest_events(self.h, m, n, len(ev_user), _ptr(ev_user, C.c_int32), _ptr(ev_item, C.c_int32), flag))
        self.m, self.n = int(m), int(n)
        self.T = self.interaction_sizes()[2]

    def interaction_sizes(self):
        v = [C.c_int64() for _ in range(5)]
        self._ck(self.lib.yue_interaction_sizes(self.h, *[C.byref(x) for x in v]))
        return tuple(x.value for x in v)          # m, n, T, nnz, n_test

    def get_interactions(self):
        m, n, T, nnz, _ = self.interaction_sizes()
        ev_indptr, uq_indptr = np.empty(m + 1, np.int64), np.empty(m + 1, np.int64)
        ev_items, uq_items = np.empty(T, np.int32), np.empty(nnz, np.int32)
        self._ck(self.lib.yue_get_interactions(self.h, _ptr(ev_indptr, C.c_int64), _ptr(ev_items, C.c_int32),
                                               _ptr(uq_indptr, C.c_int64), _ptr(uq_items, C.c_int32)))
        return ev_indptr, ev_items, uq_indptr, uq_items

    def get_test_set(self):
        m, _, _, _, nt = self.interaction_sizes()
        indptr, items = np.empty(m + 1, np.int64), np.empty(nt, np.int32)
        self._ck(self.lib.yue_get_test_set(self.h, _ptr(indptr, C.c_int64), _ptr(items, C.c_int32)))
        return indptr, items

    def set_event_offsets(self, delta):
        """Per local user: global event index = local index + delta[user] (non-contiguous shards)."""
        delta = _as(delta, np.int64)
        if len(delta) != self.m:
            raise ValueError("one offset per local user")
        self._ck(self.lib.yue_set_event_offsets(self.h, _ptr(delta, C.c_int64)))

    def set_factors(self, P, Q):
        P, Q = _as(P, np.float32), _as(Q, np.float32)
        if P.shape[0] != self.m or Q.shape[0] != self.n or P.shape[1] != Q.shape[1]:
            raise ValueError("factor shapes %s %s do not match m=%d n=%d" % (P.shape, Q.shape, self.m, self.n))
        self.k = int(P.shape[1])
        self._ck(self.lib.yue_set_factors(self.h, self.k, _ptr(P, C.c_float), _ptr(Q, C.c_float)))

    def get_factors(self, P=None, Q=None):
        """Copy the tables back; pass preallocated (e.g. pinned) arrays to avoid an allocation."""
        if P is None:
            P = np.empty((self.m, self.k), dtype=np.float32)
        if Q is None:
            Q = np.empty((self.n, self.k), dtype=np.float32)
        assert P.dtype == np.float32 and Q.dtype == np.float32 and P.flags.c_contiguous and Q.flags.c_contiguous
        self._ck(self.lib.yue_get_factors(self.h, _ptr(P, C.c_float), _ptr(Q, C.c_float)))
        return P, Q

    # -- training --------------------------------------------------------------------------
    def sample_negatives(self, seed, epoch, slot=0):
        out = np.empty(self.T, dtype=np.int32)
        self._ck(self.lib.yue_sample_negatives(self.h, seed, epoch, slot, _ptr(out, C.c_int32)))
        return out

    def bpr_epoch(self, lr, regU, regI, seed, epoch, mode=MODE_HOGWILD, want_loss=True):
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_bpr_epoch(self.h, lr, regU, regI, seed, epoch, mode,
                                        C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def bpr_epoch_part(self, lr, regU, regI, seed, epoch, part, n_parts, mode=MODE_HOGWILD, want_loss=True):
        """The part-th of n_parts consecutive sub-epochs (users in stream order)."""
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_bpr_epoch_part(self.h, lr, regU, regI, seed, epoch, mode, part, n_parts,
                                             C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def bpr_apply(self, u, i, j, lr, regU, regI, mode=MODE_SERIAL, want_loss=True):
        u, i, j = _as(u, np.int32), _as(i, np.int32), _as(j, np.int32)
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_bpr_apply(self.h, _ptr(u, C.c_int32), _ptr(i, C.c_int32), _ptr(j, C.c_int32),
                                        len(u), lr, regU, regI, mode, C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def apr_epoch(self, lr, regU, regI, eps, regA, seed, epoch, slot=0, mode=MODE_HOGWILD, want_loss=True):
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_apr_epoch(self.h, lr, regU, regI, eps, regA, seed, epoch, slot, mode,
                                        C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def apr_apply(self, u, i, j, lr, regU, regI, eps, regA, mode=MODE_SERIAL, want_loss=True):
        u, i, j = _as(u, np.int32), _as(i, np.int32), _as(j, np.int32)
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_apr_apply(self.h, _ptr(u, C.c_int32), _ptr(i, C.c_int32), _ptr(j, C.c_int32),
                                        len(u), lr, regU, regI, eps, regA, mode, C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def cune_set_implicit(self, ip_indptr, ip_items):
        """Implicit positives per user (CUNE.py:95-113): tracks of the user's similar users that it has not played."""
        ip_indptr, ip_items = _as(ip_indptr, np.int64), _as(ip_items, np.int32)
        if len(ip_indptr) != self.m + 1:
            raise ValueError("ip_indptr must have m+1 entries")
        if len(ip_items) != ip_indptr[-1]:
            raise ValueError("ip_items does not match ip_indptr[-1]")
        self._ck(self.lib.yue_cune_set_implicit(self.h, _ptr(ip_indptr, C.c_int64), _ptr(ip_items, C.c_int32)))

    def cune_epoch(self, lr, regU, regI, s, seed, epoch, mode=MODE_HOGWILD):
        """One pass of CUNE's two-level BPR loop (CUNE.py:122-174); returns the loss."""
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_cune_epoch(self.h, float(lr), float(regU), float(regI), float(s), int(seed), int(epoch),
                                         int(mode), C.byref(loss)))
        return loss.value

    # ---- LightGCN (K9, csrc/lightgcn.cuh) ----
    def gcn_set_events(self, ev_user, ev_item):
        """The training events in FILE order: LightGCN's batches are consecutive slices of them (LightGCN.py:56-66)."""
        ev_user, ev_item = _as(ev_user, np.int32), _as(ev_item, np.int32)
        if ev_user.shape != ev_item.shape or ev_user.ndim != 1:
            raise ValueError("ev_user / ev_item must be equally long vectors")
        self._ck(self.lib.yue_gcn_set_events(self.h, len(ev_user), _ptr(ev_user, C.c_int32), _ptr(ev_item, C.c_int32)))
        self._gcn_T = len(ev_user)

    def gcn_epoch(self, batch_size, lr, reg, seed, epoch, n_layers=3, step_begin=0, step_end=-1):
        """Steps [step_begin, step_end) of one pass over the batches, in one launch; returns the per-step losses."""
        n_steps = (self._gcn_T + int(batch_size) - 1) // int(batch_size)
        end = n_steps if step_end < 0 else int(step_end)
        loss = np.zeros(max(end - int(step_begin), 0), dtype=np.float64)
        self._ck(self.lib.yue_gcn_epoch(self.h, int(n_layers), int(batch_size), float(lr), float(reg), int(seed), int(epoch),
                                        int(step_begin), end, _ptr(loss, C.c_double)))
        return loss

    def gcn_apply(self, u, i, j, lr, reg, n_layers=3):
        """One Adam step on the caller's triplets (parity hook); returns the batch loss."""
        u, i, j = _as(u, np.int32), _as(i, np.int32), _as(j, np.int32)
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_gcn_apply(self.h, int(n_layers), len(u), _ptr(u, C.c_int32), _ptr(i, C.c_int32), _ptr(j, C.c_int32),
                                        float(lr), float(reg), C.byref(loss)))
        return loss.value

    def gcn_finalize(self, n_layers=3):
        """P, Q <- the propagated tables predict() ranks with (LightGCN.py:45-47); the variables return on the next step."""
        self._ck(self.lib.yue_gcn_finalize(self.h, int(n_layers)))

    def gcn_moments(self):
        """Adam's state: (m_users, m_tracks, v_users, v_tracks, steps taken since set_factors)."""
        mu, vu = np.empty((self.m, self.k), np.float32), np.empty((self.m, self.k), np.float32)
        mt, vt = np.empty((self.n, self.k), np.float32), np.empty((self.n, self.k), np.float32)
        steps = C.c_int64(0)
        self._ck(self.lib.yue_gcn_moments(self.h, _ptr(mu, C.c_float), _ptr(mt, C.c_float), _ptr(vu, C.c_float), _ptr(vt, C.c_float),
                                          C.byref(steps)))
        return mu, mt, vu, vt, steps.value

    # ---- BPR's shipped Adam training (K10, csrc/bpr_adam.cuh) ----
    def bpr_adam_sample(self, seed, step, batch=512, negatives=100):
        """The batch of step `step`: (events[batch] into the event CSR, negatives[batch, negatives]) -- check hook."""
        ev, neg = np.empty(int(batch), np.int32), np.empty((int(batch), int(negatives)), np.int32)
        self._ck(self.lib.yue_bpr_adam_sample(self.h, int(seed), int(step), int(batch), int(negatives), _ptr(ev, C.c_int32),
                                              _ptr(neg, C.c_int32)))
        return ev, neg

    def bpr_adam_steps(self, batch, negatives, lr, reg, seed, step_begin, step_end, want_loss=True):
        """Adam steps [step_begin, step_end) on sampled batch x negatives triplets; returns the per-step losses."""
        loss = np.zeros(max(int(step_end) - int(step_begin), 0), dtype=np.float64)
        self._ck(self.lib.yue_bpr_adam_steps(self.h, int(batch), int(negatives), float(lr), float(reg), int(seed), int(step_begin),
                                             int(step_end), _ptr(loss, C.c_double) if want_loss else None))
        return loss if want_loss else None

    def bpr_adam_apply(self, u, i, j, lr, reg):
        """One Adam step on the caller's triplets (parity hook); returns the loss."""
        u, i, j = _as(u, np.int32), _as(i, np.int32), _as(j, np.int32)
        if not (u.shape == i.shape == j.shape) or u.ndim != 1:
            raise ValueError("u / i / j must be equally long vectors")
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_bpr_adam_apply(self.h, len(u), _ptr(u, C.c_int32), _ptr(i, C.c_int32), _ptr(j, C.c_int32),
                                             float(lr), float(reg), C.byref(loss)))
        return loss.value

    def bpr_adam_moments(self):
        """Adam's state of this path: (m_users, m_tracks, v_users, v_tracks, steps taken since set_factors)."""
        mu, vu = np.empty((self.m, self.k), np.float32), np.empty((self.m, self.k), np.float32)
        mt, vt = np.empty((self.n, self.k), np.float32), np.empty((self.n, self.k), np.float32)
        steps = C.c_int64(0)
        self._ck(self.lib.yue_bpr_adam_moments(self.h, _ptr(mu, C.c_float), _ptr(mt, C.c_float), _ptr(vu, C.c_float),
                                               _ptr(vt, C.c_float), C.byref(steps)))
        return mu, mt, vu, vt, steps.value

    def wrmf_sweep(self, side, reg, alpha=10.0, want_loss=False):
        """One WRMF half-sweep (0: every user row from the track table, 1: every track row from the user table)."""
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_wrmf_sweep(self.h, int(side), float(reg), float(alpha), C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def wrmf_sweep_rows(self, side, row_begin, row_end, reg, alpha=10.0, want_loss=False):
        """The half-sweep restricted to rows [row_begin, row_end) (multi-GPU: every rank solves a range)."""
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_wrmf_sweep_rows(self.h, int(side), int(row_begin), int(row_end), float(reg), float(alpha),
                                              C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def wrmf_pair_counts(self):
        """(uq_counts[nnz], it_indptr[n+1], it_users[nnz], it_counts[nnz]): plays per unique pair and the track-major pairs."""
        nnz = self.interaction_sizes()[3]
        cnt, itp = np.empty(nnz, np.int32), np.empty(self.n + 1, np.int64)
        itu, itc = np.empty(nnz, np.int32), np.empty(nnz, np.int32)
        self._ck(self.lib.yue_wrmf_pair_counts(self.h, _ptr(cnt, C.c_int32), _ptr(itp, C.c_int64), _ptr(itu, C.c_int32),
                                               _ptr(itc, C.c_int32)))
        return cnt, itp, itu, itc

    def frob2(self):
        p2, q2 = C.c_double(), C.c_double()
        self._ck(self.lib.yue_frob2(self.h, C.byref(p2), C.byref(q2)))
        return p2.value, q2.value

    # -- scoring ---------------------------------------------------------------------------
    def predict(self, user):
        out = np.empty(self.n, dtype=np.float32)
        self._ck(self.lib.yue_predict(self.h, int(user), _ptr(out, C.c_float)))
        return out

    def rank_topn(self, users, N, algo=RANK_AUTO, ids=None, scores=None):
        users = _as(users, np.int32)
        B = len(users)
        if ids is None:
            ids = np.empty((B, N), dtype=np.int32)
        if scores is None:
            scores = np.empty((B, N), dtype=np.float32)
        self._ck(self.lib.yue_rank_topn(self.h, _ptr(users, C.c_int32), B, int(N), algo,
                                        _ptr(ids, C.c_int32), _ptr(scores, C.c_float)))
        return ids, scores

    def set_test_set(self, test_indptr, test_items):
        """Held-out tracks per local user (sorted unique CSR), for rank_metrics."""
        test_indptr, test_items = _as(test_indptr, np.int64), _as(test_items, np.int32)
        if len(test_indptr) != self.m + 1 or len(test_items) != test_indptr[-1]:
            raise ValueError("test CSR does not match m=%d" % self.m)
        self._ck(self.lib.yue_set_test_set(self.h, _ptr(test_indptr, C.c_int64), _ptr(test_items, C.c_int32)))

    def rank_metrics(self, cuts):
        """Metrics of the lists of the last rank_topn call, per cut-off n: dict with hits (int), precision,
        recall, F1, MAP, NDCG, distinct (coverage numerator) -- evaluation/measure.py semantics."""
        cuts = _as(cuts, np.int32)
        sums = np.zeros((len(cuts), 4), dtype=np.float64)
        distinct = np.zeros(len(cuts), dtype=np.int64)
        self._ck(self.lib.yue_rank_metrics(self.h, len(cuts), _ptr(cuts, C.c_int32), _ptr(sums, C.c_double), _ptr(distinct, C.c_int64)))
        return sums, distinct

    # -- multi-GPU plumbing ----------------------------------------------------------------
    def q_snapshot(self):
        self._ck(self.lib.yue_q_snapshot(self.h))

    def q_delta_pack(self):
        self._ck(self.lib.yue_q_delta_pack(self.h))

    def set_delta_weights(self, w):
        """Per-track factor for the summed Q deltas (sharding.saturation_weights); None = plain sum."""
        if w is None:
            self._ck(self.lib.yue_set_delta_weights(self.h, None))
            return
        w = _as(w, np.float32)
        if len(w) != self.n:
            raise ValueError("one weight per track")
        self._ck(self.lib.yue_set_delta_weights(self.h, _ptr(w, C.c_float)))

    def q_delta_apply(self):
        self._ck(self.lib.yue_q_delta_apply(self.h))

    def device_buffer(self, which):
        p, nbytes = C.c_void_p(), C.c_size_t()
        self._ck(self.lib.yue_device_buffer(self.h, which, C.byref(p), C.byref(nbytes)))
        return p.value, nbytes.value

    def stream_ptr(self):
        s = C.c_void_p()
        self._ck(self.lib.yue_stream(self.h, C.byref(s)))
        return s.value or 0

    def comm_init(self, nranks, rank, unique_id):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._ck(self.lib.yue_comm_init(self.h, nranks, rank, buf))

    def allreduce_q_delta(self):
        self._ck(self.lib.yue_allreduce_q_delta(self.h))

    # shared hot rows + overlapped exchange of the tail (include/yue_b200.h, "multi-GPU, round 2")
    def hot_tracks(self):
        n = C.c_int(0)
        out = np.empty(1024, dtype=np.int32)                   # kHotSlots = 248
        self._ck(self.lib.yue_hot_tracks(self.h, _ptr(out, C.c_int32), C.byref(n)))
        return out[:n.value].copy()

    def set_hot_tracks(self, tracks, counts, total_events):
        tracks, counts = _as(tracks, np.int32), _as(counts, np.int64)
        if len(tracks) != len(counts):
            raise ValueError("one count per hot track")
        self._ck(self.lib.yue_set_hot_tracks(self.h, _ptr(tracks, C.c_int32), _ptr(counts, C.c_int64), len(tracks), int(total_events)))

    def hot_table_export(self):
        """(64-byte CUDA IPC handle, device pointer) of this handle's hot-row table."""
        buf, p = C.create_string_buffer(64), C.c_void_p()
        self._ck(self.lib.yue_hot_table_export(self.h, buf, C.byref(p)))
        return buf.raw, p.value

    def hot_table_open(self, ipc_handle):
        p = C.c_void_p()
        self._ck(self.lib.yue_hot_table_open(self.h, C.create_string_buffer(bytes(ipc_handle), 64), C.byref(p)))
        return p.value

    def enable_peer(self, peer_device):
        self._ck(self.lib.yue_enable_peer(self.h, int(peer_device)))

    def hot_share(self, nranks, rank, tables):
        arr = (C.c_void_p * nranks)(*[C.c_void_p(t) if t else C.c_void_p(None) for t in tables])
        self._ck(self.lib.yue_hot_share(self.h, int(nranks), int(rank), arr))

    def hot_pull(self):
        self._ck(self.lib.yue_hot_pull(self.h))

    def hot_unshare(self):
        self._ck(self.lib.yue_hot_unshare(self.h))

    def q_exchange_begin(self):
        self._ck(self.lib.yue_q_exchange_begin(self.h))

    def q_exchange_reduce(self):
        self._ck(self.lib.yue_q_exchange_reduce(self.h))

    def q_exchange_reduce_peers(self, deltas):
        """deltas[r]: rank r's BUF_Q_DELTA pointer in this process (None = own)."""
        arr = (C.c_void_p * len(deltas))(*[C.c_void_p(t) if t else C.c_void_p(None) for t in deltas])
        self._ck(self.lib.yue_q_exchange_reduce_peers(self.h, len(deltas), arr))

    def q_exchange_finish(self, quiescent=False):
        self._ck(self.lib.yue_q_exchange_finish(self.h, 1 if quiescent else 0))

    def stream2_ptr(self):
        s = C.c_void_p()
        self._ck(self.lib.yue_stream2(self.h, C.byref(s)))
        return s.value or 0

    def set_sgd_concurrency(self, n_warps, n_ctas=0):
        """Warps / CTAs of the Hogwild epoch kernels (0, 0 = automatic)."""
        self._ck(self.lib.yue_set_sgd_concurrency(self.h, int(n_warps), int(n_ctas)))

    def apr_epoch_part(self, lr, regU, regI, eps, regA, seed, epoch, part, n_parts, slot=0, mode=MODE_HOGWILD, want_loss=True):
        loss = C.c_double(0.0)
        self._ck(self.lib.yue_apr_epoch_part(self.h, lr, regU, regI, eps, regA, seed, epoch, slot, mode, part, n_parts,
                                             C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    # -- measurement -----------------------------------------------------------------------
    def timer_start(self):
        self._ck(self.lib.yue_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        self._ck(self.lib.yue_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def launch_count(self):
        n = C.c_int64()
        self._ck(self.lib.yue_launch_count(self.h, C.byref(n)))
        return n.value

    def rank_stats(self):
        """(rows redone by the exact kernel, rows spilled into the pool) of the last tcgen05 ranking call"""
        a, b = C.c_int64(), C.c_int64()
        self._ck(self.lib.yue_rank_stats(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def flush_l2(self):
        self._ck(self.lib.yue_flush_l2(self.h))


def device_count():
    n = C.c_int(0)
    _lib.load().yue_device_count(C.byref(n))
    return n.value


def comm_unique_id():
    lib = _lib.load()
    buf = C.create_string_buffer(128)
    rc = lib.yue_comm_unique_id(buf)
    if rc:
        raise YueError(rc, lib.yue_last_error(None).decode())
    return buf.raw
