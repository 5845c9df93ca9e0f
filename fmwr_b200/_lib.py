"""ctypes binding of libfmwr_b200.so (include/fmwr_b200.h).

The library is the product; this module only loads it and mirrors its structs.  There is no
fallback: if the shared object is missing or a call fails the error is raised.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FMWR_LIB_PATH") or os.path.join(HERE, "libfmwr_b200.so")   # override: kernel-variant experiments only

CLASSIFICATION, REGRESSION = 10, 20
MCMC, ALS, SGD, FTRL, TDAP = 100, 200, 300, 500, 600
LL, AUC, ACC, RMSE, MSE, MAE = 0, 111, 222, 333, 444, 555
F32, F64 = 0, 1
MODE_EXACT, MODE_MINIBATCH = 0, 1
LINK_NONE, LINK_LOGISTIC, LINK_PROBIT_TABLE, LINK_CLAMP = 0, 1, 2, 3
COMPAT_SKIP_ROW0, COMPAT_TDAP_ZW_INDEX, COMPAT_MCMC_W_SD, COMPAT_MCMC_VMU_IDX, COMPAT_REFERENCE = 1, 2, 4, 8, 15

SOLVERS = {"MCMC": MCMC, "ALS": ALS, "SGD": SGD, "FTRL": FTRL, "TDAP": TDAP}
TASKS = {"CLASSIFICATION": CLASSIFICATION, "REGRESSION": REGRESSION}
METRICS = {"LL": LL, "AUC": AUC, "ACC": ACC, "RMSE": RMSE, "MSE": MSE, "MAE": MAE}


class ModelCfg(C.Structure):
    _fields_ = [("task", C.c_int32), ("keep_w0", C.c_int32), ("keep_w1", C.c_int32), ("k", C.c_int32),
                ("l2_w0", C.c_double), ("l1_w1", C.c_double), ("l2_w1", C.c_double), ("l1_v", C.c_double),
                ("l2_v", C.c_double)]


class SolverCfg(C.Structure):
    _fields_ = [("solver", C.c_int32), ("max_iter", C.c_int32), ("random_step", C.c_int32),
                ("learn_rate", C.c_double),
                ("alpha_w", C.c_double), ("alpha_v", C.c_double), ("beta_w", C.c_double), ("beta_v", C.c_double),
                ("gamma", C.c_double), ("min_target", C.c_double), ("max_target", C.c_double),
                ("mode", C.c_int32), ("batch_size", C.c_int32), ("precision", C.c_int32), ("compat", C.c_int32),
                ("enable_v", C.c_int32),
                ("visit_order", C.c_void_p), ("n_visit", C.c_int64),
                ("step_size", C.c_int32), ("metric", C.c_int32), ("convergence", C.c_double),
                ("normals", C.c_void_p), ("n_normals", C.c_int64),
                ("gammas", C.c_void_p), ("n_gammas", C.c_int64),
                ("rands", C.c_void_p), ("n_rands", C.c_int64),
                ("seed", C.c_uint64), ("warm_state", C.c_int32)]


class Trace(C.Structure):
    _fields_ = [("max_rec", C.c_int32), ("n_rec", C.c_int32), ("convergent", C.c_int32), ("iters_done", C.c_int32),
                ("eval_train", C.c_void_p), ("rec_index", C.c_void_p),
                ("snap_w0", C.c_void_p), ("snap_w", C.c_void_p), ("snap_v", C.c_void_p)]


class FmwrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("fmwr_b200 error %d: %s" % (code, msg))
        self.code = code
        self.msg = msg


_lib = None


def lib():
    """load the CUDA engine; raises when it has not been built (no fallback)"""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FmwrError(-1, "libfmwr_b200.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                "or `make -C fmwr_b200/csrc`")
        _lib = C.CDLL(LIB_PATH)
        _lib.fmwr_last_error.restype = C.c_char_p
    return _lib


def check(rc):
    if rc != 0:
        raise FmwrError(rc, lib().fmwr_last_error().decode(errors="replace"))


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def exported_symbols():
    """function names declared in include/fmwr_b200.h (used by the symbol test)"""
    import re
    hdr = os.path.join(os.path.dirname(HERE), "include", "fmwr_b200.h")
    txt = open(hdr).read()
    return sorted(set(re.findall(r"\b(fmwr_[a-z0-9_]+)\s*\(", txt)))


class Context:
    """one GPU (fmwr_ctx)"""

    def __init__(self, device=0):
        self.h = C.c_void_p()
        check(lib().fmwr_ctx_create(int(device), C.byref(self.h)))

    def close(self):
        if self.h:
            lib().fmwr_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        check(lib().fmwr_ctx_sync(self.h))

    def timer_start(self):
        check(lib().fmwr_timer_start(self.h))

    def timer_stop_ms(self):
        ms = C.c_double()
        check(lib().fmwr_timer_stop_ms(self.h, C.byref(ms)))
        return ms.value

    def launches(self):
        n = C.c_int64()
        check(lib().fmwr_ctx_launch_count(self.h, C.byref(n)))
        return n.value

    def transfer_bytes(self):
        """(host -> device, device -> host) bytes the library has copied for the caller on this context"""
        a, b = C.c_int64(), C.c_int64()
        check(lib().fmwr_ctx_transfer_bytes(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def flush_l2(self):
        check(lib().fmwr_flush_l2(self.h))

    # -- multi-GPU communicator (NCCL) ----------------------------------------------------------------
    @staticmethod
    def comm_unique_id():
        buf = (C.c_uint8 * 128)()
        check(lib().fmwr_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, id128, rank, world):
        buf = (C.c_uint8 * 128).from_buffer_copy(id128)
        check(lib().fmwr_comm_init(self.h, buf, C.c_int32(rank), C.c_int32(world)))

    def comm_destroy(self):
        check(lib().fmwr_comm_destroy(self.h))

    @staticmethod
    def comm_peer_bytes(batch_size, k, world):
        lib().fmwr_comm_peer_bytes.restype = C.c_int64
        return int(lib().fmwr_comm_peer_bytes(C.c_int64(batch_size), C.c_int32(k), C.c_int32(world)))

    def comm_peer_alloc(self, nbytes):
        buf = (C.c_uint8 * 64)()
        check(lib().fmwr_comm_peer_alloc(self.h, C.c_int64(nbytes), buf))
        return bytes(buf)

    def comm_peer_open(self, handles):
        raw = b"".join(handles)
        buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw)
        check(lib().fmwr_comm_peer_open(self.h, buf))

    def sort_pairs(self, keys, bits):
        """the engine's stable radix sort on a host array of uint32 / uint64 keys -> (sorted keys, permutation)"""
        keys = np.ascontiguousarray(keys)
        assert keys.dtype in (np.uint32, np.uint64)
        out = np.zeros_like(keys)
        perm = np.zeros(keys.size, np.uint32)
        check(lib().fmwr_sort_pairs(self.h, C.c_int32(keys.itemsize), C.c_int64(keys.size), C.c_int32(bits), ptr(keys), ptr(out), ptr(perm)))
        return out, perm

    def link_table(self, which, x):
        x = np.ascontiguousarray(x, np.float64)
        out = np.zeros_like(x)
        check(lib().fmwr_link_table_eval(self.h, int(which), C.c_int64(x.size), ptr(x), ptr(out)))
        return out


class Data:
    """device-resident dataset (fmwr_data)"""

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self.h = handle

    @classmethod
    def from_r_lists(cls, ctx, n, p, row_size, col_idx, value, labels=None):
        """the fm.matrix layout: value f64, col_idx i32, row_size i32 (R/fm_matrix.R:25-34)"""
        row_size = np.ascontiguousarray(row_size, np.int32)
        col_idx = np.ascontiguousarray(col_idx, np.int32)
        value = np.ascontiguousarray(value, np.float64)
        lab = np.ascontiguousarray(labels, np.float64) if labels is not None else None
        h = C.c_void_p()
        check(lib().fmwr_data_create(ctx.h, C.c_int64(n), C.c_int64(p), C.c_int64(col_idx.size), ptr(row_size),
                                     ptr(col_idx), ptr(value), ptr(lab), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_csr32(cls, ctx, n, p, rowptr, col, val, labels=None):
        rowptr = np.ascontiguousarray(rowptr, np.uint32)
        col = np.ascontiguousarray(col, np.uint32)
        val = np.ascontiguousarray(val, np.float32)
        lab = np.ascontiguousarray(labels, np.float32) if labels is not None else None
        h = C.c_void_p()
        check(lib().fmwr_data_create_csr32(ctx.h, C.c_int64(n), C.c_int64(p), C.c_int64(col.size), ptr(rowptr), ptr(col),
                                           ptr(val), ptr(lab), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def synth(cls, ctx, n, field_size, skew=None, value_mode=0, label_mode=1, noise=0.1, seed=20240601):
        fs = np.ascontiguousarray(field_size, np.int64)
        sk = np.ascontiguousarray(skew if skew is not None else np.zeros(fs.size), np.int32)
        h = C.c_void_p()
        check(lib().fmwr_data_synth(ctx.h, C.c_int64(n), C.c_int32(fs.size), ptr(fs), ptr(sk), C.c_int32(value_mode),
                                    C.c_int32(label_mode), C.c_double(noise), C.c_uint64(seed), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def synth_rows(cls, ctx, row_begin, n_rows, field_size, skew=None, value_mode=0, label_mode=0, noise=0.1, seed=20240601):
        fs = np.ascontiguousarray(field_size, np.int64)
        sk = np.ascontiguousarray(skew if skew is not None else np.zeros(fs.size), np.int32)
        h = C.c_void_p()
        check(lib().fmwr_data_synth_rows(ctx.h, C.c_int64(row_begin), C.c_int64(n_rows), C.c_int32(fs.size), ptr(fs), ptr(sk),
                                         C.c_int32(value_mode), C.c_int32(label_mode), C.c_double(noise), C.c_uint64(seed), C.byref(h)))
        return cls(ctx, h)

    def slice_columns(self, c0, c1):
        h = C.c_void_p()
        check(lib().fmwr_data_slice_columns(self.h, C.c_int64(c0), C.c_int64(c1), C.byref(h)))
        return Data(self.ctx, h)

    @classmethod
    def concat_rows(cls, parts):
        arr = (C.c_void_p * len(parts))(*[q.h for q in parts])
        h = C.c_void_p()
        check(lib().fmwr_data_concat_rows(arr, C.c_int32(len(parts)), C.byref(h)))
        return cls(parts[0].ctx, h)

    def close(self):
        if self.h:
            lib().fmwr_data_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def shape(self):
        n, p, nnz = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib().fmwr_data_shape(self.h, C.byref(n), C.byref(p), C.byref(nnz)))
        return n.value, p.value, nnz.value

    def get_csr(self, labels=True):
        n, p, nnz = self.shape()
        rowptr = np.zeros(n + 1, np.uint32)
        col = np.zeros(nnz, np.uint32)
        val = np.zeros(nnz, np.float32)
        y = np.zeros(n, np.float32) if labels else None
        check(lib().fmwr_data_get_csr(self.h, ptr(rowptr), ptr(col), ptr(val), ptr(y)))
        return rowptr, col, val, y

    def minibatch_info(self, batch_size, compat=COMPAT_REFERENCE):
        nb, ns, ne = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib().fmwr_data_minibatch_info(self.h, C.c_int32(batch_size), C.c_int32(compat), C.byref(nb), C.byref(ns), C.byref(ne)))
        return dict(n_batches=nb.value, n_segments=ns.value, n_entries=ne.value)

    def transpose(self):
        check(lib().fmwr_data_transpose(self.h))

    def get_csc(self):
        n, p, nnz = self.shape()
        colptr = np.zeros(p + 1, np.uint32)
        row = np.zeros(nnz, np.uint32)
        val = np.zeros(nnz, np.float32)
        check(lib().fmwr_data_get_csc(self.h, ptr(colptr), ptr(row), ptr(val)))
        return colptr, row, val

    def scales(self, norm_cols):
        n, p, nnz = self.shape()
        nc = np.ascontiguousarray(norm_cols, np.int32)
        mean = np.zeros(p)
        sd = np.zeros(p)
        check(lib().fmwr_data_scales(self.h, ptr(nc), C.c_int64(nc.size), ptr(mean), ptr(sd)))
        return mean, sd

    def set_labels(self, labels):
        lab = np.ascontiguousarray(labels, np.float64)
        check(lib().fmwr_data_set_labels(self.h, ptr(lab)))

    def restore_values(self):
        check(lib().fmwr_data_restore_values(self.h))

    def normalize(self, mean, sd):
        mean = np.ascontiguousarray(mean, np.float64)
        sd = np.ascontiguousarray(sd, np.float64)
        check(lib().fmwr_data_normalize(self.h, ptr(mean), ptr(sd)))


class Model:
    """device-resident parameters (fmwr_model)"""

    def __init__(self, ctx, cfg, p, precision=F32):
        self.ctx = ctx
        self.cfg = cfg
        self.p = int(p)
        self.k = int(cfg.k)
        self.h = C.c_void_p()
        check(lib().fmwr_model_create(ctx.h, C.byref(cfg), C.c_int64(p), C.c_int32(precision), C.byref(self.h)))

    def close(self):
        if self.h:
            lib().fmwr_model_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set(self, w0, w, v):
        w = np.ascontiguousarray(w, np.float64)
        v = np.ascontiguousarray(v, np.float64) if self.k > 0 else None
        assert w.size == self.p and (v is None or v.size == self.p * self.k)
        check(lib().fmwr_model_set(self.h, C.c_double(w0), ptr(w), ptr(v)))

    def get(self):
        w0 = C.c_double()
        w = np.zeros(self.p)
        v = np.zeros((self.p, self.k))
        check(lib().fmwr_model_get(self.h, C.byref(w0), ptr(w), ptr(v) if self.k > 0 else None))
        return w0.value, w, v

    def state_info(self):
        solver, ns = C.c_int32(), C.c_int32()
        check(lib().fmwr_model_state_info(self.h, C.byref(solver), C.byref(ns)))
        return solver.value, ns.value

    def get_state(self):
        """(solver, scal[8], sw[n_state][p], sv[n_state][p][k]) of the last training call on this handle"""
        solver, ns = self.state_info()
        scal = np.zeros(8)
        sw = np.zeros((ns, self.p))
        sv = np.zeros((ns, self.p, self.k))
        check(lib().fmwr_model_get_state(self.h, ptr(scal), ptr(sw), ptr(sv)))
        return dict(solver=solver, scal=scal, sw=sw, sv=sv)

    def set_state(self, st):
        sw = np.ascontiguousarray(st["sw"], np.float64); sv = np.ascontiguousarray(st["sv"], np.float64)
        scal = np.ascontiguousarray(st["scal"], np.float64)
        check(lib().fmwr_model_set_state(self.h, C.c_int32(int(st["solver"])), C.c_int32(sw.shape[0]), ptr(scal), ptr(sw), ptr(sv)))

    def init_random(self, mean=0.0, sd=0.01, seed=20240603):
        check(lib().fmwr_model_init_random(self.h, C.c_double(mean), C.c_double(sd), C.c_uint64(seed)))


def predict_dev(ctx, model, data, link=LINK_NONE, lo=0.0, hi=0.0):
    check(lib().fmwr_predict_dev(ctx.h, model.h, data.h, C.c_int32(link), C.c_double(lo), C.c_double(hi)))


def predict_fetch(ctx, data):
    n = data.shape()[0]
    out = np.zeros(n)
    check(lib().fmwr_predict_fetch(ctx.h, data.h, ptr(out)))
    return out


def evaluate_dev(ctx, data, task, metric):
    out = C.c_double()
    check(lib().fmwr_evaluate_dev(ctx.h, data.h, C.c_int32(task), C.c_int32(metric), C.byref(out)))
    return out.value


class TraceBuf:
    """caller-allocated fmwr_trace"""

    def __init__(self, max_rec, p=0, k=0, snapshots=False):
        self.max_rec = int(max_rec)
        self.eval_train = np.zeros(max(self.max_rec, 1))
        self.rec_index = np.zeros(max(self.max_rec, 1), np.int32)
        self.snap_w0 = np.zeros(max(self.max_rec, 1)) if snapshots else None
        self.snap_w = np.zeros((max(self.max_rec, 1), p)) if snapshots else None
        self.snap_v = np.zeros((max(self.max_rec, 1), p, k)) if snapshots else None
        self.c = Trace(max_rec=self.max_rec, eval_train=ptr(self.eval_train), rec_index=ptr(self.rec_index),
                       snap_w0=ptr(self.snap_w0), snap_w=ptr(self.snap_w), snap_v=ptr(self.snap_v))

    def result(self):
        nr = min(self.c.n_rec, self.max_rec)
        d = dict(n_rec=self.c.n_rec, convergent=bool(self.c.convergent), iters_done=self.c.iters_done,
                 eval_train=self.eval_train[:nr].copy(), rec_index=self.rec_index[:nr].copy())
        if self.snap_w0 is not None:
            d.update(snap_w0=self.snap_w0[:nr].copy(), snap_w=self.snap_w[:nr].copy(), snap_v=self.snap_v[:nr].copy())
        return d


def train_dev(ctx, model, data, scfg, trace=None, keep=()):
    """keep: numpy arrays referenced by pointer fields of scfg (kept alive for the call)"""
    check(lib().fmwr_train_dev(ctx.h, model.h, data.h, C.byref(scfg), C.byref(trace.c) if trace is not None else None))
    del keep


def train_posterior_dev(ctx, model, data, scfg, burn_in, evals=(), trace=None, keep=()):
    """train_dev plus the MCMC posterior mean of draws burn_in+1 .. max_iter: afterwards predict_fetch(ctx, data) and
    predict_fetch(ctx, e) for every e in evals return the means (an entry of None passes a null handle)"""
    arr = (C.c_void_p * max(len(evals), 1))(*[e.h if e is not None else None for e in evals])
    check(lib().fmwr_train_posterior_dev(ctx.h, model.h, data.h, C.byref(scfg), C.byref(trace.c) if trace is not None else None,
                                         C.c_int32(burn_in), arr if len(evals) else None, C.c_int32(len(evals))))
    del keep
