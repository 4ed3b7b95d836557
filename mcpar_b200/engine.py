"""ctypes binding of include/mcgpu.h -- the only way Python reaches the CUDA engine.

Host-side mirror of the reference's interface for the hot path: `Engine` plays the
role of `MCPar` (src/mcpar.hh:10-91) + `MCout` (src/mcout.hh:13-51) for one GPU.
There is no CPU path here: if libmcgpu.so is missing, or no CUDA device is visible,
construction raises.
"""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MCGPU_LIB") or os.path.join(HERE, "libmcgpu.so")   # MCGPU_LIB: A/B experiments with alternative builds

LIK = {"rosenbrock1": 0, "rosenbrock2": 1, "gaussian": 2, "dualgaussian": 3, "gaussmix": 4, "host": 100, "plugin": 101}
MODE = {"normal": 0, "verify": 1, "replay_local": 2}
ERRORS = {-1: "EINVAL", -2: "ENODEVICE", -3: "ECUDA", -4: "ESTATE", -5: "ENOMEM", -6: "ESTREAM",
          -7: "EPEER"}
P2P_HANDLE_BYTES = 64

EXPORTS = [
    "mcgpu_version", "mcgpu_device_count", "mcgpu_last_error", "mcgpu_create", "mcgpu_destroy",
    "mcgpu_set_stream", "mcgpu_set_likelihood", "mcgpu_set_covariance", "mcgpu_set_state",
    "mcgpu_set_streams", "mcgpu_burnin", "mcgpu_sample_begin", "mcgpu_sample", "mcgpu_sample_group",
    "mcgpu_set_state_sobol", "mcgpu_set_state_host", "mcgpu_step_propose", "mcgpu_step_accept",
    "mcgpu_exchange_begin", "mcgpu_exchange_end", "mcgpu_p2p_export", "mcgpu_p2p_attach",
    "mcgpu_p2p_attach_local", "mcgpu_burnin_group", "mcgpu_tuning_counters", "mcgpu_burnin_some",
    "mcgpu_tune", "mcgpu_synchronize", "mcgpu_get_state", "mcgpu_get_factor", "mcgpu_get_musig",
    "mcgpu_get_trace", "mcgpu_history_read", "mcgpu_history_attach_host", "mcgpu_history_attach_host_f32",
    "mcgpu_history_maxlike", "mcgpu_history_moments",
    "mcgpu_checkpoint_size", "mcgpu_checkpoint_save", "mcgpu_checkpoint_load",
    "mcgpu_get_stats", "mcgpu_device_ptr", "mcgpu_loglik", "mcgpu_qriguess",
    "mcgpu_set_likelihood_plugin", "mcgpu_loglik_plugin",
    "mcgpu_measure_fp64_peak",
]


class McgpuError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("mode", C.c_int32),
                ("nparam", C.c_int32), ("nchain", C.c_int64), ("chain0", C.c_int64),
                ("nchain_total", C.c_int64), ("chains_per_rank", C.c_int32), ("sync", C.c_int32),
                ("pl", C.c_double), ("armin", C.c_double), ("armax", C.c_double),
                ("dfac", C.c_double), ("ifac", C.c_double), ("seed", C.c_uint64),
                ("coin_group", C.c_int32), ("pool_m", C.c_int32), ("thin", C.c_int32),
                ("trace", C.c_int32), ("history_steps", C.c_int64),
                ("remote_mode", C.c_int32), ("pool_lag", C.c_int32)]

REMOTE_MODE = {"reference": 0, "maxmix": 0, "summix": 1, "murray": 1, 0: 0, 1: 1}


class Stats(C.Structure):
    _fields_ = [("burn_steps", C.c_int64), ("main_steps", C.c_int64), ("accepted", C.c_int64),
                ("tried", C.c_int64), ("kernel_launches", C.c_int64), ("remote_steps", C.c_int64),
                ("remote_iterations", C.c_int64), ("history_rows", C.c_int64),
                ("device_ms", C.c_double), ("exchange_wait_ns", C.c_int64), ("exchange_waits", C.c_int64),
                ("exact_fallbacks", C.c_int64)]


_lib = None


def load():
    """dlopen libmcgpu.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise McgpuError("libmcgpu.so is not built: run `python -m mcpar_b200.build` "
                             "(or __graft_entry__.build()); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        lib.mcgpu_version.restype = C.c_char_p
        lib.mcgpu_last_error.restype = C.c_char_p
        lib.mcgpu_last_error.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _check(rc, handle=None):
    if rc != 0:
        msg = load().mcgpu_last_error(handle)
        raise McgpuError("%s: %s" % (ERRORS.get(rc, rc), msg.decode() if msg else ""))


def device_count():
    return load().mcgpu_device_count()


def _plugin_path(lik, plugin):
    if lik == "plugin" and not plugin:
        raise ValueError('likelihood "plugin" needs plugin=<path of the plugin cubin> (mcpar_b200/plugin.py builds one)')
    if lik != "plugin" and plugin:
        raise ValueError('plugin= is given but the likelihood is %r, not "plugin"' % (lik,))
    return os.fsencode(os.path.abspath(plugin)) if plugin else None


def loglik(lik, nparam, x, par=None, device=0, plugin=None):
    """VLFunc::operator()(npset, x, y) on the GPU (src/vlfunc.hh:11); lik="plugin" evaluates the plugin cubin
    `plugin` (built for nparam)."""
    path = _plugin_path(lik, plugin)
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, nparam)
    y = np.empty(x.shape[0], dtype=np.float64)
    par_a = None if par is None else np.ascontiguousarray(par, dtype=np.float64).ravel()
    npar = 0 if par is None else par_a.size
    if path:
        _check(load().mcgpu_loglik_plugin(device, path, nparam, _p(par_a), npar, x.shape[0], _p(x), _p(y)))
    else:
        _check(load().mcgpu_loglik(device, LIK[lik], nparam, _p(par_a), npar, x.shape[0], _p(x), _p(y)))
    return y


def qriguess(rank, npset, nparam, plo, phi, device=0):
    """mcutil::qriguess (src/mcutil.cc:3-34) on the GPU."""
    plo = np.ascontiguousarray(plo, dtype=np.float64); phi = np.ascontiguousarray(phi, dtype=np.float64)
    out = np.empty(npset * nparam, dtype=np.float64)
    _check(load().mcgpu_qriguess(device, rank, npset, nparam, _p(plo), _p(phi), _p(out)))
    return out.reshape(npset, nparam)


def measure_fp64_peak(device=0):
    v = C.c_double(0)
    _check(load().mcgpu_measure_fp64_peak(device, C.byref(v)))
    return v.value


class DevicePtr:
    """A raw device range exposing __cuda_array_interface__ so torch can alias it
    (torch.as_tensor(ptr, device='cuda')) for the NCCL exchange."""

    def __init__(self, ptr, nbytes, dtype="<f8"):
        item = np.dtype(dtype).itemsize
        self.__cuda_array_interface__ = {"shape": (nbytes // item,), "typestr": dtype,
                                         "data": (ptr, False), "version": 2}
        self.ptr, self.nbytes = ptr, nbytes


def p2p_attach_local(engines):
    """Several engines of ONE process (same or different devices) exchange peer to peer."""
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    _check(load().mcgpu_p2p_attach_local(arr, len(engines)), engines[0].h)
    for e in engines:
        e.p2p = True


def sample_group(engines, nsteps):
    """mcgpu_sample on several peer-to-peer engines of ONE process, one exchange window at a time, in turn."""
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    _check(load().mcgpu_sample_group(arr, len(engines), nsteps), engines[0].h)


def burnin_group(engines, nburn):
    """Burn-in of several sharded engines of ONE process with job-wide tuning counters."""
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    _check(load().mcgpu_burnin_group(arr, len(engines), nburn), engines[0].h)


class Engine:
    """One GPU's share of an MCPar run.

    Mirrors MCPar(np, nc, mpisiz, mpirank, pl, armin, armax, dfac, ifac, sync)
    (src/mcpar.hh:32-33); `run` mirrors MCPar::run(nsamp, nburn, pinit, L, out, incov).
    """

    def __init__(self, nparam, nchain, *, mode="normal", nchain_total=None, chain0=0,
                 chains_per_rank=0, pl=0.9, armin=0.2, armax=0.5, dfac=0.2, ifac=1.5, sync=10,
                 seed=8675309, coin_group=32, pool_m=0, thin=1, trace=0, history_steps=0,
                 device=0, remote_mode=0, pool_lag=0):
        self.lib = load()
        cfg = Config()
        cfg.abi_version = 2
        cfg.device, cfg.mode, cfg.nparam = device, MODE[mode], nparam
        cfg.nchain, cfg.chain0 = nchain, chain0
        cfg.nchain_total = nchain if nchain_total is None else nchain_total
        cfg.chains_per_rank, cfg.sync = chains_per_rank, sync
        cfg.pl, cfg.armin, cfg.armax, cfg.dfac, cfg.ifac = pl, armin, armax, dfac, ifac
        cfg.seed, cfg.coin_group, cfg.pool_m, cfg.thin = seed, coin_group, pool_m, thin
        cfg.trace, cfg.history_steps = int(trace), history_steps
        cfg.remote_mode, cfg.pool_lag = REMOTE_MODE[remote_mode], int(pool_lag)
        self.cfg = cfg
        self.d, self.C, self.mode = nparam, nchain, mode
        self.p2p = False
        self.h = C.c_void_p()
        _check(self.lib.mcgpu_create(C.byref(cfg), C.byref(self.h)))

    # -- lifetime -------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.mcgpu_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        _check(rc, self.h)

    # -- set-up ---------------------------------------------------------------
    def set_stream(self, cuda_stream):
        self._ck(self.lib.mcgpu_set_stream(self.h, C.c_void_p(cuda_stream)))

    def set_likelihood(self, lik, par=None, plugin=None):
        """lik names a built-in likelihood, or "plugin" with plugin=<cubin path> (a user functor compiled by
        mcpar_b200/plugin.py; par is handed to it unchanged)."""
        path = _plugin_path(lik, plugin)
        par_a = None if par is None else np.ascontiguousarray(par, dtype=np.float64).ravel()
        npar = 0 if par is None else par_a.size
        if path:
            self._ck(self.lib.mcgpu_set_likelihood_plugin(self.h, path, _p(par_a), npar))
        else:
            self._ck(self.lib.mcgpu_set_likelihood(self.h, LIK[lik], _p(par_a), npar))

    def set_covariance(self, incov=None):
        inc = None if incov is None else np.ascontiguousarray(incov, dtype=np.float64).ravel()
        if inc is not None:
            assert inc.size == self.d * self.d
        self._ck(self.lib.mcgpu_set_covariance(self.h, _p(inc)))

    def set_state(self, pinit):
        pinit = np.ascontiguousarray(pinit, dtype=np.float64)
        assert pinit.size == self.C * self.d, "pinit must hold nchain*nparam values"
        self._ck(self.lib.mcgpu_set_state(self.h, _p(pinit)))

    def set_state_sobol(self, plo, phi, first_point=0):
        """mcutil::qriguess straight into the engine: chain g starts at Sobol point first_point + g in [plo, phi]."""
        plo = np.ascontiguousarray(plo, dtype=np.float64); phi = np.ascontiguousarray(phi, dtype=np.float64)
        assert plo.size == self.d and phi.size == self.d
        self._ck(self.lib.mcgpu_set_state_sobol(self.h, _p(plo), _p(phi), C.c_uint64(first_point)))

    # -- host-callback likelihood (a VLFunc that lives on the host) ---------------
    def set_state_host(self, pinit, lylast):
        pinit = np.ascontiguousarray(pinit, dtype=np.float64); lylast = np.ascontiguousarray(lylast, dtype=np.float64)
        assert pinit.size == self.C * self.d and lylast.size == self.C
        self._ck(self.lib.mcgpu_set_state_host(self.h, _p(pinit), _p(lylast)))

    def step_propose(self, out=None):
        pt = out if out is not None else np.empty((self.C, self.d))
        self._ck(self.lib.mcgpu_step_propose(self.h, _p(pt)))
        return pt

    def step_accept(self, lytrial):
        ly = np.ascontiguousarray(lytrial, dtype=np.float64)
        assert ly.size == self.C
        self._ck(self.lib.mcgpu_step_accept(self.h, _p(ly)))

    def run_host(self, nsamp, nburn, pinit, loglik, incov=None):
        """MCPar::run with a HOST likelihood callable loglik(x [n][d]) -> [n] (the VLFunc plugin call, mcpar.cc:53,60,160)."""
        self.set_likelihood("host")
        self.set_covariance(incov)
        pinit = np.ascontiguousarray(pinit, dtype=np.float64).reshape(self.C, self.d)
        self.set_state_host(pinit, loglik(pinit))
        pt = np.empty((self.C, self.d))
        for _ in range(nburn):
            self.step_propose(pt); self.step_accept(loglik(pt))
        self.sample_begin(nsamp)
        for _ in range(nsamp):
            self.step_propose(pt); self.step_accept(loglik(pt))
        self.synchronize()

    def set_streams(self, local_rank, Z, U, I=None):
        Z = np.ascontiguousarray(Z, dtype=np.float64).ravel()
        U = np.ascontiguousarray(U, dtype=np.float64).ravel()
        I = np.zeros(0, dtype=np.int32) if I is None else np.ascontiguousarray(I, dtype=np.int32).ravel()
        self._ck(self.lib.mcgpu_set_streams(self.h, local_rank, _p(Z), C.c_size_t(Z.size), _p(U),
                                            C.c_size_t(U.size), _p(I), C.c_size_t(I.size)))

    # -- stepping -------------------------------------------------------------
    def burnin(self, nburn):
        self._ck(self.lib.mcgpu_burnin(self.h, nburn))

    def burnin_some(self, nmax):
        done, pend = C.c_int(0), C.c_int(0)
        self._ck(self.lib.mcgpu_burnin_some(self.h, nmax, C.byref(done), C.byref(pend)))
        return done.value, bool(pend.value)

    def tune(self):
        self._ck(self.lib.mcgpu_tune(self.h))

    def tuning_counters(self):
        p = C.c_void_p()
        self._ck(self.lib.mcgpu_tuning_counters(self.h, C.byref(p)))
        return DevicePtr(p.value, 16, "<i8")

    def sample_begin(self, nsamp):
        self._ck(self.lib.mcgpu_sample_begin(self.h, nsamp))

    def sample(self, nsteps):
        self._ck(self.lib.mcgpu_sample(self.h, nsteps))

    def exchange_begin(self):
        p = C.c_void_p(); tot = C.c_size_t(); off = C.c_size_t(); own = C.c_size_t()
        self._ck(self.lib.mcgpu_exchange_begin(self.h, C.byref(p), C.byref(tot), C.byref(off), C.byref(own)))
        return DevicePtr(p.value, tot.value), off.value, own.value

    def exchange_end(self):
        self._ck(self.lib.mcgpu_exchange_end(self.h))

    # -- peer-to-peer exchange (in-kernel stores over NVLink instead of an all-gather call) ----
    def p2p_export(self):
        """This engine's exchange-region handle (bytes) for mcgpu_p2p_attach in other processes."""
        buf = C.create_string_buffer(P2P_HANDLE_BYTES)
        self._ck(self.lib.mcgpu_p2p_export(self.h, buf, C.c_size_t(P2P_HANDLE_BYTES)))
        return buf.raw

    def p2p_attach(self, world, rank, handles):
        """handles: the world exported handles in rank order (own entry is ignored)."""
        blob = b"".join(handles)
        assert len(blob) == world * P2P_HANDLE_BYTES
        self._ck(self.lib.mcgpu_p2p_attach(self.h, world, rank, blob))
        self.p2p = True

    def synchronize(self):
        self._ck(self.lib.mcgpu_synchronize(self.h))

    def run(self, nsamp, nburn, pinit, lik, par=None, incov=None, plugin=None):
        """MCPar::run on this engine's chains (single engine: exchange is internal)."""
        self.set_likelihood(lik, par, plugin=plugin)
        self.set_covariance(incov)
        self.set_state(pinit)
        self.burnin(nburn)
        self.sample_begin(nsamp)
        self.sample(nsamp)
        self.synchronize()

    # -- read-back ------------------------------------------------------------
    def state(self):
        C_, d = self.C, self.d
        out = {k: np.empty((C_, d)) for k in ("p", "mu", "sig", "psum2")}
        out["ly"] = np.empty(C_)
        self._ck(self.lib.mcgpu_get_state(self.h, _p(out["p"]), _p(out["ly"]), _p(out["mu"]),
                                          _p(out["sig"]), _p(out["psum2"])))
        return out

    def factor(self, local_rank=0):
        f = np.empty((self.d, self.d))
        self._ck(self.lib.mcgpu_get_factor(self.h, local_rank, _p(f)))
        return f

    def musig(self, local_rank=0):
        n = self.cfg.nchain_total if self.mode == "verify" else (
            self.cfg.pool_m if 0 < self.cfg.pool_m < self.cfg.nchain_total else self.cfg.nchain_total)
        m = np.empty((n, self.d, 2))
        self._ck(self.lib.mcgpu_get_musig(self.h, local_rank, _p(m)))
        return m

    def trace(self, local_rank, nsteps):
        Cr, d = self.cfg.chains_per_rank, self.d
        t = {"accept": np.zeros((nsteps, Cr), dtype=np.uint8), "trial_ly": np.zeros((nsteps, Cr)),
             "trial_p": np.zeros((nsteps, Cr, d)), "cfac": np.zeros((nsteps, Cr)),
             "remote": np.zeros(nsteps, dtype=np.uint8), "iters": np.zeros(nsteps, dtype=np.int32),
             "cursors": np.zeros(3, dtype=np.int64)}
        self._ck(self.lib.mcgpu_get_trace(self.h, local_rank, _p(t["accept"]), _p(t["trial_ly"]),
                                          _p(t["trial_p"]), _p(t["cfac"]), _p(t["remote"]),
                                          _p(t["iters"]), _p(t["cursors"])))
        return t

    def history(self, first=0, count=None, out=None):
        st = self.stats()
        kept = st["history_rows"] // self.C
        if count is None:
            if first == 0 and self.cfg.history_steps and kept > self.cfg.history_steps:
                first = kept - self.cfg.history_steps          # the ring holds the last history_steps kept steps
            count = kept - first
        rows = out if out is not None else np.empty((count, self.C, self.d + 1))
        self._ck(self.lib.mcgpu_history_read(self.h, C.c_int64(first), C.c_int64(count), _p(rows)))
        return rows

    def attach_host_sink(self, rows):
        """rows: C-contiguous float64 (or float32: the reference's MCout element type; narrowed on the
        device) [capacity_steps][nchain][nparam+1] host array (kept alive by the caller); subsequent
        sample() calls drain into it asynchronously."""
        if rows is None:
            self._ck(self.lib.mcgpu_history_attach_host(self.h, None, C.c_size_t(0)))
            self._sink = None
            return
        assert rows.dtype in (np.float64, np.float32) and rows.flags.c_contiguous and rows.shape[1:] == (self.C, self.d + 1)
        self._sink = rows
        fn = self.lib.mcgpu_history_attach_host if rows.dtype == np.float64 else self.lib.mcgpu_history_attach_host_f32
        self._ck(fn(self.h, _p(rows), C.c_size_t(rows.shape[0])))

    def maxlike(self):
        out = np.empty(self.d + 1)
        self._ck(self.lib.mcgpu_history_maxlike(self.h, _p(out)))
        return out[:-1], out[-1]

    def moments(self):
        mean = np.empty(self.d); cov = np.empty((self.d, self.d))
        self._ck(self.lib.mcgpu_history_moments(self.h, _p(mean), _p(cov)))
        return mean, cov

    # -- checkpoint / restart -------------------------------------------------
    def checkpoint(self):
        """Opaque blob (numpy uint8) from which an engine of the same configuration continues bit for bit."""
        n = C.c_size_t()
        self._ck(self.lib.mcgpu_checkpoint_size(self.h, C.byref(n)))
        buf = np.empty(n.value, dtype=np.uint8)
        self._ck(self.lib.mcgpu_checkpoint_save(self.h, _p(buf), n))
        return buf

    def restore(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self._ck(self.lib.mcgpu_checkpoint_load(self.h, _p(blob), C.c_size_t(blob.size)))

    def stats(self):
        s = Stats()
        self._ck(self.lib.mcgpu_get_stats(self.h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def device_ptr(self, which):
        p = C.c_void_p(); n = C.c_size_t()
        self._ck(self.lib.mcgpu_device_ptr(self.h, which, C.byref(p), C.byref(n)))
        return DevicePtr(p.value, n.value)
