"""ctypes binding of the product library `libjtb_check.so` (C ABI in include/jtb_check.h).

This is the same boundary a JVM host binds through JNI (see INTEGRATION.md).  There is NO fallback:
if the CUDA library is missing or no device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

from . import abi
from .history import CModel, FlatHistory, as_c_history

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("JTB_LIB_PATH") or os.path.join(_HERE, "libjtb_check.so")  # env: A/B experiments only
CSRC = os.path.join(_HERE, "csrc")
_SOURCES = ["jtb_abi.cu", "jtb_prep.cpp", "jtb_multi.cpp"]
_DEPS = _SOURCES + ["jtb_prep.h", "jtb_expand.h", "jtb_wgl.cuh", "jtb_search.cuh", "jtb_scout.cuh", "jtb_scans.cuh",
                    "jtb_table_bench.cuh", "jtb_level.cuh", "jtb_partition.cuh"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-ldl"]

EXPORTS = ["jtb_abi_version", "jtb_device_count", "jtb_create", "jtb_destroy", "jtb_last_error",
           "jtb_check_linearizable", "jtb_check_set_full", "jtb_check_bank_totals",
           "jtb_table_bench", "jtb_get_stats", "jtb_struct_size", "jtb_prepare_seconds", "jtb_prepare_info",
           "jtb_final_configs", "jtb_gather_bench", "jtb_host_alloc", "jtb_host_free", "jtb_partition_by_key", "jtb_ledger_balances", "jtb_multi_create", "jtb_multi_create_error", "jtb_multi_destroy", "jtb_multi_n_gpus",
           "jtb_multi_last_error", "jtb_multi_check_linearizable", "jtb_multi_check_set_full"]

_lib = None
_lock = threading.Lock()


class NativeError(RuntimeError):
    pass


def build(force: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    deps = [os.path.join(CSRC, f) for f in _DEPS]
    deps.append(os.path.join(_HERE, "..", "include", "jtb_check.h"))
    stale = (not os.path.exists(LIB_PATH)
             or any(os.path.getmtime(d) > os.path.getmtime(LIB_PATH) for d in deps))
    if force or stale:
        cmd = [_nvcc(), *NVCC_FLAGS, "-o", LIB_PATH] + [os.path.join(CSRC, f) for f in _SOURCES]
        subprocess.check_call(cmd)
    return LIB_PATH


def _nvcc() -> str:
    """nvcc of the CUDA toolkit PyTorch finds ($CUDA_HOME, $CUDA_PATH, nvcc on $PATH, the default install), so the
    build works for users whose PATH lacks the toolkit's bin directory."""
    from torch.utils.cpp_extension import CUDA_HOME
    if CUDA_HOME is None:
        raise NativeError("no CUDA toolkit found: set CUDA_HOME or put nvcc on PATH")
    return os.path.join(CUDA_HOME, "bin", "nvcc")


def lib() -> C.CDLL:
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; "
                                  "g.build()'` (there is no CPU fallback)")
            L = C.CDLL(LIB_PATH)
            L.jtb_abi_version.restype = C.c_int
            L.jtb_struct_size.restype = C.c_long
            L.jtb_prepare_seconds.restype = C.c_double
            L.jtb_prepare_seconds.argtypes = [C.c_void_p, C.c_void_p]
            L.jtb_prepare_info.restype = C.c_double
            L.jtb_prepare_info.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
            L.jtb_device_count.restype = C.c_int
            L.jtb_create.restype = C.c_void_p
            L.jtb_create.argtypes = [C.c_void_p]
            L.jtb_destroy.argtypes = [C.c_void_p]
            L.jtb_last_error.restype = C.c_char_p
            L.jtb_last_error.argtypes = [C.c_void_p]
            L.jtb_check_linearizable.argtypes = [C.c_void_p] * 5
            L.jtb_final_configs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
            L.jtb_check_set_full.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
            L.jtb_check_bank_totals.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
            L.jtb_table_bench.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
            L.jtb_gather_bench.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_int,
                                           C.c_void_p, C.c_void_p]
            L.jtb_multi_create.restype = C.c_void_p
            L.jtb_multi_create.argtypes = [C.c_void_p, C.c_int]
            L.jtb_multi_create_error.restype = C.c_char_p
            L.jtb_multi_destroy.argtypes = [C.c_void_p]
            L.jtb_multi_n_gpus.argtypes = [C.c_void_p]
            L.jtb_multi_last_error.restype = C.c_char_p
            L.jtb_multi_last_error.argtypes = [C.c_void_p]
            L.jtb_multi_check_linearizable.argtypes = [C.c_void_p] * 6
            L.jtb_multi_check_set_full.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
            if L.jtb_abi_version() != abi.ABI_VERSION:
                raise NativeError("ABI version mismatch between libjtb_check.so and abi.py")
            _lib = L
    return _lib


class Context:
    """One checker context = one CUDA device + stream + cached device buffers (`jtb_ctx`)."""

    def __init__(self, device: int = 0, table_bytes: int = 0, max_configs: int = 0,
                 time_budget_ms: int = 0, search_ctas: int = 0, eager_reads: bool = True,
                 scouts: bool = True, engine: str = "auto", beam: bool = True) -> None:
        """engine: "auto" (chosen from the history, DESIGN.md section 4), "level", "worklist"; beam=False skips the beam
        sweep that histories with crashed ops get first."""
        L = lib()
        flags = (0 if eager_reads else abi.OPT_NO_EAGER_READS) | (0 if scouts else abi.OPT_NO_SCOUTS)
        flags |= {"auto": 0, "level": abi.OPT_ENGINE_LEVEL, "worklist": abi.OPT_ENGINE_WORKLIST}[engine]
        flags |= 0 if beam else abi.OPT_NO_BEAM
        opts = abi.COpts(device, flags, table_bytes, max_configs, time_budget_ms, search_ctas)
        self._h = L.jtb_create(C.byref(opts))
        if not self._h:
            raise NativeError("jtb_create failed: no CUDA device available (no CPU fallback)")

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().jtb_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _err(self) -> str:
        return lib().jtb_last_error(self._h).decode()

    # ---- hot path A9 ----------------------------------------------------------------------------
    def check_linearizable(self, h: FlatHistory, model: CModel) -> dict:
        ch = as_c_history(h)
        shards = (abi.CLinShard * h.n_shards)()
        res = abi.CLinResult()
        rc = lib().jtb_check_linearizable(self._h, C.addressof(ch), C.addressof(model),
                                          C.addressof(shards), C.addressof(res))
        if rc != 0:
            raise NativeError(f"jtb_check_linearizable rc={rc}: {self._err()}")
        return {
            "valid": res.valid, "n_failures": res.n_failures, "configs": res.configs_explored,
            "probes": res.probes, "hbm_bytes_algorithmic": res.hbm_bytes_algorithmic,
            "key_bytes": res.key_bytes, "seconds_kernel": res.seconds_kernel,
            "seconds_total": res.seconds_total,
            "shards": [{"valid": s.valid, "witness_index": s.witness_index,
                        "previous_ok_index": s.previous_ok_index, "cause": s.cause,
                        "configs": s.configs_explored, "probes": s.probes} for s in shards],
        }

    # ---- hot path A4 ----------------------------------------------------------------------------
    def check_set_full(self, h: FlatHistory, linearizable: bool = True) -> dict:
        ch = as_c_history(h)
        shards = (abi.CSetFullShard * h.n_shards)()
        out, bufs = abi.alloc_setfull_out(h, shards)
        rc = lib().jtb_check_set_full(self._h, C.addressof(ch), int(linearizable), C.addressof(out))
        if rc != 0:
            raise NativeError(f"jtb_check_set_full rc={rc}: {self._err()}")
        return abi.setfull_to_dict(out, shards, bufs)

    # ---- hot path A8 ----------------------------------------------------------------------------
    def check_bank_totals(self, h: FlatHistory, model: CModel, total_amount: int = 0) -> dict:
        ch = as_c_history(h)
        res = abi.CBankResult()
        rc = lib().jtb_check_bank_totals(self._h, C.addressof(ch), C.addressof(model),
                                         C.c_int64(total_amount), C.addressof(res))
        if rc != 0:
            raise NativeError(f"jtb_check_bank_totals rc={rc}: {self._err()}")
        return {
            "valid": res.valid, "reference_throws": res.reference_throws, "read_count": res.read_count,
            "error_count": res.error_count,
            "first_error_index": res.first_error_index, "first_error_type": res.first_error_type,
            "count_by_type": list(res.count_by_type),
            "first_index_by_type": list(res.first_index_by_type),
            "last_index_by_type": list(res.last_index_by_type),
            "worst_index_by_type": list(res.worst_index_by_type),
            "lowest_total": res.lowest_total, "highest_total": res.highest_total,
            "lowest_index": res.lowest_index, "highest_index": res.highest_index,
            "seconds": res.seconds_total, "seconds_kernel": res.seconds_kernel,
        }

    def final_configs(self, h: FlatHistory, model: CModel, shard: int = 0, cap: int = 10) -> dict:
        """knossos' :configs of an INVALID shard (`jtb_final_configs`): call directly after `check_linearizable`
        on the same history.  Returns {"total": all such configurations, "configs": the first `cap` of them}."""
        ch = as_c_history(h)
        buf = (abi.CFinalConfig * max(cap, 1))()
        total = C.c_int64(0)
        rc = lib().jtb_final_configs(self._h, C.addressof(ch), C.addressof(model), shard, C.addressof(buf), cap,
                                     C.addressof(total))
        if rc != 0:
            raise NativeError(f"jtb_final_configs rc={rc}: {self._err()}")
        return {"total": total.value, "configs": abi.final_configs_to_list(buf, min(cap, total.value))}

    def stats(self) -> dict:
        out = (C.c_ulonglong * 24)()
        lib().jtb_get_stats(C.c_void_p(self._h), out, 24)
        names = ["configs", "probes", "expansions", "ring_tail", "ring_head", "idle_polls",
                 "max_probe_len", "table_slots", "grid", "ring_entries", "attempts", "kernel_us",
                 "h2d_bytes", "d2h_bytes", "kernel_launches", "scout_steps", "scout_configs",
                 "scout_decided", "scouts", "engine_level", "beam_levels", "beam_configs", "beam_decided", "beam_attempts"]
        return {n: int(out[i]) for i, n in enumerate(names)}

    # ---- SURVEY 8(f) N2: independent/subhistory and ledger->bank on the device ------------------------------
    def partition_by_key(self, event_key) -> dict:
        """Stable partition of the events by key: {"order", "shard_off", "key_ids"} (numpy arrays)."""
        import numpy as np
        k = np.ascontiguousarray(event_key, dtype=np.int64)
        n = int(k.shape[0])
        cap = max(1, n)
        order = np.empty(n, dtype=np.int32)
        off = np.empty(cap + 1, dtype=np.int64)
        ids = np.empty(cap, dtype=np.int64)
        nk = C.c_int32(0)
        rc = lib().jtb_partition_by_key(self._h, C.c_int64(n), k.ctypes.data_as(C.c_void_p), order.ctypes.data_as(C.c_void_p),
                                        off.ctypes.data_as(C.c_void_p), ids.ctypes.data_as(C.c_void_p), C.c_int32(cap), C.byref(nk))
        if rc != 0:
            raise NativeError(f"jtb_partition_by_key rc={rc}: {self._err()}")
        return {"order": order, "shard_off": off[:nk.value + 1].copy(), "key_ids": ids[:nk.value].copy()}

    def ledger_balances(self, credits_posted, debits_posted):
        import numpy as np
        c = np.ascontiguousarray(credits_posted, dtype=np.int64)
        d = np.ascontiguousarray(debits_posted, dtype=np.int64)
        out = np.empty(c.shape[0], dtype=np.int32)
        rc = lib().jtb_ledger_balances(self._h, C.c_int64(c.shape[0]), c.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p),
                                       out.ctypes.data_as(C.c_void_p))
        if rc != 0:
            raise NativeError(f"jtb_ledger_balances rc={rc}: {self._err()}")
        return out

    # ---- K2 microbenchmark ----------------------------------------------------------------------
    def table_bench(self, n_keys: int, variant: int = 0, rounds: int = 3) -> dict:
        ins, prb, found = C.c_double(), C.c_double(), C.c_uint64()
        rc = lib().jtb_table_bench(self._h, n_keys, variant, rounds, C.addressof(ins),
                                   C.addressof(prb), C.addressof(found))
        if rc != 0:
            raise NativeError(f"jtb_table_bench rc={rc}: {self._err()}")
        return {"insert_seconds": ins.value, "probe_seconds": prb.value, "found": found.value,
                "n_keys": n_keys, "rounds": rounds, "variant": variant}


class MultiContext:
    """`jtb_multi`: the in-library multi-GPU fan-out (one process, n_gpus devices, one NCCL all-reduce(MAX) of the
    per-shard verdict vector) — what a single-process JVM host binds instead of `independent/checker`'s thread pool."""

    def __init__(self, n_gpus: int = 0, table_bytes: int = 0, max_configs: int = 0, time_budget_ms: int = 0,
                 eager_reads: bool = True, scouts: bool = True) -> None:
        L = lib()
        flags = (0 if eager_reads else abi.OPT_NO_EAGER_READS) | (0 if scouts else abi.OPT_NO_SCOUTS)
        opts = abi.COpts(0, flags, table_bytes, max_configs, time_budget_ms, 0)
        self._h = L.jtb_multi_create(C.byref(opts), n_gpus)
        if not self._h:
            raise NativeError(f"jtb_multi_create failed: {L.jtb_multi_create_error().decode()}")
        self.n_gpus = L.jtb_multi_n_gpus(self._h)

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().jtb_multi_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def check_linearizable(self, h: FlatHistory, model: CModel) -> dict:
        ch = as_c_history(h)
        shards = (abi.CLinShard * h.n_shards)()
        res = abi.CLinResult()
        dev = (C.c_int32 * max(1, h.n_shards))()
        rc = lib().jtb_multi_check_linearizable(self._h, C.addressof(ch), C.addressof(model), C.addressof(shards),
                                                C.addressof(res), C.addressof(dev))
        if rc != 0:
            raise NativeError(f"jtb_multi_check_linearizable rc={rc}: {lib().jtb_multi_last_error(self._h).decode()}")
        return {
            "valid": res.valid, "n_failures": res.n_failures, "configs": res.configs_explored, "probes": res.probes,
            "hbm_bytes_algorithmic": res.hbm_bytes_algorithmic, "key_bytes": res.key_bytes,
            "seconds_kernel": res.seconds_kernel, "seconds_total": res.seconds_total,
            "device_of_shard": [dev[s] for s in range(h.n_shards)],
            "shards": [{"valid": s.valid, "witness_index": s.witness_index, "previous_ok_index": s.previous_ok_index,
                        "cause": s.cause, "configs": s.configs_explored, "probes": s.probes} for s in shards],
        }

    def check_set_full(self, h: FlatHistory, linearizable: bool = True) -> dict:
        ch = as_c_history(h)
        shards = (abi.CSetFullShard * h.n_shards)()
        out = abi.CSetFullOut()
        out.shards = C.cast(shards, C.c_void_p)
        dev = (C.c_int32 * max(1, h.n_shards))()
        rc = lib().jtb_multi_check_set_full(self._h, C.addressof(ch), int(linearizable), C.addressof(out),
                                            C.addressof(dev))
        if rc != 0:
            raise NativeError(f"jtb_multi_check_set_full rc={rc}: {lib().jtb_multi_last_error(self._h).decode()}")
        fields = [f for f, _ in abi.CSetFullShard._fields_]
        return {"valid": out.valid, "n_failures": out.n_failures, "raia_valid": out.raia_valid,
                "n_suspect": out.n_suspect, "seconds_kernel": out.seconds_kernel, "seconds_total": out.seconds_total,
                "device_of_shard": [dev[s] for s in range(h.n_shards)],
                "shards": [{f: getattr(s, f) for f in fields} for s in shards]}


def gather_bench(ctx: "Context", table_bytes: int, in_flight: int = 4, wide: int = 1, iters: int = 64,
                 ctas_per_sm: int = 8, rounds: int = 3) -> dict:
    """Random 16 B gathers over a table of `table_bytes` (see `jtb_gather_bench`)."""
    sec, n = C.c_double(), C.c_uint64()
    rc = lib().jtb_gather_bench(ctx._h, table_bytes, in_flight, wide, iters, ctas_per_sm, rounds, C.addressof(sec),
                                C.addressof(n))
    if rc != 0:
        raise NativeError(f"jtb_gather_bench rc={rc}: {ctx._err()}")
    return {"table_bytes": table_bytes, "in_flight": in_flight, "wide": wide, "ctas_per_sm": ctas_per_sm,
            "probes": n.value, "seconds": sec.value, "Gprobes_s": n.value / sec.value / 1e9,
            "algo_GBps": 16 * wide * n.value / sec.value / 1e9}


def prepare_seconds(h: FlatHistory, model: CModel) -> float:
    """Host preparation time only (no GPU needed)."""
    ch = as_c_history(h)
    return lib().jtb_prepare_seconds(C.addressof(ch), C.addressof(model))


def prepare_info(h: FlatHistory, model: CModel) -> dict:
    """Host preparation only (no GPU needed): the layout the device search would use."""
    ch = as_c_history(h)
    info = (C.c_longlong * 4)()
    sec = lib().jtb_prepare_info(C.addressof(ch), C.addressof(model), C.addressof(info))
    return {"seconds": sec, "key_bytes": info[0], "slot_lanes": info[1], "max_classes": info[2], "ranks": info[3]}


def device_count() -> int:
    return lib().jtb_device_count()


def pinned_copy(a):
    """A copy of numpy array `a` in page-locked host memory (jtb_host_alloc): H2D copies of it run at the PCIe rate.
    The block is released when the returned array (and every view of it) is gone."""
    import weakref

    import numpy as np
    L = lib()
    L.jtb_host_alloc.restype = C.c_void_p
    L.jtb_host_alloc.argtypes = [C.c_size_t]
    L.jtb_host_free.argtypes = [C.c_void_p]
    ptr = L.jtb_host_alloc(max(a.nbytes, 16))
    if not ptr:
        raise NativeError("jtb_host_alloc failed")
    raw = (C.c_char * max(a.nbytes, 1)).from_address(ptr)
    base = np.frombuffer(raw, dtype=a.dtype, count=a.size)      # every view of the result keeps `base` alive
    weakref.finalize(base, L.jtb_host_free, C.c_void_p(ptr))
    out = base.reshape(a.shape)
    out[...] = a
    return out


def pin_history(h: FlatHistory) -> FlatHistory:
    """The history with its payload (the read id lists: the bulk of a set-full history) in page-locked memory."""
    import dataclasses
    return dataclasses.replace(h, payload=pinned_copy(h.payload))
