"""ctypes binding of the CPU oracle (libjtb_oracle.so).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

from jepsen_tigerbeetle_b200 import abi
from jepsen_tigerbeetle_b200.history import CModel, FlatHistory, as_c_history

ALGO_BRUTE, ALGO_LINEAR, ALGO_WGL, ALGO_WGL_COMPACT, ALGO_LEVEL, ALGO_LAZY_BANK = 0, 1, 2, 3, 4, 5
_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_TMP_SO = None


def _cpu_stamp() -> str:
    """Identity of the host CPU: the oracle is compiled -march=native, so a library built on another machine
    (it travels to the GPU box with the snapshot) must be rebuilt there."""
    try:
        model, flags = "", ""
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and not model:
                model = line.split(":", 1)[1].strip()
            elif line.startswith("flags") and not flags:
                flags = line.split(":", 1)[1].strip()
            if model and flags:
                break
        import hashlib
        return model + " " + hashlib.sha1(flags.encode()).hexdigest()[:12]
    except OSError:
        return "unknown"


def build(force: bool = False) -> str:
    global _TMP_SO
    so = os.path.join(_HERE, "libjtb_oracle.so")
    stamp_file = os.path.join(_HERE, ".build_cpu")
    srcs = [os.path.join(_HERE, f) for f in ("lin_oracle.cpp", "scan_oracle.cpp", "oracle_common.h", "Makefile")]
    srcs.append(os.path.join(_HERE, "..", "include", "jtb_check.h"))
    stale = not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs)
    stamp = _cpu_stamp()
    try:
        other_cpu = open(stamp_file).read() != stamp
    except OSError:
        other_cpu = True
    if not (force or stale or other_cpu):
        return so
    if not os.access(_HERE, os.W_OK):
        # a read-only tree: compile once per process into a private temporary directory, leaving the tree as it is
        if force or _TMP_SO is None:
            _TMP_SO = os.path.join(tempfile.mkdtemp(prefix="jtb_oracle_"), "libjtb_oracle.so")
            subprocess.check_call(["make", "-C", _HERE, "-B", "-s", "OUT=" + _TMP_SO], stdout=subprocess.DEVNULL)
        return _TMP_SO
    subprocess.check_call(["make", "-C", _HERE, "-B", "-s"], stdout=subprocess.DEVNULL)
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return so


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.jtbo_last_error.restype = C.c_char_p
        _LIB.jtbo_scan_last_error.restype = C.c_char_p
    return _LIB


def check_linearizable(h: FlatHistory, model: CModel, algo: int = ALGO_WGL_COMPACT,
                       max_configs: int = 0, canon_info: bool = True, n_threads: int = 1,
                       eager_reads: bool = False) -> dict:
    ch = as_c_history(h)
    shards = (abi.CLinShard * h.n_shards)()
    res = abi.CLinResult()
    rc = lib().jtbo_check_linearizable(C.byref(ch), C.byref(model), algo, C.c_uint64(max_configs),
                                       int(bool(canon_info)) | (2 if eager_reads else 0), n_threads, shards, C.byref(res))
    if rc != 0:
        raise RuntimeError(lib().jtbo_last_error().decode())
    return {
        "valid": res.valid, "n_failures": res.n_failures, "configs": res.configs_explored,
        "probes": res.probes, "seconds": res.seconds_total,
        "shards": [{"valid": s.valid, "witness_index": s.witness_index,
                    "previous_ok_index": s.previous_ok_index, "cause": s.cause,
                    "configs": s.configs_explored, "probes": s.probes} for s in shards],
    }


def final_configs(h: FlatHistory, model: CModel, shard: int = 0, cap: int = 10, eager_reads: bool = False) -> dict:
    """Twin of `jtb_final_configs`: knossos' :configs of an INVALID shard; total = -1 when it is not INVALID."""
    ch = as_c_history(h)
    buf = (abi.CFinalConfig * max(cap, 1))()
    total = C.c_int64(0)
    rc = lib().jtbo_final_configs(C.byref(ch), C.byref(model), 1 | (2 if eager_reads else 0), shard, buf, cap,
                                  C.byref(total))
    if rc != 0:
        raise RuntimeError(lib().jtbo_last_error().decode())
    return {"total": total.value, "configs": abi.final_configs_to_list(buf, max(0, min(cap, total.value)))}


def check_set_full(h: FlatHistory, linearizable: bool = True) -> dict:
    ch = as_c_history(h)
    shards = (abi.CSetFullShard * h.n_shards)()
    out, bufs = abi.alloc_setfull_out(h, shards)
    rc = lib().jtbo_check_set_full(C.byref(ch), int(linearizable), C.byref(out))
    if rc != 0:
        raise RuntimeError(lib().jtbo_scan_last_error().decode())
    return abi.setfull_to_dict(out, shards, bufs)


def check_bank_totals(h: FlatHistory, model: CModel, total_amount: int = 0) -> dict:
    ch = as_c_history(h)
    res = abi.CBankResult()
    rc = lib().jtbo_check_bank_totals(C.byref(ch), C.byref(model), C.c_int64(total_amount),
                                      C.byref(res))
    if rc != 0:
        raise RuntimeError(lib().jtbo_scan_last_error().decode())
    return bank_to_dict(res)


def bank_to_dict(res) -> dict:
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
