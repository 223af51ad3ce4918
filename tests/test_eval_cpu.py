"""On-device evaluate_policy, CPU side: the closed-form targets / first slots against SB3's per-env targets, the per-env record
function of csrc/qs_eval.cuh (compiled with g++) against the NumPy restatement of SB3's loop, the C-ABI refusals and the ctypes
layout of qs_eval_args."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from eval_oracle import random_streams, sb3_episodes
from harness_util import ROOT, ptr


@pytest.fixture(scope="module")
def he(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("he") / "libqs_host_eval.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", os.path.join(ROOT, "tests", "host_harness", "harness_eval.cpp"),
                           "-o", out])
    lib = C.CDLL(out)
    i64 = C.c_int64
    for f in ("he_target", "he_base"):
        getattr(lib, f).argtypes = [i64] * 3
        getattr(lib, f).restype = i64
    lib.he_active.argtypes = [i64] * 4
    lib.he_active.restype = i64
    lib.he_record.argtypes = [i64] * 4 + [C.c_int32, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p] + [C.c_void_p] * 5
    lib.he_record.restype = i64
    return lib


@pytest.fixture(scope="module")
def ev():
    from rl_aerial_manipulator_b200 import evaluation
    return evaluation


def _sb3_targets(E, G):
    return np.array([(E + i) // G for i in range(G)], dtype=np.int64)


def test_closed_form_equals_sb3_targets_small(he, ev):
    for G in range(1, 71):
        ids = np.arange(G + 1)
        for E in range(1, 201):
            tgt = _sb3_targets(E, G)
            base = np.concatenate([[0], np.cumsum(tgt)])
            np.testing.assert_array_equal(ev.targets(E, G, ids[:G]), tgt)
            np.testing.assert_array_equal(ev.first_slot(E, G, ids), base)
            assert [he.he_target(E, G, int(i)) for i in range(G)] == tgt.tolist()
            assert [he.he_base(E, G, int(i)) for i in ids] == base.tolist()
            assert base[-1] == E
            for off, n in ((0, G), (G // 3, G - G // 3), (G - 1, 1)):
                assert he.he_active(E, G, off, n) == int((tgt[off:off + n] > 0).sum())


@pytest.mark.parametrize("E,G", [(10, 1 << 20), (1 << 20, 1 << 20), (7 * 4099 + 3, 4099), (10_000, 4096), (3, 65_537),
                                 (7 * 1_000_003 + 3, 1_000_003), (1, 1)])
def test_closed_form_equals_sb3_targets_large(he, ev, E, G):
    tgt = (E + np.arange(G, dtype=np.int64)) // G
    base = np.concatenate([[0], np.cumsum(tgt)])
    ids = np.arange(G + 1)
    np.testing.assert_array_equal(ev.targets(E, G, ids[:G]), tgt)
    np.testing.assert_array_equal(ev.first_slot(E, G, ids), base)
    probe = np.unique(np.concatenate([np.arange(min(G, 50)), np.arange(max(0, G - 50), G), np.random.default_rng(0).integers(0, G, 200)]))
    assert [he.he_target(E, G, int(i)) for i in probe] == tgt[probe].tolist()
    assert [he.he_base(E, G, int(i)) for i in probe] + [he.he_base(E, G, G)] == base[probe].tolist() + [E]
    assert he.he_active(E, G, 0, G) == int((tgt > 0).sum())


def _host_run(he, E, G, flags, ret, ln, shards):
    """Drive the host-compiled record function shard by shard over the whole stream; returns the merged slot arrays and the summed
    remaining after every step."""
    T = flags.shape[0]
    f64 = ret.dtype == np.float64
    slot = {k: np.zeros(E, dtype=dt) for k, dt in (("ret", np.float64), ("len", np.int32), ("flags", np.uint8), ("step", np.int32))}
    remaining = np.zeros(T, dtype=np.int64)
    for off, n in shards:
        first = he.he_base(E, G, off)
        m = he.he_base(E, G, off + n) - first
        out = {k: np.zeros(max(m, 1), dtype=v.dtype) for k, v in slot.items()}
        count = np.zeros(n, dtype=np.int32)
        rem = he.he_active(E, G, off, n)
        for t in range(T):
            f = np.ascontiguousarray(flags[t, off:off + n])
            r = np.ascontiguousarray(ret[t, off:off + n])
            l_ = np.ascontiguousarray(ln[t, off:off + n])
            rem -= he.he_record(E, G, off, n, t, ptr(f), ptr(r), int(f64), ptr(l_), ptr(count), ptr(out["ret"]), ptr(out["len"]),
                                ptr(out["flags"]), ptr(out["step"]))
            remaining[t] += rem
        for k in slot:
            slot[k][first:first + m] = out[k][:m]
    return slot, remaining


@pytest.mark.parametrize("f64", [True, False])
def test_record_function_equals_sb3_loop(he, f64):
    rng = np.random.default_rng(1 if f64 else 2)
    for G, E, T, p in ((1, 1, 30, 0.2), (1, 7, 100, 0.1), (31, 31, 60, 0.05), (33, 3 * 33 + 5, 200, 0.05), (70, 200, 120, 0.1),
                       (64, 10, 80, 0.03), (97, 1000, 400, 0.2)):
        flags, ret, ln = random_streams(rng, T, G, p, f64)
        want = sb3_episodes(E, flags, ret, ln)
        for shards in ([(0, G)], [(0, G // 2), (G // 2, G - G // 2)] if G > 1 else [(0, G)]):
            slot, remaining = _host_run(he, E, G, flags, ret, ln, shards)
            np.testing.assert_array_equal(remaining, want["remaining"])
            if want["remaining"][-1] != 0:
                continue                      # stream too short to finish: the filled slots are compared below anyway
            for k in ("ret", "len", "flags", "step"):
                np.testing.assert_array_equal(slot[k], want["slot_" + k], err_msg=f"{k} G={G} E={E} shards={shards}")
            # SB3's episode lists = the slots sorted by (completion step, env id)
            env_id = np.repeat(np.arange(G), want["targets"])
            order = np.lexsort((env_id, slot["step"]))
            np.testing.assert_array_equal(slot["ret"][order], want["ret"])
            np.testing.assert_array_equal(slot["len"][order], want["len"])
            np.testing.assert_array_equal(env_id[order], want["env_id"])


def test_ctypes_layout_matches_header(tmp_path):
    from rl_aerial_manipulator_b200 import _cabi
    fields = [f for f, _ in _cabi.QsEvalArgs._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "quadsim.h"\nint main(void) {\n'
                   '  printf("%zu %d", sizeof(qs_eval_args), QS_EVAL_STATE_WORDS);\n'
                   + "".join(f'  printf(" %zu", offsetof(qs_eval_args, {f}));\n' for f in fields) + '  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    A = _cabi.QsEvalArgs
    assert got == [C.sizeof(A), _cabi.EVAL_STATE_WORDS] + [getattr(A, f).offset for f in fields]


def test_eval_entry_points_refuse_bad_arguments():
    """Argument checks return QS_EINVAL before any device memory is touched, so aligned dummy pointers suffice."""
    from rl_aerial_manipulator_b200 import _cabi
    lib = _cabi.load_library()
    dummy = 1 << 20

    def args(**kw):
        a = _cabi.QsEvalArgs()
        a.n, a.env_id_offset, a.n_global, a.n_eval_episodes = 64, 0, 64, 10
        for f in ("flags", "ep_return", "ep_len", "count", "state", "ret_out", "len_out", "flags_out", "step_out"):
            setattr(a, f, dummy)
        for k, v in kw.items():
            setattr(a, k, v)
        return a
    cases = [(dict(n=0), b"n must be >= 1"), (dict(n_eval_episodes=0), b"n_eval_episodes must be >= 1"),
             (dict(env_id_offset=1), b"env_id_offset + n <= n_global"), (dict(env_id_offset=-1), b"0 <= env_id_offset"),
             (dict(n_global=0), b"n_global"), (dict(count=None), b"count and state"), (dict(state=None), b"count and state"),
             (dict(n_eval_episodes=1 << 40, n_global=64), b"fit in int32")]
    for fn in (lib.qs_eval_begin, lib.qs_eval_record):
        assert fn(None, None) == -1 and b"args is NULL" in lib.qs_eval_last_error()
        for kw, msg in cases:
            assert fn(C.byref(args(**kw)), None) == -1, kw
            assert msg in lib.qs_eval_last_error(), (kw, lib.qs_eval_last_error())
    for f in ("flags", "ep_return", "ep_len", "ret_out", "len_out", "flags_out", "step_out"):
        assert lib.qs_eval_record(C.byref(args(**{f: None})), None) == -1, f
        assert b"must not be NULL" in lib.qs_eval_last_error()
    assert lib.qs_eval_record(C.byref(args(return_is_f64=2)), None) == -1
    assert b"return_is_f64" in lib.qs_eval_last_error()
