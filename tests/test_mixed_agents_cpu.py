"""CPU: the C ABI of mixed agent batches (colo_mixed_qlearning_*) -- the struct mirror, the prototypes and the argument
checks that fail before any CUDA call.  The per-instance rejections need a mixed-tables handle, which only a device
can make: tests/test_gpu_mixed_agents.py covers them."""
import ctypes as C
import re

from colosseum_b200 import _cabi
from colosseum_b200.build import build_library
from test_mixed_batch_cpu import _fields, _header


def test_qlearning_inst_mirror_and_prototypes_match_header():
    txt = _header()
    assert _fields(txt, "colo_qlearning_inst") == [f[0] for f in _cabi.QLearningInst._fields_]
    assert all(f[1] is C.c_double for f in _cabi.QLearningInst._fields_)
    assert _fields(txt, "colo_qlearning_args") == [f[0] for f in _cabi.QLearningArgs._fields_]
    assert "typedef struct colo_mixed_qlearning colo_mixed_qlearning;" in txt
    for name in ("colo_mixed_qlearning_create", "colo_mixed_qlearning_sizes", "colo_mixed_qlearning_steps",
                 "colo_mixed_qlearning_destroy"):
        assert re.search(r"\b" + name + r"\s*\(", txt), name
        assert name in _cabi.PROTOTYPES, name
    build_library()
    for name in _cabi.PROTOTYPES:
        assert hasattr(_cabi.lib(), name), name


def _no_launch(call):
    build_library()
    lib = _cabi.lib()
    before = lib.colo_launch_count()
    rc = call(lib)
    assert lib.colo_launch_count() == before
    return rc, _cabi.last_error()


def test_create_rejects_missing_handle_and_bad_flag():
    insts = (_cabi.QLearningInst * 1)()
    out = C.c_void_p()
    rc, err = _no_launch(lambda lib: lib.colo_mixed_qlearning_create(None, 1, insts, None, C.byref(out)))
    assert rc == -2 and out.value is None and "tables" in err
    fake = C.c_void_p(1 << 20)  # never dereferenced: the flag is checked first
    rc, err = _no_launch(lambda lib: lib.colo_mixed_qlearning_create(fake, 2, insts, None, C.byref(out)))
    assert rc == -2 and out.value is None and "episodic" in err


def test_steps_and_sizes_reject_a_missing_handle():
    args = _cabi.QLearningArgs()
    rc, err = _no_launch(lambda lib: lib.colo_mixed_qlearning_steps(None, C.byref(args), 1, 0, None))
    assert rc == -2 and "handle" in err
    q, v = C.c_longlong(), C.c_longlong()
    rc, err = _no_launch(lambda lib: lib.colo_mixed_qlearning_sizes(None, C.byref(q), C.byref(v)))
    assert rc == -2 and "handle" in err
