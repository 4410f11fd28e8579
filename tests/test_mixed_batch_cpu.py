"""CPU: the C ABI of mixed batches (colo_mixed_tables_*) -- struct mirrors and argument checks that fail before any
CUDA call, so they run without a GPU."""
import ctypes as C
import os
import re

from conftest import ROOT
from colosseum_b200 import _cabi
from colosseum_b200.build import build_library


def _header():
    txt = open(os.path.join(ROOT, "include", "colosseum_b200.h")).read()
    return re.sub(r"/\*.*?\*/", "", txt, flags=re.S)


def _fields(txt, cname):
    end = txt.index("} " + cname + ";")
    body = txt[txt.rindex("typedef struct {", 0, end) + len("typedef struct {"):end]
    out = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            out += [re.findall(r"[A-Za-z_][A-Za-z0-9_]*", part)[-1] for part in decl.split(",")]
    return out


def test_mixed_abi_structs_match_header():
    """the mixed calls take the existing colo_mdp_tables / colo_env_batch (mirrors in field order) and an opaque
    handle: no new struct has to be mirrored"""
    txt = _header()
    assert "typedef struct colo_mixed_tables colo_mixed_tables;" in txt
    assert "} colo_mixed_tables;" not in txt
    for cname, mirror in (("colo_mdp_tables", _cabi.MdpTables), ("colo_env_batch", _cabi.EnvBatch)):
        assert _fields(txt, cname) == [f[0] for f in mirror._fields_], cname
    for name in ("colo_mixed_tables_create", "colo_mixed_tables_destroy", "colo_mixed_visits_size",
                 "colo_mixed_env_reset", "colo_mixed_env_step", "colo_mixed_env_random_steps"):
        assert re.search(r"\b" + name + r"\s*\(", txt), name
        assert name in _cabi.PROTOTYPES, name


def _fake_tables(succ=True, S=5, A=2):
    """host struct with non-null (never dereferenced) pointers: the checks look at shapes and NULLs only"""
    t = _cabi.MdpTables()
    t.S, t.A, t.H = S, A, 0
    fake = 1 << 20
    t.rew_q, t.n_cls, t.nq = fake, 1, 2
    t.start_cum, t.start_idx, t.n_start = fake, fake, 1
    if succ:
        t.succ_cum, t.succ_idx, t.succ_len, t.Ksucc = fake, fake, fake, 3
    return t


def _create(tables, n_envs, mode=2):
    build_library()
    lib = _cabi.lib()
    n = len(tables)
    arr = (_cabi.MdpTables * max(n, 1))(*tables)
    sizes = (C.c_longlong * max(n, 1))(*n_envs)
    seeds = (C.c_ulonglong * max(n, 1))(*([0] * n))
    out = C.c_void_p()
    before = lib.colo_launch_count()
    rc = lib.colo_mixed_tables_create(arr, n, sizes, seeds, mode, None, C.byref(out))
    assert lib.colo_launch_count() == before
    return rc, _cabi.last_error(), out.value


def test_create_rejects_an_instance_without_successor_tables():
    rc, err, h = _create([_fake_tables(), _fake_tables(), _fake_tables(succ=False)], [4, 4, 4])
    assert rc == -2 and h is None  # COLO_ERR_ARG
    assert "instance 2" in err and "successor" in err


def test_create_rejects_an_instance_without_envs():
    rc, err, h = _create([_fake_tables(), _fake_tables()], [3, 0])
    assert rc == -2 and h is None
    assert "instance 1" in err and "n_envs" in err


def test_create_rejects_no_instances():
    rc, err, h = _create([], [])
    assert rc == -2 and h is None
    assert "n_inst" in err


def test_create_rejects_dense_mode_without_cdf():
    rc, err, h = _create([_fake_tables(), _fake_tables()], [2, 2], mode=0)
    assert rc == -2 and h is None
    assert "instance 0" in err and "cdf" in err
