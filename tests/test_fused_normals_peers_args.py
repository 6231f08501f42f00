"""The multi-GPU fused-normal entry points without a GPU: prototypes and record width against the header, scratch sizes,
and argument checks that fail before anything is launched (the device pointers below are never dereferenced)."""

import ctypes as C
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
NEW = ["ddn_fuse_finish_partial_normals", "ddn_fuse_merge_normals_scratch_bytes", "ddn_fuse_merge_peers_normals",
       "ddn_fuse_finish_hashed_partial_normals", "ddn_fuse_merge_hashed_normals_scratch_bytes", "ddn_fuse_merge_hashed_peers_normals"]
FAKE = 1 << 20  # an aligned address no call below reaches a kernel with


def _header():
    return (ROOT / "include" / "ddn_b200.h").read_text()


def _n_params(name):
    m = re.search(r"DDN_API int " + name + r"\(([^;]*)\)\s*;", _header())
    assert m, name
    return len([p for p in m.group(1).split(",") if p.strip()])


def test_record_width_matches_header():
    from depthdensifier_b200 import _lib

    m = re.search(r"#define DDN_RECORD_NORMAL_WORDS (\d+)", _header())
    assert m and int(m.group(1)) == _lib.RECORD_NORMAL_WORDS == 10
    assert _lib.RECORD_NORMAL_WORDS % 2 == 0 and _lib.RECORD_WORDS % 2 == 0  # whole 16-byte pieces


@pytest.mark.parametrize("name", NEW)
def test_prototypes_match_header(name):
    from depthdensifier_b200 import _lib

    assert name in _lib.SYMBOLS
    assert len(_lib.SYMBOLS[name][1]) == _n_params(name)
    base = name.replace("_normals", "")
    # the normals forms take the base form's parameters plus one pointer (normal in, or out_normal), or the same ones
    extra = 0 if name.endswith("scratch_bytes") else 1
    assert len(_lib.SYMBOLS[name][1]) == len(_lib.SYMBOLS[base][1]) + extra


def _session():
    from depthdensifier_b200 import _lib

    return _lib.FuseSession(FAKE, FAKE, 1 << 16, None, FAKE, FAKE, FAKE)


def _hash(cap_voxels=1000):
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    sizes = [C.c_int64(0) for _ in range(5)]
    assert lib.ddn_hash_fuse_sizes(cap_voxels, *[C.byref(x) for x in sizes]) == 0
    return _lib.HashFuse(FAKE, FAKE, FAKE, FAKE, FAKE, sizes[0].value, cap_voxels)


def _fails(rc, lib, text):
    assert rc != 0
    assert text.encode() in lib.ddn_last_error_string(), lib.ddn_last_error_string()


def test_scratch_sizes(lib_built):
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    for cap_out in (4096, 1 << 20):
        for R in (1, 2, 16):
            plain, normals = C.c_int64(0), C.c_int64(0)
            assert lib.ddn_fuse_merge_scratch_bytes(1 << 16, R, cap_out, C.byref(plain)) == 0
            assert lib.ddn_fuse_merge_normals_scratch_bytes(1 << 16, R, cap_out, C.byref(normals)) == 0
            assert normals.value >= plain.value + 32 * cap_out
            assert lib.ddn_fuse_merge_hashed_scratch_bytes(R, cap_out, C.byref(plain)) == 0
            assert lib.ddn_fuse_merge_hashed_normals_scratch_bytes(R, cap_out, C.byref(normals)) == 0
            assert normals.value >= plain.value + 32 * cap_out
    assert lib.ddn_fuse_merge_normals_scratch_bytes(1 << 16, 0, 10, C.byref(plain)) != 0
    assert lib.ddn_fuse_merge_hashed_normals_scratch_bytes(17, 10, C.byref(plain)) != 0
    assert lib.ddn_fuse_merge_hashed_normals_scratch_bytes(2, 10, None) != 0


def test_finish_partial_normals_rejects(lib_built):
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    s = _session()
    f = lambda normal, records: lib.ddn_fuse_finish_partial_normals(C.byref(s), 10, 0, FAKE, FAKE, None, 1, normal, records, 16, None)
    _fails(f(None, FAKE), lib, "null pointer")
    _fails(f(FAKE, FAKE + 8), lib, "16-byte aligned")
    _fails(f(FAKE, None), lib, "16-byte aligned")
    empty = _lib.FuseSession()
    _fails(lib.ddn_fuse_finish_partial_normals(C.byref(empty), 10, 0, FAKE, FAKE, None, 1, FAKE, FAKE, 16, None), lib, "session")


def test_merge_peers_normals_rejects(lib_built):
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    s = _session()
    cap, R = 1024, 2
    need = C.c_int64(0)
    assert lib.ddn_fuse_merge_normals_scratch_bytes(s.cap_units, R, cap, C.byref(need)) == 0
    prefix = (C.c_void_p * R)(FAKE, FAKE)

    def f(records=(FAKE, FAKE), scratch_bytes=need.value, out_normal=FAKE, accum_bytes=cap * 64 + 16, scratch=FAKE):
        return lib.ddn_fuse_merge_peers_normals(C.byref(s), 0, R, (C.c_void_p * R)(*records), prefix, FAKE, scratch, scratch_bytes, None,
                                                0, FAKE, FAKE, FAKE, FAKE, out_normal, cap, FAKE, accum_bytes, None)

    _fails(f(out_normal=None), lib, "null pointer")
    _fails(f(accum_bytes=cap * 40 + 16), lib, "64 bytes")  # the plain form's accumulator is too small
    _fails(f(scratch_bytes=need.value - 1), lib, "ddn_fuse_merge_normals_scratch_bytes")
    plain = C.c_int64(0)
    assert lib.ddn_fuse_merge_scratch_bytes(s.cap_units, R, cap, C.byref(plain)) == 0
    _fails(f(scratch_bytes=plain.value), lib, "ddn_fuse_merge_normals_scratch_bytes")
    _fails(f(scratch=FAKE + 8), lib, "merge scratch")
    _fails(f(records=(FAKE, None)), lib, "null peer pointer")
    _fails(f(records=(FAKE, FAKE + 8)), lib, "16-byte aligned")


def test_hashed_partial_normals_rejects(lib_built):
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    s, hf = _session(), _hash()
    n = 100

    def f(normal=FAKE, records=FAKE, accum_bytes=n * 64 + 16, samples=FAKE):
        return lib.ddn_fuse_finish_hashed_partial_normals(C.byref(s), C.byref(hf), 0, n, 0, FAKE, FAKE, None, 1, normal, None, 0, records,
                                                          n, samples, FAKE, accum_bytes, None)

    _fails(f(normal=None), lib, "null pointer")
    _fails(f(records=FAKE + 8), lib, "16-byte aligned")
    _fails(f(samples=None), lib, "samples")
    _fails(f(accum_bytes=n * 40 + 16), lib, "n_points * 64 bytes")
    bad = _lib.HashFuse()
    _fails(lib.ddn_fuse_finish_hashed_partial_normals(C.byref(s), C.byref(bad), 0, n, 0, FAKE, FAKE, None, 1, FAKE, None, 0, FAKE, n, FAKE,
                                                      FAKE, n * 64 + 16, None), lib, "hash buffers")


def test_merge_hashed_peers_normals_rejects(lib_built):
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    s, hf = _session(), _hash()
    cap, R = 512, 2
    need = C.c_int64(0)
    assert lib.ddn_fuse_merge_hashed_normals_scratch_bytes(R, cap, C.byref(need)) == 0
    samples = (C.c_void_p * R)(FAKE, FAKE)

    def f(records=(FAKE, FAKE), scratch_bytes=need.value, out_normal=FAKE, cap_out=cap):
        return lib.ddn_fuse_merge_hashed_peers_normals(C.byref(s), C.byref(hf), 0, R, (C.c_void_p * R)(*records), samples, FAKE, FAKE,
                                                       scratch_bytes, FAKE, FAKE, FAKE, FAKE, out_normal, cap_out, None)

    _fails(f(out_normal=None), lib, "null pointer")
    _fails(f(scratch_bytes=need.value - 1), lib, "ddn_fuse_merge_hashed_normals_scratch_bytes")
    plain = C.c_int64(0)
    assert lib.ddn_fuse_merge_hashed_scratch_bytes(R, cap, C.byref(plain)) == 0
    _fails(f(scratch_bytes=plain.value), lib, "ddn_fuse_merge_hashed_normals_scratch_bytes")
    _fails(f(records=(None, FAKE)), lib, "null peer pointer")
    _fails(f(records=(FAKE + 8, FAKE)), lib, "16-byte aligned")
    _fails(f(cap_out=hf.cap_voxels + 1), lib, "cap_voxels")
