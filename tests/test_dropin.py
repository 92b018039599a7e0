"""The reference's C API (bpe/inc/bpe.h) on top of the engine: llmtokenizer_b200/dropin.
CPU: the library builds, exports every bpe.h function, and its host-side pieces (containers, decode,
pair-file format) behave like the reference's.  GPU: our caller with main.c's call sequence - and,
when it was built in the development container, the UNMODIFIED reference main.c compiled against the
drop-in tree - print exactly what the reference prints."""
import ctypes as C
import hashlib
import io
import os
import subprocess

import numpy as np
import pytest

import oracle_api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "llmtokenizer_b200", "dropin")
BPE_H_FUNCS = ["get_file", "dump_pairs", "read_pairs", "print_text", "print_graph", "compress", "decompress",
               "render_pairs", "resolve_pair", "is_less", "compress_n", "bpe_encode_file",
               "dyn_arr_create", "dyn_arr_free", "dyn_arr_set", "dyn_arr_get", "dyn_arr_append", "dyn_arr_max",
               "dyn_arr_min", "dyn_arr_sort", "hash_table_create", "hash_table_destroy", "hash_table_insert",
               "hash_table_delete", "hash_table_search", "hash_table_clear", "hash_table_merge"]
# MD5 of what the unmodified reference main.c prints for testing.txt (SURVEY.md §4)
REF_STDOUT_MD5_TESTING_TXT = "fb3902a9d35af8d2f36c817ae211e7b0"


class Pair(C.Structure):
    _fields_ = [("a", C.c_uint32), ("b", C.c_uint32)]


class DynArr(C.Structure):
    _fields_ = [("len", C.c_size_t), ("last_index", C.c_size_t), ("item_size", C.c_size_t), ("nodes", C.c_void_p)]


@pytest.fixture(scope="module")
def lib():
    from llmtokenizer_b200 import _lib
    _lib.load()  # libbpe.so depends on libbpe_cuda.so
    path = os.path.join(DROPIN, "libbpe.so")
    assert os.path.exists(path), "run `python -m llmtokenizer_b200.build`"
    L = C.CDLL(path)
    L.dyn_arr_create.restype = C.POINTER(DynArr)
    L.dyn_arr_create.argtypes = [C.c_size_t, C.c_size_t]
    L.dyn_arr_set.argtypes = [C.POINTER(DynArr), C.c_size_t, C.c_void_p]
    L.dyn_arr_get.argtypes = [C.POINTER(DynArr), C.c_size_t, C.c_void_p]
    L.dyn_arr_free.argtypes = [C.POINTER(DynArr)]
    L.read_pairs.restype = C.POINTER(DynArr)
    L.read_pairs.argtypes = [C.c_char_p]
    L.dump_pairs.argtypes = [C.c_char_p, C.POINTER(DynArr)]
    L.dump_pairs.restype = C.c_bool
    L.decompress.restype = C.c_void_p
    L.decompress.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(DynArr)]
    L.compress.restype = C.POINTER(DynArr)
    L.compress.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p]
    return L


def vocabulary(lib, merges):
    arr = lib.dyn_arr_create(512, 8)
    for i in range(256):
        p = Pair(i, 0)
        assert lib.dyn_arr_set(arr, i, C.byref(p))
    for k, (a, b) in enumerate(merges):
        p = Pair(int(a), int(b))
        assert lib.dyn_arr_set(arr, 256 + k, C.byref(p))
    return arr


def test_exports(lib):
    for name in BPE_H_FUNCS:
        assert hasattr(lib, name), name


def test_host_side_decode_and_pair_file(lib, tmp_path):
    g = oracle_api.golden("testing_txt")
    arr = vocabulary(lib, g["merges"])
    assert arr.contents.last_index == 255 + len(g["merges"])
    # resolve_pair (bpe.c:23-92) is host code: the last id expands to what the oracle says
    lib.resolve_pair.restype = C.c_void_p
    lib.resolve_pair.argtypes = [C.c_uint32, C.POINTER(DynArr), C.c_void_p]
    last = 255 + len(g["merges"])
    s = lib.resolve_pair(last, arr, None)
    assert s and C.string_at(s) == oracle_api.load().decode(np.array([last], np.uint32), g["merges"])
    C.CDLL(None).free(C.c_void_p(s))
    p = str(tmp_path / "pairs.bin").encode()
    assert lib.dump_pairs(p, arr)
    assert os.path.getsize(p) == 8 * len(g["merges"])        # LE {u32,u32} records from id 256, all of them
    back = lib.read_pairs(p)
    assert back.contents.last_index == arr.contents.last_index
    q = Pair()
    for k in (256, 256 + len(g["merges"]) - 1):
        assert lib.dyn_arr_get(back, k, C.byref(q)) and (q.a, q.b) == tuple(int(x) for x in g["merges"][k - 256])
    lib.dyn_arr_free(back)
    lib.dyn_arr_free(arr)


def test_hostile_vocabularies_are_rejected(lib, tmp_path):
    """A pairs file is input: an id that refers to itself or to a later id (300 = (65, 300)) must not send the
    expansion into a cycle or past its buffer (resolve_pair / render_pairs, bpe.c:23-128), and read_pairs refuses it."""
    lib.resolve_pair.restype = C.c_void_p
    lib.resolve_pair.argtypes = [C.c_uint32, C.POINTER(DynArr), C.c_void_p]
    arr = vocabulary(lib, [(97, 98), (65, 257), (258, 97), (256, 256)])   # 257 refers to itself, 258 to a later id
    assert not lib.resolve_pair(257, arr, None) and not lib.resolve_pair(258, arr, None)
    s = lib.resolve_pair(259, arr, None)                                   # 259 = (256, 256) is fine
    assert s and C.string_at(s) == b"abab"
    C.CDLL(None).free(C.c_void_p(s))
    lib.dyn_arr_free(arr)
    bad = tmp_path / "bad.bin"
    np.array([[97, 98], [65, 257]], dtype="<u4").tofile(bad)
    assert not lib.read_pairs(str(bad).encode())
    # left-deep chains far beyond the old 128-entry stack: id 256+k = (256+k-1, 'x')
    deep = [(97, 98)] + [(256 + k, 120) for k in range(2000)]
    arr = vocabulary(lib, deep)
    s = lib.resolve_pair(256 + 2000, arr, None)
    assert s and C.string_at(s) == b"ab" + b"x" * 2000
    C.CDLL(None).free(C.c_void_p(s))
    lib.dyn_arr_free(arr)


def test_print_text_matches_the_reference_format(lib, tmp_path):
    """bpe.c:182-196: 32..126 as the character, everything else as [id]; one block write per MB instead of one printf
    per token, same bytes."""
    ids = np.concatenate([np.arange(0, 300, dtype=np.uint32), np.random.default_rng(1).integers(0, 70000, 300_000).astype(np.uint32)])
    want = "".join(chr(int(t)) if 32 <= t <= 126 else f"[{int(t)}]" for t in ids) + "\n"
    src = tmp_path / "p.c"
    src.write_text('#include "bpe/inc/bpe.h"\n#include <stdio.h>\nint main(int c, char **v){FILE *f=fopen(v[1],"rb");fseek(f,0,SEEK_END);'
                   'long n=ftell(f)/4;rewind(f);uint32_t *t=malloc(n*4+4);if(fread(t,4,n,f)!=(size_t)n)return 1;print_text(t,(int)n);return 0;}\n')
    exe = tmp_path / "p"
    subprocess.check_call(["gcc", "-O1", "-o", str(exe), str(src), "-I", DROPIN, "-L", DROPIN, "-lbpe", f"-Wl,-rpath,{DROPIN}",
                           "-L", os.path.join(ROOT, "llmtokenizer_b200"), "-lbpe_cuda", f"-Wl,-rpath,{os.path.join(ROOT, 'llmtokenizer_b200')}"])
    data = tmp_path / "ids.bin"
    ids.astype("<u4").tofile(data)
    out = subprocess.run([str(exe), str(data)], capture_output=True, check=True).stdout
    assert out.decode("latin-1") == want


@pytest.mark.gpu
def test_decompress_inverts_compress(lib):
    # decompress() (bpe.c:341-394) runs the GPU decode: decompress(compress(x)) == x
    for name in ("testing_txt", "kat_k11"):
        g = oracle_api.golden(name)
        arr = vocabulary(lib, g["merges"])
        ids = np.ascontiguousarray(g["ids"], dtype=np.uint32)
        s = lib.decompress(ids.ctypes.data, len(ids), arr)
        assert s and C.string_at(s) == g["input"].tobytes().split(b"\0")[0]
        C.CDLL(None).free(C.c_void_p(s))
        lib.dyn_arr_free(arr)


def test_compress_argument_errors(lib, tmp_path):
    enc, n = C.c_void_p(), C.c_size_t()
    assert not lib.compress(None, C.byref(enc), C.byref(n))                      # bpe.c:548
    assert not lib.compress(b"/nonexistent/file", C.byref(enc), C.byref(n))      # bpe.c:133-137


def expected_stdout(ids):
    out = io.StringIO()
    import llmtokenizer_b200 as L
    L.print_text(ids, file=out)
    return out.getvalue().encode()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["testing_txt", "kat_k4", "kat_k11", "rt20k"])
def test_main_prints_what_the_reference_prints(name, tmp_path):
    g = oracle_api.golden(name)
    src = tmp_path / "in.txt"
    src.write_bytes(g["input"].tobytes())
    want = expected_stdout(g["ids"])
    exe = os.path.join(DROPIN, "example_main")
    r = subprocess.run([exe, str(src)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    assert r.stdout == want and b"round trip ok" in r.stderr
    if name == "testing_txt":
        assert hashlib.md5(r.stdout).hexdigest() == REF_STDOUT_MD5_TESTING_TXT
    ref_main = os.path.join(DROPIN, "_build", "ref_main")   # unmodified reference main.c against the drop-in headers
    if os.path.exists(ref_main):
        r2 = subprocess.run([ref_main, str(src)], capture_output=True)
        assert r2.returncode == 0 and r2.stdout == want
        if name == "testing_txt":
            assert hashlib.md5(r2.stdout).hexdigest() == REF_STDOUT_MD5_TESTING_TXT


@pytest.mark.gpu
def test_short_file_message(tmp_path):
    src = tmp_path / "a.txt"
    src.write_bytes(b"a")
    r = subprocess.run([os.path.join(DROPIN, "example_main"), str(src)], capture_output=True)
    assert r.returncode != 0 and r.stdout == b"Error: File contains less than 2 characters\n"   # bpe.c:558-563
