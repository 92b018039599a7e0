"""Host-side mirror of the reference's BPE interface (bpe/inc/bpe.h) on top of the CUDA engine.

Names and argument meaning follow the reference: compress() trains + encodes a file
(bpe.c:541-811), decompress() expands ids (bpe.c:341-394), dump_pairs()/read_pairs() use the
reference's merge-table file format (bpe.c:243-339), print_text() renders ids the way main.c
prints them (bpe.c:182-196).  The additive pieces (merge cap, stand-alone encode, GPU count,
resident contexts) are keyword arguments / extra functions.

All heavy lifting happens in libbpe_cuda.so; nothing here computes merges on the CPU.
"""
import ctypes as C
import os
import sys

import numpy as np

from . import _lib
from ._lib import Pair, Stats

ERRORS = {-1: "invalid argument", -2: "File contains less than 2 characters", -3: "out of memory",
          -4: "CUDA/NCCL failure or no usable device", -5: "engine state error"}


class BpeCudaError(RuntimeError):
    def __init__(self, rc):
        msg = _lib.load().bpe_cuda_last_error()
        super().__init__(f"bpe_cuda rc={rc} ({ERRORS.get(rc, '?')}): {msg.decode() if msg else ''}")
        self.rc = rc


def _as_bytes_array(data):
    if isinstance(data, (bytes, bytearray, memoryview)):
        return np.frombuffer(data, dtype=np.uint8)
    arr = np.asarray(data)
    if arr.dtype != np.uint8:
        raise TypeError("corpus must be bytes or a uint8 array")
    return np.ascontiguousarray(arr)


def _pairs_to_numpy(ptr, n):
    if n == 0:
        return np.zeros((0, 2), dtype=np.uint32)
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint32)), shape=(n, 2)).copy()


def train(data, max_merges=0, n_gpus=1):
    """bytes -> (merges [k,2] uint32, ids [m] uint32, stats dict).  max_merges=0: to exhaustion."""
    lib = _lib.load()
    arr = _as_bytes_array(data)
    merges = C.POINTER(Pair)()
    tokens = C.POINTER(C.c_uint32)()
    nm, nt = C.c_size_t(), C.c_size_t()
    st = Stats()
    rc = lib.bpe_cuda_train(arr.ctypes.data, arr.size, max_merges, n_gpus, C.byref(merges), C.byref(nm), C.byref(tokens),
                            C.byref(nt), C.byref(st))
    if rc:
        raise BpeCudaError(rc)
    try:
        m = _pairs_to_numpy(merges, nm.value)
        t = np.ctypeslib.as_array(tokens, shape=(nt.value,)).copy() if nt.value else np.zeros(0, np.uint32)
    finally:
        lib.bpe_cuda_free(merges)
        lib.bpe_cuda_free(tokens)
    return m, t, st.as_dict()


def train_file(path, max_merges=0, n_gpus=1):
    """train() on a file: read in pinned 32 MB pieces that are copied, widened and counted while the next one is read
    (bpe.c:130-180, 555, 580-584 in front of the merge loop)."""
    lib = _lib.load()
    merges = C.POINTER(Pair)()
    tokens = C.POINTER(C.c_uint32)()
    nm, nt = C.c_size_t(), C.c_size_t()
    st = Stats()
    rc = lib.bpe_cuda_train_file(str(path).encode(), max_merges, n_gpus, C.byref(merges), C.byref(nm), C.byref(tokens), C.byref(nt),
                                 C.byref(st))
    if rc:
        raise BpeCudaError(rc)
    try:
        m = _pairs_to_numpy(merges, nm.value)
        t = np.ctypeslib.as_array(tokens, shape=(nt.value,)).copy() if nt.value else np.zeros(0, np.uint32)
    finally:
        lib.bpe_cuda_free(merges)
        lib.bpe_cuda_free(tokens)
    return m, t, st.as_dict()


def encode_file(path, merges, n_gpus=1):
    lib = _lib.load()
    mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
    tokens = C.POINTER(C.c_uint32)()
    nt = C.c_size_t()
    st = Stats()
    rc = lib.bpe_cuda_encode_file(str(path).encode(), mg.ctypes.data, mg.shape[0], n_gpus, C.byref(tokens), C.byref(nt), C.byref(st))
    if rc:
        raise BpeCudaError(rc)
    try:
        t = np.ctypeslib.as_array(tokens, shape=(nt.value,)).copy() if nt.value else np.zeros(0, np.uint32)
    finally:
        lib.bpe_cuda_free(tokens)
    return t, st.as_dict()


def encode(data, merges, n_gpus=1):
    """Apply a learned merge list (rank r -> id 256+r) to bytes -> (ids, stats)."""
    lib = _lib.load()
    arr = _as_bytes_array(data)
    mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
    tokens = C.POINTER(C.c_uint32)()
    nt = C.c_size_t()
    st = Stats()
    rc = lib.bpe_cuda_encode(arr.ctypes.data, arr.size, mg.ctypes.data, mg.shape[0], n_gpus, C.byref(tokens), C.byref(nt),
                             C.byref(st))
    if rc:
        raise BpeCudaError(rc)
    try:
        t = np.ctypeslib.as_array(tokens, shape=(nt.value,)).copy() if nt.value else np.zeros(0, np.uint32)
    finally:
        lib.bpe_cuda_free(tokens)
    return t, st.as_dict()


def _as_batch(docs):
    """docs: a sequence of bytes-like objects, or a (uint8 array, uint64 offsets) tuple -> (bytes, offsets) arrays.
    Only an offsets array of dtype uint64 selects the tuple form: a tuple of two uint8 documents stays two documents."""
    if (isinstance(docs, tuple) and len(docs) == 2 and isinstance(docs[0], np.ndarray) and isinstance(docs[1], np.ndarray)
            and docs[1].dtype == np.uint64):
        data = _as_bytes_array(docs[0])
        off = np.ascontiguousarray(docs[1])
        if off.ndim != 1 or off.size < 1 or int(off[-1]) > data.size:
            raise ValueError("offsets must be 1-D, hold n_docs + 1 values and end inside the byte array")
        return data, off
    parts = [memoryview(d).cast("B") for d in docs]
    off = np.zeros(len(parts) + 1, dtype=np.uint64)
    np.cumsum([p.nbytes for p in parts], out=off[1:])
    return np.frombuffer(b"".join(parts), dtype=np.uint8), off


def encode_batch(docs, merges):
    """Encode every document on its own (each cut at its first NUL) in one call on device 0.
    -> (ids uint32[m], offsets uint64[n_docs + 1], stats): ids[offsets[i]:offsets[i+1]] == encode(docs[i], merges)."""
    lib = _lib.load()
    data, off = _as_batch(docs)
    mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
    tokens = C.POINTER(C.c_uint32)()
    toff = C.POINTER(C.c_uint64)()
    nt = C.c_size_t()
    st = Stats()
    rc = lib.bpe_cuda_encode_batch(data.ctypes.data, off.ctypes.data, off.size - 1, mg.ctypes.data, mg.shape[0],
                                   C.byref(tokens), C.byref(toff), C.byref(nt), C.byref(st))
    if rc:
        raise BpeCudaError(rc)
    try:
        t = np.ctypeslib.as_array(tokens, shape=(nt.value,)).copy() if nt.value else np.zeros(0, np.uint32)
        o = np.ctypeslib.as_array(toff, shape=(off.size,)).copy()
    finally:
        lib.bpe_cuda_free(tokens)
        lib.bpe_cuda_free(toff)
    return t, o, st.as_dict()


def _as_id_batch(docs):
    """docs: a sequence of id arrays, or a (uint32 ids, uint64 offsets) tuple as encode_batch() returns ->
    (ids, offsets) arrays.  As in _as_batch, only an offsets array of dtype uint64 selects the tuple form."""
    if (isinstance(docs, tuple) and len(docs) == 2 and isinstance(docs[0], np.ndarray) and isinstance(docs[1], np.ndarray)
            and docs[1].dtype == np.uint64):
        ids = np.ascontiguousarray(np.asarray(docs[0], dtype=np.uint32).reshape(-1))
        off = np.ascontiguousarray(docs[1])
        if off.ndim != 1 or off.size < 1 or int(off[-1]) > ids.size:
            raise ValueError("offsets must be 1-D, hold n_docs + 1 values and end inside the id array")
        return ids, off
    parts = [np.asarray(d, dtype=np.uint32).reshape(-1) for d in docs]
    off = np.zeros(len(parts) + 1, dtype=np.uint64)
    np.cumsum([p.size for p in parts], out=off[1:])
    ids = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint32)
    return np.ascontiguousarray(ids, dtype=np.uint32), off


def decode_batch(docs, merges):
    """Decode every id sequence of a batch in one call on device 0 -> (bytes, offsets uint64[n_docs + 1], stats):
    bytes[offsets[i]:offsets[i+1]] == decode(docs[i], merges)[0].  decode_batch(encode_batch(d, m)[:2], m) round-trips."""
    lib = _lib.load()
    ids, off = _as_id_batch(docs)
    mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
    out = C.POINTER(C.c_uint8)()
    boff = C.POINTER(C.c_uint64)()
    nb = C.c_size_t()
    st = Stats()
    rc = lib.bpe_cuda_decode_batch(ids.ctypes.data if ids.size else None, off.ctypes.data, off.size - 1,
                                   mg.ctypes.data if mg.size else None, mg.shape[0], C.byref(out), C.byref(boff),
                                   C.byref(nb), C.byref(st))
    if rc:
        raise BpeCudaError(rc)
    try:
        b = C.string_at(out, nb.value)
        o = np.ctypeslib.as_array(boff, shape=(off.size,)).copy()
    finally:
        lib.bpe_cuda_free(out)
        lib.bpe_cuda_free(boff)
    return b, o, st.as_dict()


def decode(tokens, merges):
    """ids -> bytes through the merge list (what decompress() computes, bpe.c:341-394) -> (bytes, stats)."""
    lib = _lib.load()
    tk = np.ascontiguousarray(np.asarray(tokens, dtype=np.uint32).reshape(-1))
    mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
    out = C.POINTER(C.c_uint8)()
    nb = C.c_size_t()
    st = Stats()
    rc = lib.bpe_cuda_decode(tk.ctypes.data if tk.size else None, tk.size, mg.ctypes.data if mg.size else None, mg.shape[0],
                             C.byref(out), C.byref(nb), C.byref(st))
    if rc:
        raise BpeCudaError(rc)
    try:
        b = C.string_at(out, nb.value)
    finally:
        lib.bpe_cuda_free(out)
    return b, st.as_dict()


class Context:
    """One GPU: keeps a corpus shard resident in HBM; train/encode can run on it repeatedly."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        self.h = C.c_void_p()
        rc = self.lib.bpe_cuda_ctx_create(device, C.byref(self.h))
        if rc:
            raise BpeCudaError(rc)

    def close(self):
        if self.h:
            self.lib.bpe_cuda_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name, value):
        if self.lib.bpe_cuda_ctx_set_option(self.h, name.encode(), int(value)):
            raise ValueError(f"unknown option {name}")

    def set_comm(self, rank, world, unique_id: bytes):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        rc = self.lib.bpe_cuda_ctx_set_comm(self.h, rank, world, buf)
        if rc:
            raise BpeCudaError(rc)

    def upload(self, data):
        arr = _as_bytes_array(data)
        rc = self.lib.bpe_cuda_ctx_upload(self.h, arr.ctypes.data, arr.size)
        if rc:
            raise BpeCudaError(rc)

    def upload_ptr(self, host_ptr, n):
        rc = self.lib.bpe_cuda_ctx_upload(self.h, host_ptr, n)
        if rc:
            raise BpeCudaError(rc)

    def upload_device(self, dev_ptr, n):
        rc = self.lib.bpe_cuda_ctx_upload_device(self.h, dev_ptr, n)
        if rc:
            raise BpeCudaError(rc)

    def train(self, max_merges=0):
        st = Stats()
        rc = self.lib.bpe_cuda_ctx_train(self.h, max_merges, C.byref(st))
        if rc:
            raise BpeCudaError(rc)
        return st.as_dict()

    def encode(self, merges):
        mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
        st = Stats()
        rc = self.lib.bpe_cuda_ctx_encode(self.h, mg.ctypes.data, mg.shape[0], C.byref(st))
        if rc:
            raise BpeCudaError(rc)
        return st.as_dict()

    def encode_batch(self, docs, merges):
        """encode_batch() on this context: the resident shard and the last train/encode results stay as they are, and
        the pair -> rank table is kept for the next batch with the same merge list."""
        data, off = _as_batch(docs)
        mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
        ids = np.empty(max(1, int(off[-1]) - int(off[0])), dtype=np.uint32)   # ids <= bytes
        toff = np.empty(off.size, dtype=np.uint64)
        st = Stats()
        rc = self.lib.bpe_cuda_ctx_encode_batch(self.h, data.ctypes.data, off.ctypes.data, off.size - 1, mg.ctypes.data,
                                                mg.shape[0], ids.ctypes.data, toff.ctypes.data, C.byref(st))
        if rc:
            raise BpeCudaError(rc)
        return ids[:int(toff[-1])].copy(), toff, st.as_dict()

    def decode(self, merges, download=True):
        """Expand this rank's token stream of the last run on the device -> bytes (or their count)."""
        mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
        nb = C.c_size_t()
        rc = self.lib.bpe_cuda_ctx_decode(self.h, mg.ctypes.data if mg.size else None, mg.shape[0], C.byref(nb))
        if rc:
            raise BpeCudaError(rc)
        if not download:
            return nb.value
        buf = np.zeros(nb.value, dtype=np.uint8)
        rc = self.lib.bpe_cuda_ctx_decode_download(self.h, buf.ctypes.data if nb.value else None)
        if rc:
            raise BpeCudaError(rc)
        return buf.tobytes()

    def decode_batch(self, docs, merges, download=True):
        """decode_batch() on this context -> (bytes, offsets, stats).  With download=False the bytes stay on the device
        (as after decode()) and the first element is their count.  The resident shard and the last train/encode
        results stay as they are, and the flattened vocabulary is kept for the next call with the same merge list."""
        ids, off = _as_id_batch(docs)
        mg = np.ascontiguousarray(np.asarray(merges, dtype=np.uint32).reshape(-1, 2))
        boff = np.empty(off.size, dtype=np.uint64)
        nb = C.c_size_t()
        st = Stats()
        rc = self.lib.bpe_cuda_ctx_decode_batch(self.h, ids.ctypes.data if ids.size else None, off.ctypes.data, off.size - 1,
                                                mg.ctypes.data if mg.size else None, mg.shape[0], boff.ctypes.data,
                                                C.byref(nb), C.byref(st))
        if rc:
            raise BpeCudaError(rc)
        if not download:
            return nb.value, boff, st.as_dict()
        buf = np.zeros(nb.value, dtype=np.uint8)
        rc = self.lib.bpe_cuda_ctx_decode_download(self.h, buf.ctypes.data if nb.value else None)
        if rc:
            raise BpeCudaError(rc)
        return buf.tobytes(), boff, st.as_dict()

    def decode_mismatches(self):
        """Bytes of the last decode that differ from the resident shard (compared on the device)."""
        d = C.c_uint64()
        rc = self.lib.bpe_cuda_ctx_decode_compare(self.h, C.byref(d))
        if rc:
            raise BpeCudaError(rc)
        return d.value

    def result_sizes(self):
        nm, nt = C.c_size_t(), C.c_size_t()
        self.lib.bpe_cuda_ctx_result_sizes(self.h, C.byref(nm), C.byref(nt))
        return nm.value, nt.value

    def download(self, merges=True, tokens=True):
        nm, nt = self.result_sizes()
        m = np.zeros((nm, 2), dtype=np.uint32)
        t = np.zeros(nt, dtype=np.uint32)
        rc = self.lib.bpe_cuda_ctx_download(self.h, m.ctypes.data if merges and nm else None,
                                            t.ctypes.data if tokens and nt else None)
        if rc:
            raise BpeCudaError(rc)
        return m, t

    def download_into(self, merges_ptr, tokens_ptr):
        rc = self.lib.bpe_cuda_ctx_download(self.h, merges_ptr, tokens_ptr)
        if rc:
            raise BpeCudaError(rc)


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    rc = _lib.load().bpe_cuda_nccl_unique_id(buf)
    if rc:
        raise BpeCudaError(rc)
    return buf.raw


# ---- reference-shaped helpers (bpe/inc/bpe.h) ---------------------------------------------------
def get_file(path):
    """bpe.c:130-180: whole file; compress() then cuts it at the first NUL (bpe.c:555)."""
    with open(path, "rb") as f:
        return f.read()


def compress(path, max_merges=0, n_gpus=1):
    """bpe.c:541-811.  Returns (pair_arr, encoding): pair_arr[i] = (i, 0) for i < 256 and the k-th
    merge at 256+k, exactly the dyn_arr the reference returns; None on failure like the reference."""
    if path is None:
        return None
    if not os.path.isfile(path) or not os.access(path, os.R_OK):
        print(f"fopen: {os.strerror(2 if not os.path.exists(path) else 13)}", file=sys.stderr)  # bpe.c:135
        return None
    try:
        merges, ids, _ = train_file(path, max_merges=max_merges, n_gpus=n_gpus)
    except BpeCudaError as e:
        if e.rc == -2:
            print("Error: File contains less than 2 characters")  # stdout, bpe.c:560
        else:
            print(str(e), file=sys.stderr)
        return None
    pair_arr = np.zeros((256 + len(merges), 2), dtype=np.uint32)
    pair_arr[:256, 0] = np.arange(256, dtype=np.uint32)  # bpe.c:598-608
    pair_arr[256:] = merges
    return pair_arr, ids


def print_text(text, length=None, file=None):
    """bpe.c:182-196."""
    out = file or sys.stdout
    n = len(text) if length is None else length
    parts = []
    for t in text[:n]:
        t = int(t)
        parts.append(f"[{t}]" if t < 32 or t > 126 else chr(t))
    out.write("".join(parts) + "\n")


def dump_pairs(path, pair_arr):
    """Merge table file, the reference's record format (bpe.c:243-278: LE {u32 a,u32 b} from id 256).
    Unlike the reference (uint16_t counter, `< last_index`, bpe.c:258) every merge is written."""
    arr = np.asarray(pair_arr, dtype=np.uint32).reshape(-1, 2)
    arr[256:].astype("<u4").tofile(path)
    return True


def read_pairs(path):
    """bpe.c:280-339."""
    m = np.fromfile(path, dtype="<u4")
    m = m[: (m.size // 2) * 2].reshape(-1, 2)
    pair_arr = np.zeros((256 + len(m), 2), dtype=np.uint32)
    pair_arr[:256, 0] = np.arange(256, dtype=np.uint32)
    pair_arr[256:] = m
    return pair_arr
