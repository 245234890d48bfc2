"""Batch engine: the frisk hot path on one B200 through the C ABI.

Host side (pure CPU, testable without a GPU): ``PackedGenome`` (FASTA / in-memory scaffolds ->
2-bit planes, replaces iterFasta + countN, F:139-164 / F:106-118) and ``WindowList`` (candidate
windows, replaces crawlGenome's enumeration, F:194-251).

Device side: ``DeviceGenome`` (planes resident in HBM as torch tensors -- torch is only the
allocator/stream provider), ``background`` / ``finalize`` / ``genome_ivom`` / ``score`` (thin
wrappers of the C entry points) and ``run`` (the whole path, one GPU).  ``run_host`` is the single
C call from pinned host buffers used for end-to-end timing.
"""
from __future__ import annotations

import ctypes as C
import sys
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib

SeqLike = Union[np.ndarray, bytes, str]


def _torch_loaded() -> bool:
    return "torch" in sys.modules


class DevBuf:
    """Device memory owned through the C ABI (frisk_b200_device_alloc): what holds the planes when PyTorch is
    not in the process (the CLI path never imports it: the import alone takes longer than the run)."""

    def __init__(self, nbytes: int):
        p = C.c_void_p()
        _lib.check(_lib.lib().frisk_b200_device_alloc(C.byref(p), int(nbytes)), "frisk_b200_device_alloc")
        self._p, self.nbytes = p, int(nbytes)

    def data_ptr(self) -> int:
        return int(self._p.value or 0)

    def __del__(self):
        try:
            if self._p:
                _lib.lib().frisk_b200_device_free(self._p)
                self._p = C.c_void_p()
        except Exception:
            pass


def _device_index(device) -> int:
    if isinstance(device, int):
        return device
    text = str(device)
    return int(text.split(":")[1]) if ":" in text else 0


def _ptr(a) -> C.c_void_p:
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(int(a.data_ptr()))     # torch tensor


def _as_u8(seq: SeqLike) -> np.ndarray:
    if isinstance(seq, str):
        seq = seq.encode()
    if isinstance(seq, (bytes, bytearray)):
        return np.frombuffer(seq, dtype=np.uint8)
    return np.ascontiguousarray(seq, dtype=np.uint8)


_TORCH_DTYPE = {"uint8": "uint8", "uint32": "int32", "uint64": "int64", "float64": "float64", "int64": "int64", "int32": "int32"}


def _alloc(shape, dtype, pinned: bool) -> np.ndarray:
    """Host array, page-locked through torch when a GPU is present (the numpy view keeps the
    tensor's storage alive through its .base chain)."""
    dtype = np.dtype(dtype)
    if pinned:
        import torch
        if torch.cuda.is_available():
            t = torch.empty(shape, dtype=getattr(torch, _TORCH_DTYPE[dtype.name])).pin_memory()
            return t.numpy().view(dtype)
    return np.empty(shape, dtype=dtype)


_STAGING = {}


def _staging(tag: str, shape, dtype) -> np.ndarray:
    """A page-locked staging array that is reused from call to call (grown when too small): page-locking tens of MB
    costs milliseconds.  The contents are only valid until the next call with the same tag -- copy out of it."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    buf = _STAGING.get(tag)
    if buf is None or buf.nbytes < n:
        buf = _alloc(n + n // 4 + 4096, np.uint8, True)
        _STAGING[tag] = buf
    return buf[:n].view(dtype).reshape(shape)


def _alloc_u32(n: int, pinned: bool) -> np.ndarray:
    return _alloc(n, np.uint32, pinned)


def read_fasta_file(path: str) -> np.ndarray:
    """The file's bytes; ``.gz`` is inflated the way the reference opens it (F:144-147)."""
    if path.endswith(".gz"):
        import gzip
        with gzip.open(path, "rb") as fh:
            return np.frombuffer(fh.read(), dtype=np.uint8)
    return np.fromfile(path, dtype=np.uint8)


def is_bgzf(buf) -> bool:
    """Whether ``buf`` begins with a BGZF block (bgzip / samtools): a gzip member with CM 8, FLG = FEXTRA only and a
    ``BC`` extra subfield of length 2.  Such files are inflated on the device; a plain gzip member is not BGZF."""
    a = _as_u8(buf)
    if a.shape[0] < 18 or bytes(a[:4]) != b"\x1f\x8b\x08\x04":
        return False
    xlen = int(a[10]) | int(a[11]) << 8
    extra = bytes(a[12:12 + xlen])
    q = 0
    while q + 4 <= len(extra):
        slen = extra[q + 2] | extra[q + 3] << 8
        if extra[q:q + 2] == b"BC" and slen == 2:
            return True
        q += 4 + slen
    return False


def is_gzip(buf) -> bool:
    """Whether ``buf`` begins with a gzip member (1f 8b, CM 8) that is not BGZF: gzip, pigz, NCBI / Ensembl / UCSC
    ``.fa.gz``.  Such files are inflated on the device too (frisk_gzip.cu)."""
    a = _as_u8(buf)
    return a.shape[0] >= 18 and bytes(a[:3]) == b"\x1f\x8b\x08" and not is_bgzf(a)


TWOBIT_SIGNATURE = 0x1A412743


def is_2bit(buf) -> bool:
    """Whether ``buf`` begins with the signature of a UCSC .2bit file, in either byte order (a big-endian file stores
    every integer byte-swapped).  Such files are decoded on the device straight into the planes (frisk_twobit.cu)."""
    a = _as_u8(buf)
    return a.shape[0] >= 16 and int.from_bytes(bytes(a[:4]), "little") in (TWOBIT_SIGNATURE, 0x4327411A)


def read_genome_file(path: str) -> Tuple[np.ndarray, bool]:
    """(bytes, bgzf): a BGZF file as it is on disk (the device inflates it), any other file as ``read_fasta_file``
    gives it (a single-member ``.gz`` inflated on the host, text as it is)."""
    raw = np.fromfile(path, dtype=np.uint8)
    if is_bgzf(raw):
        return raw, True
    return (read_fasta_file(path) if path.endswith(".gz") else raw), False


def read_genome_raw(path: str) -> Tuple[np.ndarray, str]:
    """(bytes, kind) as the file is on disk: kind "2bit" (a UCSC .2bit file, by its signature, whatever the extension),
    "bgzf" (BGZF), "gzip" (a ``.gz`` with a plain gzip member) or "text".  Compressed files are left to the device to
    inflate; a ``.gz`` that is neither is read by ``read_fasta_file``."""
    raw = np.fromfile(path, dtype=np.uint8)
    if is_2bit(raw):
        return raw, "2bit"
    if is_bgzf(raw):
        return raw, "bgzf"
    if path.endswith(".gz"):
        return (raw, "gzip") if is_gzip(raw) else (read_fasta_file(path), "text")
    return raw, "text"


def open_genome_file(path: str, opener) -> "DeviceGenome":
    """``opener(bytes, kind)`` on the file as it is on disk; a gzip file the device refuses as unsupported (more than one
    member) is inflated on the host by ``read_fasta_file`` and opened as text."""
    buf, kind = read_genome_raw(path)
    if kind != "gzip":
        return opener(buf, kind)
    try:
        return opener(buf, kind)
    except _lib.FriskError as e:
        if e.code != _lib.E_UNSUPPORTED:
            raise
    return opener(read_fasta_file(path), "text")


def bgzf_text_len(gz) -> int:
    """Inflated size of a BGZF buffer, from its block headers and trailers alone (FriskError: not BGZF)."""
    buf = _as_u8(gz)
    nb, tl = C.c_uint64(0), C.c_uint64(0)
    _lib.check(_lib.lib().frisk_b200_bgzf_blocks(_ptr(buf), buf.shape[0], 0, None, None, None, None, C.byref(nb), C.byref(tl)),
               "frisk_b200_bgzf_blocks")
    return int(tl.value)


def twobit_records(buf) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(name_off, name_len, seq_len) of a .2bit buffer, parsed and checked on the host (frisk_b200_2bit_records;
    FriskError E_FORMAT for a malformed file).  Name offsets index ``buf``."""
    L = _lib.lib()
    a = _as_u8(buf)
    n, bases = C.c_uint64(0), C.c_uint64(0)
    _lib.check(L.frisk_b200_2bit_records(_ptr(a), a.shape[0], 0, None, None, None, C.byref(n), C.byref(bases)),
               "frisk_b200_2bit_records")
    R = int(n.value)
    name_off = np.zeros(R, np.uint64); name_len = np.zeros(R, np.uint32); seq_len = np.zeros(R, np.uint64)
    _lib.check(L.frisk_b200_2bit_records(_ptr(a), a.shape[0], R, _ptr(name_off), _ptr(name_len), _ptr(seq_len), C.byref(n),
                                         C.byref(bases)), "frisk_b200_2bit_records")
    return name_off, name_len, seq_len


def _name_source(L, h, buf: np.ndarray, device_text: bool) -> np.ndarray:
    """What a handle's name offsets index: the caller's text, or -- a BGZF, gzip or .2bit open, whose text never leaves
    the device or does not exist -- the handle's buffer of names (copied: it goes with the handle)."""
    if not device_text:
        return buf
    p, n = C.c_void_p(), C.c_uint64(0)
    _lib.check(L.frisk_b200_fasta_name_text(h, C.byref(p), C.byref(n)), "frisk_b200_fasta_name_text")
    return np.frombuffer(C.string_at(p.value, n.value), dtype=np.uint8) if n.value else np.zeros(0, np.uint8)


def _decode_names(buf: np.ndarray, name_off: np.ndarray, name_len: np.ndarray) -> List[str]:
    """Header tokens -> str.  All name bytes are gathered with one fancy-index (a 1 M-scaffold
    assembly must not pay a numpy slice of a multi-GB buffer per record), then cut up."""
    n = len(name_off)
    if n == 0:
        return []
    lens = name_len.astype(np.int64)
    ends = np.cumsum(lens)
    starts = ends - lens
    idx = np.repeat(name_off.astype(np.int64) - starts, lens) + np.arange(int(ends[-1]), dtype=np.int64)
    flat = buf[idx].tobytes().decode()
    return [flat[a:b] for a, b in zip(starts.tolist(), ends.tolist())]


class LazyNames:
    """The scaffold names of a FASTA text, decoded from the header positions on first use: a fragmented assembly has a
    million of them, and a caller that only wants rows (``row_scaf`` indexes the scaffolds) never pays for the strings."""

    def __init__(self, buf: np.ndarray, name_off: np.ndarray, name_len: np.ndarray):
        self._src = (buf, name_off, name_len)
        self._n = int(len(name_off))
        self._names: Optional[List[str]] = None

    def _all(self) -> List[str]:
        if self._names is None:
            self._names = _decode_names(*self._src)
            self._src = None
        return self._names

    def __len__(self) -> int:
        return self._n

    def __getitem__(self, i):
        return self._all()[i]

    def __iter__(self):
        return iter(self._all())

    def __eq__(self, other):
        return list(self) == list(other)

    def __repr__(self):
        return "LazyNames(%d)" % self._n


@dataclass
class WindowList:
    """Candidate windows in crawlGenome order (F:194-251), before the 30 % unresolved filter."""
    off: np.ndarray      # uint64 absolute base offset in the packed planes
    length: np.ndarray   # uint32
    scaf: np.ndarray     # uint32 scaffold index
    start: np.ndarray    # int64, reference coordinates (F:243/F:245)
    stop: np.ndarray     # int64

    def __len__(self) -> int:
        return int(self.off.shape[0])

    @property
    def max_len(self) -> int:
        m = self.__dict__.get("_max_len")
        if m is None:                                  # (a pass over the list: computed once, the one-call paths ask every call)
            m = int(self.length.max()) if len(self) else 0
            self.__dict__["_max_len"] = m
        return m

    def slice(self, a: int, b: int) -> "WindowList":
        return WindowList(self.off[a:b], self.length[a:b], self.scaf[a:b], self.start[a:b], self.stop[a:b])


@dataclass
class PackedGenome:
    names: List[str]
    scaf_len: np.ndarray          # uint64
    scaf_off: np.ndarray          # uint64 (multiples of 128)
    padded_len: int
    codes: np.ndarray             # uint32, padded_len/16 words
    inv: np.ndarray               # uint32, padded_len/32 words
    low: Optional[np.ndarray]     # uint32 or None when the input has no lower case
    total_len: int                # F:323
    nn_total: int                 # F:325: characters that are not upper-case ATGC
    n_lower: int
    pinned: bool = False          # planes (and the window arrays derived from them) are page-locked

    # ------------------------------------------------------------------ constructors
    @classmethod
    def from_scaffolds(cls, scaffolds: Sequence[Tuple[str, SeqLike]], pinned: bool = False,
                       threads: int = 0) -> "PackedGenome":
        names = [n for n, _ in scaffolds]
        arrs = [_as_u8(s) for _, s in scaffolds]
        lens = np.array([a.shape[0] for a in arrs], dtype=np.uint64)
        src = np.concatenate(arrs) if arrs else np.zeros(0, np.uint8)
        end = np.cumsum(lens, dtype=np.uint64)
        off = end - lens
        return cls._pack(names, src, off, end, lens, pinned, threads)

    @classmethod
    def from_fasta_bytes(cls, text: Union[bytes, np.ndarray], pinned: bool = False, threads: int = 0) -> "PackedGenome":
        L = _lib.lib()
        buf = _as_u8(text)
        n = C.c_uint64(0)
        # one pass over the text with a guessed record capacity (one record per 2 KiB + 1024); a second one with the exact
        # count only when the guess was too small (the scan reports the count either way)
        cap = buf.shape[0] // 2048 + 1024
        while True:
            name_off = np.zeros(cap, np.uint64); name_len = np.zeros(cap, np.uint32)
            body_off = np.zeros(cap, np.uint64); body_end = np.zeros(cap, np.uint64); seq_len = np.zeros(cap, np.uint64)
            rc = L.frisk_b200_fasta_scan(_ptr(buf), buf.shape[0], cap, _ptr(name_off), _ptr(name_len), _ptr(body_off),
                                         _ptr(body_end), _ptr(seq_len), C.byref(n))
            if rc == _lib.E_CAPACITY and int(n.value) > cap:
                cap = int(n.value)
                continue
            _lib.check(rc, "frisk_b200_fasta_scan")
            break
        k = int(n.value)
        return cls._pack(_decode_names(buf, name_off[:k], name_len[:k]), buf, body_off[:k], body_end[:k], seq_len[:k], pinned,
                         threads)

    @classmethod
    def from_2bit_bytes(cls, buf: Union[bytes, np.ndarray], pinned: bool = False) -> "PackedGenome":
        """A UCSC .2bit buffer decoded on the host (frisk_b200_2bit_unpack_host): the same planes, records and countN
        statistics as the genome's FASTA through ``from_fasta_bytes``."""
        L = _lib.lib()
        a = _as_u8(buf)
        name_off, name_len, lens = twobit_records(a)
        n = len(lens)
        scaf_off = np.zeros(n, np.uint64)
        padded = C.c_uint64(0)
        _lib.check(L.frisk_b200_pack_layout(_ptr(lens), n, _ptr(scaf_off), C.byref(padded)), "frisk_b200_pack_layout")
        P = int(padded.value)
        codes = _alloc_u32(P // 16, pinned)
        inv = _alloc_u32(P // 32, pinned)
        low = _alloc_u32(P // 32, pinned)
        stats = np.zeros(3, np.uint64)
        _lib.check(L.frisk_b200_2bit_unpack_host(_ptr(a), a.shape[0], P, _ptr(codes), _ptr(inv), _ptr(low), _ptr(stats)),
                   "frisk_b200_2bit_unpack_host")
        n_lower = int(stats[2])
        return cls(_decode_names(a, name_off, name_len), lens, scaf_off, P, codes, inv, low if n_lower else None, int(stats[0]),
                   int(stats[1]), n_lower, bool(pinned))

    @classmethod
    def from_fasta(cls, path: str, pinned: bool = False, threads: int = 0) -> "PackedGenome":
        """A FASTA file (``.gz`` inflated on the host), or a .2bit file, recognised by its signature."""
        raw = np.fromfile(path, dtype=np.uint8)
        if is_2bit(raw):
            return cls.from_2bit_bytes(raw, pinned)
        return cls.from_fasta_bytes(read_fasta_file(path) if path.endswith(".gz") else raw, pinned, threads)

    @classmethod
    def _pack(cls, names, src, src_off, src_end, lens, pinned, threads) -> "PackedGenome":
        L = _lib.lib()
        n = len(names)
        lens = np.ascontiguousarray(lens, np.uint64)
        src_off = np.ascontiguousarray(src_off, np.uint64)
        src_end = np.ascontiguousarray(src_end, np.uint64)
        scaf_off = np.zeros(n, np.uint64)
        padded = C.c_uint64(0)
        _lib.check(L.frisk_b200_pack_layout(_ptr(lens), n, _ptr(scaf_off), C.byref(padded)), "frisk_b200_pack_layout")
        P = int(padded.value)
        codes = _alloc_u32(P // 16, pinned)
        inv = _alloc_u32(P // 32, pinned)
        low = _alloc_u32(P // 32, pinned)
        stats = np.zeros(3, np.uint64)
        _lib.check(L.frisk_b200_pack(_ptr(src), _ptr(src_off), _ptr(src_end), _ptr(lens), _ptr(scaf_off), n, P,
                                     _ptr(codes), _ptr(inv), _ptr(low), _ptr(stats), threads), "frisk_b200_pack")
        n_lower = int(stats[2])
        return cls(names, lens, scaf_off, P, codes, inv, low if n_lower else None, int(stats[0]), int(stats[1]), n_lower,
                   bool(pinned))

    # ------------------------------------------------------------------ host logic
    def windows(self, w: int = 5000, step: int = 2500, scaffolds_all: bool = False) -> WindowList:
        L = _lib.lib()
        n = C.c_uint64(0)
        nsc = len(self.names)
        if w < 1 or step < 1:
            _lib.check(_lib.E_INVALID, "frisk_b200_windows")
        # one pass: a scaffold yields at most len // step + 2 windows (the grid, the tail jump-back, the --scaffoldsAll rescue)
        cap = int((self.scaf_len.astype(np.int64) // step + 2).sum()) if nsc else 0
        pinned = self.pinned
        off = _alloc(cap, np.uint64, pinned); ln = _alloc(cap, np.uint32, pinned)     # these two go to the device
        sc = np.zeros(cap, np.uint32)
        st = np.zeros(cap, np.int64); sp = np.zeros(cap, np.int64)
        _lib.check(L.frisk_b200_windows(_ptr(self.scaf_len), _ptr(self.scaf_off), nsc, w, step, int(scaffolds_all), cap,
                                        _ptr(off), _ptr(ln), _ptr(sc), _ptr(st), _ptr(sp), C.byref(n)),
                   "frisk_b200_windows")
        k = int(n.value)
        return WindowList(off[:k], ln[:k], sc[:k], st[:k], sp[:k])

    def inv_sparse(self) -> Tuple[np.ndarray, np.ndarray]:
        """The invalid plane's non-zero words as (word index, word) arrays (frisk_b200_plane_sparse),
        page-locked when the planes are; computed once."""
        if getattr(self, "_inv_sparse", None) is None:
            L = _lib.lib()
            n = C.c_uint64(0)
            nw = self.inv.shape[0]
            _lib.check(L.frisk_b200_plane_sparse(_ptr(self.inv), nw, 0, None, None, C.byref(n)), "frisk_b200_plane_sparse")
            cap = int(n.value)
            idx = _alloc(max(cap, 1), np.uint32, self.pinned)
            val = _alloc(max(cap, 1), np.uint32, self.pinned)
            _lib.check(L.frisk_b200_plane_sparse(_ptr(self.inv), nw, cap, _ptr(idx), _ptr(val), C.byref(n)),
                       "frisk_b200_plane_sparse")
            self._inv_sparse = (idx[:cap], val[:cap])
        return self._inv_sparse

    def prefers_sparse(self) -> bool:
        """Upload the invalid plane as its non-zero words?  (when that is at most a quarter of the dense plane; cached)"""
        v = getattr(self, "_prefers_sparse", None)
        if v is None:
            v = 8 * len(self.inv_sparse()[0]) <= self.inv.nbytes // 4 and self.padded_len // 32 < 2 ** 32
            self._prefers_sparse = v
        return v

    def ex_max(self, kmax: int, valid_kmax: int) -> int:
        """exMax (F:344): kmax-words that contain an invalid character."""
        possible = np.maximum(self.scaf_len.astype(np.int64) - kmax + 1, 0).sum()
        return int(possible) - int(valid_kmax)

    @property
    def genome_space(self) -> int:
        return self.total_len - self.nn_total     # F:379

    @property
    def plane_bytes(self) -> int:
        if self.codes is None:      # planes exist on the device only (DeviceGenome.from_fasta_bytes)
            return self.padded_len // 4 + self.padded_len // 8 * (2 if self.n_lower else 1)
        return self.codes.nbytes + self.inv.nbytes + (self.low.nbytes if self.low is not None else 0)


# ---------------------------------------------------------------------- device side
class DeviceGenome:
    """The packed planes resident in HBM (torch tensors used purely as device buffers)."""

    def __init__(self, g: PackedGenome, device="cuda:0", stream=None, planes=None):
        _lib.require_device()
        self.host = g
        if planes is not None and isinstance(planes[0], DevBuf):
            self.device = device                      # native planes: torch is not needed (and may not be loaded)
            self.codes, self.inv, self.low = planes
            return
        import torch
        self.device = torch.device(device)
        if planes is not None:
            self.codes, self.inv, self.low = planes
            return
        with torch.cuda.device(self.device):
            self.codes = torch.from_numpy(g.codes.view(np.int32)).to(self.device, non_blocking=True)
            self.inv = torch.from_numpy(g.inv.view(np.int32)).to(self.device, non_blocking=True)
            self.low = torch.from_numpy(g.low.view(np.int32)).to(self.device, non_blocking=True) if g.low is not None else None

    @classmethod
    def from_fasta_bytes_native(cls, text: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """``from_fasta_bytes`` without PyTorch: the planes are DevBuf allocations (cudaMalloc through the C
        ABI), work goes to the default stream.  Used by the CLI."""
        return cls._open_native(text, device, "text")

    @classmethod
    def from_bgzf_bytes_native(cls, gz: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """``from_fasta_bytes_native`` for a BGZF buffer: the compressed bytes go to the GPU and are inflated there."""
        return cls._open_native(gz, device, "bgzf")

    @classmethod
    def from_gzip_bytes_native(cls, gz: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """``from_fasta_bytes_native`` for one gzip member: the compressed bytes go to the GPU and are inflated there
        (FriskError E_UNSUPPORTED for a multi-member file)."""
        return cls._open_native(gz, device, "gzip")

    @classmethod
    def from_2bit_bytes_native(cls, buf: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """``from_fasta_bytes_native`` for a UCSC .2bit buffer: the file goes to the GPU and is decoded there."""
        return cls._open_native(buf, device, "2bit")

    @classmethod
    def _open_native(cls, text, device, kind: str) -> "DeviceGenome":
        _lib.require_device()
        L = _lib.lib()
        buf = _as_u8(text)
        _lib.check(L.frisk_b200_set_device(_device_index(device)), "frisk_b200_set_device")
        h = C.c_void_p()
        nrec, padded = C.c_uint64(0), C.c_uint64(0)
        stats = np.zeros(3, np.uint64)
        what = _OPENERS[kind]
        _lib.check(getattr(L, what)(_ptr(buf), buf.shape[0], None, C.byref(h), C.byref(nrec), C.byref(padded), _ptr(stats)), what)
        try:
            names_buf = _name_source(L, h, buf, kind != "text")
            R, P = int(nrec.value), int(padded.value)
            name_off = np.zeros(R, np.uint64); name_len = np.zeros(R, np.uint32)
            seq_len = np.zeros(R, np.uint64); scaf_off = np.zeros(R, np.uint64)
            _lib.check(L.frisk_b200_fasta_records(h, _ptr(name_off), _ptr(name_len), _ptr(seq_len), _ptr(scaf_off)),
                       "frisk_b200_fasta_records")
            codes, inv = DevBuf(P // 4), DevBuf(P // 8)
            low = DevBuf(P // 8) if int(stats[2]) else None
            _lib.check(L.frisk_b200_fasta_pack(h, _ptr(codes), _ptr(inv), _ptr(low), None), "frisk_b200_fasta_pack")
        finally:
            L.frisk_b200_fasta_close(h, None)
        names = _decode_names(names_buf, name_off, name_len)
        g = PackedGenome(names, seq_len, scaf_off, P, None, None, None, int(stats[0]), int(stats[1]), int(stats[2]), False)
        return cls(g, str(device), planes=(codes, inv, low))

    @classmethod
    def from_fasta_bytes(cls, text: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """Device-side ingest (frisk_ingest.cu): the raw FASTA text goes to the GPU once and is
        tokenised and 2-bit packed there; only the record table comes back.  ``self.host`` is a
        PackedGenome without host planes (names, lengths, layout, countN statistics)."""
        return cls._open(text, device, "text")

    @classmethod
    def from_bgzf_bytes(cls, gz: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """``from_fasta_bytes`` for a BGZF buffer (bgzip, samtools): the compressed bytes go to the GPU and are inflated
        there (frisk_bgzf.cu), straight into the ingest's text buffer; the text never exists on the host."""
        return cls._open(gz, device, "bgzf")

    @classmethod
    def from_gzip_bytes(cls, gz: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """``from_fasta_bytes`` for one gzip member (gzip, pigz): the compressed bytes go to the GPU and are inflated there
        (frisk_gzip.cu), straight into the ingest's text buffer.  FriskError E_UNSUPPORTED for a multi-member file."""
        return cls._open(gz, device, "gzip")

    @classmethod
    def from_2bit_bytes(cls, buf: Union[bytes, np.ndarray], device="cuda:0") -> "DeviceGenome":
        """``from_fasta_bytes`` for a UCSC .2bit buffer (frisk_twobit.cu): the file goes to the GPU in one copy and its
        packed bases, N blocks and mask blocks are decoded there straight into the planes."""
        return cls._open(buf, device, "2bit")

    @classmethod
    def _open(cls, text, device, kind: str) -> "DeviceGenome":
        import torch
        _lib.require_device()
        L = _lib.lib()
        buf = _as_u8(text)
        dev = torch.device(device)
        what = _OPENERS[kind]
        opener = getattr(L, what)
        with torch.cuda.device(dev):
            st = _stream_ptr(dev)
            h = C.c_void_p()
            nrec, padded = C.c_uint64(0), C.c_uint64(0)
            stats = np.zeros(3, np.uint64)
            _lib.check(opener(_ptr(buf), buf.shape[0], st, C.byref(h), C.byref(nrec), C.byref(padded), _ptr(stats)), what)
            try:
                names_buf = _name_source(L, h, buf, kind != "text")
                R, P = int(nrec.value), int(padded.value)
                name_off = np.zeros(R, np.uint64); name_len = np.zeros(R, np.uint32)
                seq_len = np.zeros(R, np.uint64); scaf_off = np.zeros(R, np.uint64)
                _lib.check(L.frisk_b200_fasta_records(h, _ptr(name_off), _ptr(name_len), _ptr(seq_len), _ptr(scaf_off)),
                           "frisk_b200_fasta_records")
                codes = torch.empty(P // 16, dtype=torch.int32, device=dev)
                inv = torch.empty(P // 32, dtype=torch.int32, device=dev)
                low = torch.empty(P // 32, dtype=torch.int32, device=dev) if int(stats[2]) else None
                _lib.check(L.frisk_b200_fasta_pack(h, _ptr(codes), _ptr(inv), _ptr(low), st), "frisk_b200_fasta_pack")
            finally:
                L.frisk_b200_fasta_close(h, st)
        names = LazyNames(names_buf, name_off, name_len)
        g = PackedGenome(names, seq_len, scaf_off, P, None, None, None, int(stats[0]), int(stats[1]), int(stats[2]), False)
        return cls(g, dev, planes=(codes, inv, low))

    @classmethod
    def from_fasta(cls, path: str, device="cuda:0") -> "DeviceGenome":
        """A FASTA file: BGZF and single-member gzip are inflated on the device, a multi-member ``.gz`` on the host
        (``read_fasta_file``); a .2bit file is decoded on the device."""
        return open_genome_file(path, lambda buf, kind: cls._open(buf, device, kind))

    def to_host(self) -> PackedGenome:
        """Copy the planes back (tests; the host packer must agree bit for bit)."""
        g = self.host
        low = self.low.cpu().numpy().view(np.uint32) if self.low is not None else None
        return PackedGenome(g.names, g.scaf_len, g.scaf_off, g.padded_len, self.codes.cpu().numpy().view(np.uint32),
                            self.inv.cpu().numpy().view(np.uint32), low, g.total_len, g.nn_total, g.n_lower, False)


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NULL_CTX = _NullCtx()


def _device_ctx(device):
    """``torch.cuda.device(device)`` -- or nothing when that device is current already (entering and leaving the context
    costs ~10 us of cudaSetDevice calls, which shows in a 1 ms call)."""
    import torch
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    return _NULL_CTX if torch.cuda.current_device() == idx else torch.cuda.device(dev)


def _stream_ptr(device) -> C.c_void_p:
    if not _torch_loaded():
        return C.c_void_p(0)                 # no torch in the process: the default stream
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def background(dg: DeviceGenome, kmax: int, mask_host: bool = False, d_fwd=None, first_base: int = 0,
               last_base: Optional[int] = None):
    """Forward-strand counts (adds into d_fwd, a device int64 tensor of table_size(1,kmax))."""
    import torch
    if d_fwd is None:
        d_fwd = torch.zeros(_lib.table_size(1, kmax), dtype=torch.int64, device=dg.device)
    if last_base is None:
        last_base = dg.host.padded_len - 32      # the last word is padding, only read as look-ahead
    with torch.cuda.device(dg.device):
        _lib.check(_lib.lib().frisk_b200_background(_ptr(dg.codes), _ptr(dg.inv), _ptr(dg.low), first_base, last_base,
                                                    kmax, int(mask_host), _ptr(d_fwd), _stream_ptr(dg.device)),
                   "frisk_b200_background")
    return d_fwd


def finalize(d_fwd, kmax: int, symmetric: bool = True):
    """-> (d_tables int64[table_size(1,kmax)], d_valid int64[1]) on the device of d_fwd."""
    import torch
    d_tables = torch.empty_like(d_fwd)
    d_valid = torch.zeros(1, dtype=torch.int64, device=d_fwd.device)
    with torch.cuda.device(d_fwd.device):
        _lib.check(_lib.lib().frisk_b200_finalize_tables(_ptr(d_fwd), kmax, int(symmetric), _ptr(d_tables), _ptr(d_valid),
                                                         _stream_ptr(d_fwd.device)), "frisk_b200_finalize_tables")
    return d_tables, d_valid


def genome_ivom(d_tables, kmin: int, kmax: int, genome_space: int):
    import torch
    d_ig = torch.empty(2 * 4 ** kmax, dtype=torch.float64, device=d_tables.device)
    with torch.cuda.device(d_tables.device):
        _lib.check(_lib.lib().frisk_b200_genome_ivom(_ptr(d_tables), kmin, kmax, int(genome_space), _ptr(d_ig),
                                                     _stream_ptr(d_tables.device)), "frisk_b200_genome_ivom")
    return d_ig


def score(dg: DeviceGenome, wins: WindowList, d_ig, kmin: int, kmax: int, rip: bool = True, dump: bool = False):
    """-> (d_rows float64[n,5], d_status int32[n], d_dump uint16-as-int16[n, table_size(1,kmax)] or None)."""
    import torch
    n = len(wins)
    dev = dg.device
    d_rows = torch.empty((n, 5), dtype=torch.float64, device=dev)
    d_status = torch.empty(n, dtype=torch.int32, device=dev)
    d_dump = torch.empty((n, _lib.table_size(1, kmax)), dtype=torch.int16, device=dev) if dump else None
    if n == 0:
        return d_rows, d_status, d_dump
    d_off = torch.from_numpy(wins.off.view(np.int64)).to(dev, non_blocking=True)
    d_len = torch.from_numpy(wins.length.view(np.int32)).to(dev, non_blocking=True)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().frisk_b200_score(_ptr(dg.codes), _ptr(dg.inv), _ptr(dg.low), _ptr(d_off), _ptr(d_len), n,
                                               wins.max_len, _ptr(d_ig), kmin, kmax, int(rip), _ptr(d_rows),
                                               _ptr(d_status), _ptr(d_dump), _stream_ptr(dev)), "frisk_b200_score")
    return d_rows, d_status, d_dump


_SLOT_CACHE = {}


def feature_slots(kmin: int, kmax: int) -> Tuple[np.ndarray, int]:
    """(slot int32[table_size(1,kmax)], n_features): position of every kept k-mer in the composition vector
    of frisk_b200_region_features (scrubMirrors order, F:797-811), -1 for the dropped mirror images."""
    key = (kmin, kmax)
    if key not in _SLOT_CACHE:
        slot = np.zeros(_lib.table_size(1, kmax), np.int32)
        n = C.c_uint64(0)
        _lib.check(_lib.lib().frisk_b200_feature_slots(kmin, kmax, _ptr(slot), C.byref(n)), "frisk_b200_feature_slots")
        _SLOT_CACHE[key] = (slot, int(n.value))
    return _SLOT_CACHE[key]


def region_features(dg: DeviceGenome, off: np.ndarray, length: np.ndarray, kmin: int = 1, kmax: int = 6) -> np.ndarray:
    """Strand-symmetric k-mer proportion vectors of the regions [off, off+length) of the packed planes, one
    CTA per region (frisk_b200_region_features): the reference's per-anomaly computeKmers(pcaMode, sym) +
    scrubMirrors + flattenKmerMap(prop=True), F:1571-1591, for every region at once.  -> float64 [n, F]."""
    import torch
    _lib.require_device()
    slot, nf = feature_slots(kmin, kmax)
    n = len(off)
    dev = dg.device
    d_out = torch.empty((n, nf), dtype=torch.float64, device=dev)
    if n:
        d_off = torch.from_numpy(np.ascontiguousarray(off, np.uint64).view(np.int64)).to(dev)
        d_len = torch.from_numpy(np.ascontiguousarray(length, np.uint32).view(np.int32)).to(dev)
        d_slot = torch.from_numpy(slot).to(dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().frisk_b200_region_features(_ptr(dg.codes), _ptr(dg.inv), _ptr(d_off), _ptr(d_len), n, kmin, kmax,
                                                             _ptr(d_slot), nf, _ptr(d_out), _stream_ptr(dev)),
                       "frisk_b200_region_features")
    return d_out.cpu().numpy()


@dataclass
class HotPathResult:
    kmin: int
    kmax: int
    tables: np.ndarray            # uint64, orders kmin..kmax concatenated, reference dict order
    meta: Tuple[int, int, int]    # totalLen, exMax, nnTotal (F:356-359)
    names: List[str]              # one per emitted row
    coords: np.ndarray            # int64 [n,2] start, stop
    rows: np.ndarray              # float64 [n,5] windowKLD, GC, PI, SI, CRI
    status: np.ndarray            # uint32 [n] FRISK_ROW_* bits (never EXCLUDED)
    n_candidates: int = 0
    win_index: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int64))  # candidate index of each row
    row_scaf: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int64))   # scaffold index (in the query) of each row
    win_tables: Optional[np.ndarray] = None   # uint16 [n, table_size(kmin,kmax)] when dump=True
    collective: str = ""                      # multi-GPU: how the counters were combined
    scaf_names: List[str] = field(default_factory=list)    # the query's scaffold names (row_scaf indexes this)

    def tsv_body(self, with_rip: bool) -> bytes:
        """The rows as the reference writes them to raw_window_scores.bed (F:1493): tab-separated,
        floats as str(float) -- formatted by frisk_b200_format_rows (threads) instead of a Python loop."""
        n = len(self.rows)
        enc = [s.encode() for s in self.scaf_names]
        lens = np.array([len(b) for b in enc], dtype=np.uint32)
        offs = (np.cumsum(lens, dtype=np.uint64) - lens).astype(np.uint64)
        blob = np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8)
        row_name = np.ascontiguousarray(self.row_scaf, dtype=np.uint32)
        start = np.ascontiguousarray(self.coords[:, 0], dtype=np.int64)
        stop = np.ascontiguousarray(self.coords[:, 1], dtype=np.int64)
        rows = np.ascontiguousarray(self.rows, dtype=np.float64)
        nv = 5 if with_rip else 2
        cap = int(lens[row_name].sum()) + n * (44 + 26 * nv) + 16 if n else 16
        out = np.empty(cap, dtype=np.uint8)
        nb = C.c_uint64(0)
        _lib.check(_lib.lib().frisk_b200_format_rows(_ptr(blob), _ptr(offs), _ptr(lens), _ptr(row_name), _ptr(start), _ptr(stop),
                                                     _ptr(rows), n, nv, _ptr(out), cap, C.byref(nb), 0), "frisk_b200_format_rows")
        return out[:int(nb.value)].tobytes()

    def raise_reference_errors(self) -> None:
        """The reference aborts on the first window that raises; mirror that when asked."""
        bad = np.nonzero(self.status & (_lib.ROW_KLD_ZERODIV | _lib.ROW_GC_ZERODIV))[0]
        if bad.size:
            i = int(bad[0])
            raise ZeroDivisionError("window %s:%d-%d: float division by zero (reference F:437/F:136)"
                                    % (self.names[i], self.coords[i, 0], self.coords[i, 1]))
        bad = np.nonzero(self.status & _lib.ROW_LOG_DOMAIN)[0]
        if bad.size:
            raise ValueError("math domain error (reference F:470)")


def _slice_orders(tab: np.ndarray, kmin: int, kmax: int) -> np.ndarray:
    return tab[..., _lib.table_size(1, kmin - 1):_lib.table_size(1, kmax)] if kmin > 1 else tab[..., :_lib.table_size(1, kmax)]


def assemble(query: PackedGenome, host: PackedGenome, wins: WindowList, tables_1k: np.ndarray, valid_kmax: int,
             rows: np.ndarray, status: np.ndarray, kmin: int, kmax: int, dump: Optional[np.ndarray] = None,
             names: bool = True) -> HotPathResult:
    """``names=False`` leaves the per-row name list empty (``row_scaf`` + ``scaf_names`` carry the same information
    without a Python object per row: millions of rows of a fragmented assembly)."""
    keep = (status & _lib.ROW_EXCLUDED) == 0
    n_all = len(status)
    if bool(keep.all()):
        # nothing excluded (the usual case for a genome without long N runs): plain copies instead of gathers -- this is
        # tens of MB per million windows, and host time counts in the ingest-inclusive figures
        idx = np.arange(n_all, dtype=np.int64)
        take = lambda a: np.array(a[:n_all], copy=True)
    else:
        idx = np.nonzero(keep)[0]
        take = lambda a: a[idx]
    want_names = bool(names)
    scaf = take(wins.scaf)
    names = [query.names[s] for s in scaf] if want_names else []
    if idx.size:
        coords = np.empty((idx.size, 2), np.int64)
        coords[:, 0] = take(wins.start)
        coords[:, 1] = take(wins.stop)
    else:
        coords = np.zeros((0, 2), np.int64)
    meta = (host.total_len, host.ex_max(kmax, valid_kmax), host.nn_total)
    wt = None
    if dump is not None:
        wt = _slice_orders(take(dump), kmin, kmax)
    return HotPathResult(kmin, kmax, _slice_orders(tables_1k, kmin, kmax).copy(), meta, names, coords,
                         take(rows), take(status).astype(np.uint32, copy=False), len(wins), idx, scaf.astype(np.int64), wt,
                         scaf_names=list(query.names) if want_names else query.names)


class Pipeline:
    """The device-resident hot path: planes, window list and all work buffers live in HBM; one
    ``enqueue()`` launches background -> [all-reduce] -> finalize -> genome IVOM -> score on the
    current stream without any host synchronisation (so it can be timed with CUDA events, replayed,
    or captured in a CUDA graph)."""

    def __init__(self, query: PackedGenome, host: Optional[PackedGenome] = None, kmin: int = 1, kmax: int = 8,
                 w: int = 5000, step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False,
                 rip: bool = True, device="cuda:0", dump: bool = False, allreduce=None,
                 genome_space: Optional[int] = None, wins: Optional[WindowList] = None,
                 bg_range: Optional[Tuple[int, int]] = None, peers=None):
        import torch
        _lib.require_device()
        rc = 0 if 1 <= kmin <= kmax else _lib.E_INVALID
        if kmax > _lib.MAX_K:
            rc = _lib.E_UNSUPPORTED
        _lib.check(rc, "frisk_b200 Pipeline(kmin=%d, kmax=%d)" % (kmin, kmax))
        # query / host may be PackedGenome (host planes, uploaded here) or DeviceGenome (already resident)
        host = host if host is not None else query
        self.dq = query if isinstance(query, DeviceGenome) else DeviceGenome(query, device)
        self.dh = self.dq if host is query else (host if isinstance(host, DeviceGenome) else DeviceGenome(host, device))
        query, host = self.dq.host, self.dh.host
        self.query, self.host = query, host
        self.kmin, self.kmax, self.mask_host, self.rip = kmin, kmax, mask_host, rip
        self.allreduce = allreduce
        # dist.PeerExchange: the all-reduce fused into the finalise kernels (counters summed straight
        # out of every rank's buffer over NVLink); `allreduce` is then unused
        self.peers = peers if (peers is not None and peers.available) else None
        self.genome_space = self.host.genome_space if genome_space is None else int(genome_space)
        self.wins = wins if wins is not None else query.windows(w, step, scaffolds_all)
        # base range of the host planes this pipeline counts (multi-GPU: a rank's slice; the last
        # 32-base word is padding, only ever read as look-ahead)
        self.bg_range = (0, host.padded_len - 32) if bg_range is None else (int(bg_range[0]), int(bg_range[1]))
        dev = self.dq.device
        self.device = dev
        n = len(self.wins)
        tsz = _lib.table_size(1, kmax)
        self.d_fwd = torch.zeros(tsz, dtype=torch.int64, device=dev)
        self.d_tables = torch.empty(tsz, dtype=torch.int64, device=dev)
        self.d_valid = torch.zeros(1, dtype=torch.int64, device=dev)
        self.d_ig = torch.empty(2 * 4 ** kmax, dtype=torch.float64, device=dev)
        self.d_rows = torch.empty((n, 5), dtype=torch.float64, device=dev)
        self.d_status = torch.empty(n, dtype=torch.int32, device=dev)
        self.d_dump = torch.empty((n, tsz), dtype=torch.int16, device=dev) if dump else None
        self.d_off = torch.from_numpy(self.wins.off.view(np.int64)).to(dev, non_blocking=True)
        self.d_len = torch.from_numpy(self.wins.length.view(np.int32)).to(dev, non_blocking=True)
        self.launches_per_step = 4          # bg_count, bg_reduce, finalize_ivom (cooperative), score_windows

    def enqueue(self, marks=None) -> None:
        """Launch one pass.  ``marks`` (optional list) receives a CUDA event after each stage:
        [start, background done, tables+IVOM done, score done]."""
        import torch
        L = _lib.lib()
        dev = self.device

        def mark():
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(torch.cuda.current_stream(dev))
                marks.append(ev)

        with torch.cuda.device(dev):
            st = _stream_ptr(dev)
            d_fwd = self.peers.local() if self.peers is not None else self.d_fwd
            mark()                           # a step includes zeroing its counters
            d_fwd.zero_()
            dh = self.dh
            _lib.check(L.frisk_b200_background(_ptr(dh.codes), _ptr(dh.inv), _ptr(dh.low), self.bg_range[0], self.bg_range[1],
                                               self.kmax, int(self.mask_host), _ptr(d_fwd), st), "frisk_b200_background")
            mark()
            space = self.genome_space
            if self.peers is not None:      # counters summed from every rank's buffer inside the (one) finalising launch
                self.peers.finalize_ivom(self.kmin, self.kmax, int(space), self.d_tables, self.d_valid, self.d_ig, st)
            else:
                if self.allreduce is not None:
                    space = self.allreduce(self.d_fwd, space)
                _lib.check(L.frisk_b200_finalize_ivom(_ptr(self.d_fwd), None, None, 0, 0, 0, self.kmin, self.kmax, int(space),
                                                      _ptr(self.d_tables), _ptr(self.d_valid), _ptr(self.d_ig), st),
                           "frisk_b200_finalize_ivom")
            mark()
            n = len(self.wins)
            if n:
                dq = self.dq
                _lib.check(L.frisk_b200_score(_ptr(dq.codes), _ptr(dq.inv), _ptr(dq.low), _ptr(self.d_off), _ptr(self.d_len),
                                              n, self.wins.max_len, _ptr(self.d_ig), self.kmin, self.kmax, int(self.rip),
                                              _ptr(self.d_rows), _ptr(self.d_status), _ptr(self.d_dump), st),
                           "frisk_b200_score")
            mark()

    def step_from_host(self, out: "HostOutputs") -> "HostOutputs":
        """One end-to-end pass without any allocation: H2D of the (pinned) host planes into the
        resident device buffers, every kernel (with the all-reduce when one is set), D2H of rows,
        status, tables and the valid-word count into ``out`` (pinned).  Returns after the stream is
        idle.  This is the multi-GPU counterpart of the single C call frisk_b200_run_host."""
        import torch
        dev = self.device
        with torch.cuda.device(dev):
            for dg in ((self.dh,) if self.dh is self.dq else (self.dh, self.dq)):
                g = dg.host
                dg.codes.copy_(torch.from_numpy(g.codes.view(np.int32)), non_blocking=True)
                dg.inv.copy_(torch.from_numpy(g.inv.view(np.int32)), non_blocking=True)
                if dg.low is not None:
                    dg.low.copy_(torch.from_numpy(g.low.view(np.int32)), non_blocking=True)
            self.d_off.copy_(torch.from_numpy(self.wins.off.view(np.int64)), non_blocking=True)
            self.d_len.copy_(torch.from_numpy(self.wins.length.view(np.int32)), non_blocking=True)
            self.enqueue()
            n = len(self.wins)
            if n:
                torch.from_numpy(out.rows[:n]).copy_(self.d_rows, non_blocking=True)
                torch.from_numpy(out.status[:n].view(np.int32)).copy_(self.d_status, non_blocking=True)
            torch.from_numpy(out.tables.view(np.int64)).copy_(self.d_tables, non_blocking=True)
            torch.from_numpy(out.valid.view(np.int64)).copy_(self.d_valid, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        return out

    def result(self, names: bool = True) -> HotPathResult:
        import torch
        torch.cuda.synchronize(self.device)
        tables = self.d_tables.cpu().numpy().view(np.uint64)
        n = len(self.wins)
        if n >= (1 << 16):                      # large row sets come back through page-locked memory (pageable: ~3 GB/s)
            h_rows = _staging("rows", (n, 5), np.float64)       # (assemble copies what it keeps)
            h_stat = _staging("status", (n,), np.int32)
            torch.from_numpy(h_rows).copy_(self.d_rows, non_blocking=True)
            torch.from_numpy(h_stat).copy_(self.d_status, non_blocking=True)
            torch.cuda.synchronize(self.device)
            rows, status = h_rows, h_stat.view(np.uint32)
        else:
            rows = self.d_rows.cpu().numpy()
            status = self.d_status.cpu().numpy().view(np.uint32)
        dmp = self.d_dump.cpu().numpy().view(np.uint16) if self.d_dump is not None else None
        return assemble(self.query, self.host, self.wins, tables, int(self.d_valid.item()), rows, status,
                        self.kmin, self.kmax, dmp, names=names)


def run(query, host=None, kmin: int = 1, kmax: int = 8, w: int = 5000,
        step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False, rip: bool = True,
        device="cuda:0", dump: bool = False, allreduce=None, genome_space: Optional[int] = None,
        wins: Optional[WindowList] = None) -> HotPathResult:
    """Stages 2+3 of the reference's main() (F:1442, F:1478-1494) on one GPU: H2D of the planes,
    one Pipeline pass, D2H of tables and rows.  ``allreduce`` (multi-GPU): see frisk_b200/dist.py;
    ``host`` is then this rank's shard and the returned tables are the global ones (meta's
    totalLen/exMax/nnTotal stay per-shard and are summed by the caller)."""
    pipe = Pipeline(query, host, kmin, kmax, w, step, mask_host, scaffolds_all, rip, device, dump, allreduce,
                    genome_space, wins)
    pipe.enqueue()
    return pipe.result()


def run_sweep(query, kmaxes: Sequence[int] = tuple(range(1, 9)), kmin: int = 1, w: int = 5000, step: int = 2500,
              mask_host: bool = False, scaffolds_all: bool = False, rip: bool = True, device="cuda:0", fused: bool = True):
    """Scores for several --maxWordSize values in one go (BASELINE config C3: the k sweep 1..8, i.e. eight
    reference runs ``-m kmin -k k'``).  The count of x-words does not depend on kmax (F:338-351 counts every
    order independently), so ONE background pass at max(kmaxes) serves every k'; per k' only the genome
    IVOM table and the window kernel run.  Returns {k': HotPathResult}."""
    import torch
    _lib.require_device()
    if fused:                                   # kmax' = 1..8, kmin 1: one window kernel for all of them
        sw = Sweep(query, kmaxes, kmin, w, step, mask_host, scaffolds_all, rip, device)
        if sw.fused:
            sw.enqueue()
            return sw.results()
        query = sw.dq
    dq = query if isinstance(query, DeviceGenome) else DeviceGenome(query, device)
    g = dq.host
    top = max(kmaxes)
    d_tables, _ = finalize(background(dq, top, mask_host), top)
    wins = g.windows(w, step, scaffolds_all)
    out = {}
    for k in sorted(set(int(x) for x in kmaxes)):
        if k < kmin:
            continue
        tsz = _lib.table_size(1, k)
        d_tab_k = d_tables[:tsz]
        d_ig = genome_ivom(d_tab_k, kmin, k, g.genome_space)
        d_rows, d_status, _ = score(dq, wins, d_ig, kmin, k, rip)
        torch.cuda.synchronize(dq.device)
        tables = d_tab_k.cpu().numpy().view(np.uint64)
        valid = int(tables[_lib.table_size(1, k - 1) if k > 1 else 0:].sum()) // 2      # both strands were added
        out[k] = assemble(g, g, wins, tables, valid, d_rows.cpu().numpy(), d_status.cpu().numpy().view(np.uint32), kmin, k)
    return out


class Sweep:
    """BASELINE config C3 as a resident, replayable object: scores for kmax' = kmaxes (kmin fixed) from ONE counting pass
    (see ``run_sweep``), every buffer allocated up front so that ``enqueue`` only launches: background at max(kmaxes),
    [all-reduce], finalise, then per k' the genome IVOM table and the window kernel.  Multi-GPU (rank / world /
    allreduce): every rank holds the whole genome, counts its slice of the base range and scores its slice of the
    window list for every k' (the scheme of dist.score_balanced)."""

    def __init__(self, query, kmaxes: Sequence[int] = tuple(range(1, 9)), kmin: int = 1, w: int = 5000, step: int = 2500,
                 mask_host: bool = False, scaffolds_all: bool = False, rip: bool = True, device="cuda:0", rank: int = 0,
                 world: int = 1, allreduce=None, fused: bool = True):
        import torch
        from . import dist as fdist
        _lib.require_device()
        self.dq = query if isinstance(query, DeviceGenome) else DeviceGenome(query, device)
        g = self.dq.host
        self.kmaxes = sorted(set(int(k) for k in kmaxes if int(k) >= kmin))
        self.kmin, self.mask_host, self.rip, self.top = kmin, mask_host, rip, max(self.kmaxes)
        self.allreduce = allreduce
        self.wins_all = g.windows(w, step, scaffolds_all)
        a, b = fdist.split_windows(self.wins_all.length, world)[rank]
        self.wins = self.wins_all.slice(a, b)
        self.bg_range = fdist.split_base_range(g.padded_len, world)[rank] if world > 1 else (0, g.padded_len - 32)
        dev = self.dq.device
        self.device = dev
        n = len(self.wins)
        tsz = _lib.table_size(1, self.top)
        self.d_fwd = torch.zeros(tsz, dtype=torch.int64, device=dev)
        self.d_tables = torch.empty(tsz, dtype=torch.int64, device=dev)
        self.d_valid = torch.zeros(1, dtype=torch.int64, device=dev)
        self.d_ig = {k: torch.empty(2 * 4 ** k, dtype=torch.float64, device=dev) for k in self.kmaxes}
        self.d_rows = {k: torch.empty((n, 5), dtype=torch.float64, device=dev) for k in self.kmaxes}
        self.d_status = {k: torch.empty(n, dtype=torch.int32, device=dev) for k in self.kmaxes}
        self.d_off = torch.from_numpy(self.wins.off.view(np.int64)).to(dev)
        self.d_len = torch.from_numpy(self.wins.length.view(np.int32)).to(dev)
        self.launches = 0
        # kmax' = 1..8 with kmin 1 and windows the shared-memory kernels hold: one fused launch (frisk_b200_score_sweep)
        self.fused = bool(fused) and self.kmaxes == list(range(1, 9)) and kmin == 1 and 0 < self.wins.max_len <= 8186
        if self.fused:
            mk = lambda ts: (C.c_void_p * 8)(*[C.c_void_p(int(ts[k].data_ptr())) for k in range(1, 9)])
            self._ig_ptrs, self._row_ptrs, self._st_ptrs = mk(self.d_ig), mk(self.d_rows), mk(self.d_status)

    def enqueue(self, marks=None) -> None:
        import torch
        L = _lib.lib()
        dev, g, dq = self.device, self.dq.host, self.dq
        n = len(self.wins)

        def mark():
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(torch.cuda.current_stream(dev))
                marks.append(ev)

        with torch.cuda.device(dev):
            st = _stream_ptr(dev)
            mark()
            self.d_fwd.zero_()
            _lib.check(L.frisk_b200_background(_ptr(dq.codes), _ptr(dq.inv), _ptr(dq.low), self.bg_range[0], self.bg_range[1], self.top,
                                               int(self.mask_host), _ptr(self.d_fwd), st), "frisk_b200_background")
            if self.allreduce is not None:
                self.allreduce(self.d_fwd, g.genome_space)
            _lib.check(L.frisk_b200_finalize_tables(_ptr(self.d_fwd), self.top, 1, _ptr(self.d_tables), _ptr(self.d_valid), st),
                       "frisk_b200_finalize_tables")
            mark()
            launches = 5                                   # count, reduce, totals, low, symmetrise
            fused = self.fused and n > 0
            for k in self.kmaxes:
                _lib.check(L.frisk_b200_genome_ivom(_ptr(self.d_tables), self.kmin, k, int(g.genome_space), _ptr(self.d_ig[k]), st),
                           "frisk_b200_genome_ivom")
                if fused:
                    launches += 1
                    continue
                if n:
                    _lib.check(L.frisk_b200_score(_ptr(dq.codes), _ptr(dq.inv), _ptr(dq.low), _ptr(self.d_off), _ptr(self.d_len), n,
                                                  self.wins.max_len, _ptr(self.d_ig[k]), self.kmin, k, int(self.rip),
                                                  _ptr(self.d_rows[k]), _ptr(self.d_status[k]), None, st), "frisk_b200_score")
                launches += 2 + (1 if k >= 7 else 0)       # kmax 7, 8: + the (usually empty) hand-over launch
                mark()
            if fused:                                      # ONE window kernel for all eight kmax' (+ eight empty hand-over launches)
                _lib.check(L.frisk_b200_score_sweep(_ptr(dq.codes), _ptr(dq.inv), _ptr(dq.low), _ptr(self.d_off), _ptr(self.d_len), n,
                                                    self.wins.max_len, self._ig_ptrs, 8, int(self.rip), self._row_ptrs, self._st_ptrs, st),
                           "frisk_b200_score_sweep")
                launches += 9
                mark()
            self.launches = launches

    def checksums(self):
        """Sum of the KLD scores of this rank's rows, per k' (N-independent after a sum over ranks)."""
        import torch
        out = []
        for k in self.kmaxes:
            ok = self.d_status[k] == 0
            kld = self.d_rows[k][:, 0]
            out.append(torch.where(ok, kld, torch.zeros_like(kld)).sum())
        return torch.stack(out)

    def results(self):
        """{k': HotPathResult} of this rank's rows (the order-k' tables are the prefix of the top-order tables)."""
        import torch
        torch.cuda.synchronize(self.device)
        g = self.dq.host
        out = {}
        for k in self.kmaxes:
            tables = self.d_tables[:_lib.table_size(1, k)].cpu().numpy().view(np.uint64)
            valid = int(tables[_lib.table_size(1, k - 1) if k > 1 else 0:].sum()) // 2      # both strands were added
            out[k] = assemble(g, g, self.wins, tables, valid, self.d_rows[k].cpu().numpy(),
                              self.d_status[k].cpu().numpy().view(np.uint32), self.kmin, k)
        return out


def run_host(query: PackedGenome, host: Optional[PackedGenome] = None, kmin: int = 1, kmax: int = 8, w: int = 5000,
             step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False, rip: bool = True,
             wins: Optional[WindowList] = None, out=None, stream: int = 0, assemble_result: bool = True,
             sparse: Optional[bool] = None):
    """Same path as ``run`` but as ONE C call from host buffers (frisk_b200_run_host): H2D of the
    planes and window list, all kernels, D2H of rows/status/tables.  Used for end-to-end timing;
    ``assemble_result=False`` returns the raw HostOutputs (rows of every candidate window, status
    flags, tables) without building the Python-side row list."""
    _lib.require_device()
    host = host or query
    if wins is None:
        wins = query.windows(w, step, scaffolds_all)
    n = len(wins)
    if out is None:
        out = HostOutputs(n, kmax)
    # ``sparse``: upload the (nearly empty) invalid planes as their non-zero words
    # (frisk_b200_run_host_sparse); None = whenever that is at most a quarter of the dense plane
    if sparse is None:
        sparse = host.prefers_sparse() and (query is host or query.prefers_sparse())
    if sparse:
        (hi, hv), (qi, qv) = host.inv_sparse(), query.inv_sparse()
        rc = _lib.lib().frisk_b200_run_host_sparse(
            _ptr(host.codes), _ptr(hi), _ptr(hv), len(hi), _ptr(host.low), host.padded_len,
            _ptr(query.codes), _ptr(qi), _ptr(qv), len(qi), _ptr(query.low), query.padded_len,
            _ptr(wins.off), _ptr(wins.length), n, wins.max_len, kmin, kmax, int(mask_host), int(rip),
            int(host.genome_space), _ptr(out.rows), _ptr(out.status), _ptr(out.tables), _ptr(out.valid), C.c_void_p(stream))
        _lib.check(rc, "frisk_b200_run_host_sparse")
    else:
        rc = _lib.lib().frisk_b200_run_host(
            _ptr(host.codes), _ptr(host.inv), _ptr(host.low), host.padded_len,
            _ptr(query.codes), _ptr(query.inv), _ptr(query.low), query.padded_len,
            _ptr(wins.off), _ptr(wins.length), n, wins.max_len, kmin, kmax, int(mask_host), int(rip),
            int(host.genome_space), _ptr(out.rows), _ptr(out.status), _ptr(out.tables), _ptr(out.valid), C.c_void_p(stream))
        _lib.check(rc, "frisk_b200_run_host")
    if not assemble_result:
        return out
    return assemble(query, host, wins, out.tables, int(out.valid[0]), out.rows[:n], out.status[:n], kmin, kmax)


def run_resident(dq: DeviceGenome, dh: Optional[DeviceGenome] = None, kmin: int = 1, kmax: int = 8, w: int = 5000,
                 step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False, rip: bool = True,
                 wins: Optional[WindowList] = None, out=None, assemble_result: bool = True):
    """``run_host`` for planes that are already on the device (frisk_b200_run_resident): one C call
    that uploads the window list, runs every kernel and downloads rows/status/tables."""
    _lib.require_device()
    dh = dh or dq
    query, host = dq.host, dh.host
    if wins is None:
        wins = query.windows(w, step, scaffolds_all)
    n = len(wins)
    native = isinstance(dq.codes, DevBuf)
    if out is None:
        out = HostOutputs(n, kmax, pinned=not native)

    def call():
        return _lib.lib().frisk_b200_run_resident(
            _ptr(dh.codes), _ptr(dh.inv), _ptr(dh.low), host.padded_len,
            _ptr(dq.codes), _ptr(dq.inv), _ptr(dq.low), query.padded_len,
            _ptr(wins.off), _ptr(wins.length), n, wins.max_len, kmin, kmax, int(mask_host), int(rip),
            int(host.genome_space), _ptr(out.rows), _ptr(out.status), _ptr(out.tables), _ptr(out.valid),
            _stream_ptr(dq.device))

    if native:
        _lib.check(_lib.lib().frisk_b200_set_device(_device_index(dq.device)), "frisk_b200_set_device")
        rc = call()
    else:
        with _device_ctx(dq.device):
            rc = call()
    _lib.check(rc, "frisk_b200_run_resident")
    if not assemble_result:
        return out
    return assemble(query, host, wins, out.tables, int(out.valid[0]), out.rows[:n], out.status[:n], kmin, kmax)


class _HandlePlane:
    """A plane that belongs to a frisk_b200_fasta handle (frisk_b200_fasta_planes): just its device address."""

    def __init__(self, ptr):
        self._p = int(ptr or 0)

    def data_ptr(self) -> int:
        return self._p


def _genome_from_handle(L, h, buf, device_text: bool = False) -> PackedGenome:
    nrec, padded = C.c_uint64(0), C.c_uint64(0)
    stats = np.zeros(3, np.uint64)
    _lib.check(L.frisk_b200_fasta_info(h, C.byref(nrec), C.byref(padded), _ptr(stats)), "frisk_b200_fasta_info")
    R = int(nrec.value)
    name_off = np.zeros(R, np.uint64); name_len = np.zeros(R, np.uint32)
    seq_len = np.zeros(R, np.uint64); scaf_off = np.zeros(R, np.uint64)
    _lib.check(L.frisk_b200_fasta_records(h, _ptr(name_off), _ptr(name_len), _ptr(seq_len), _ptr(scaf_off)),
               "frisk_b200_fasta_records")
    return PackedGenome(LazyNames(_name_source(L, h, buf, device_text), name_off, name_len), seq_len, scaf_off, int(padded.value), None, None, None,
                        int(stats[0]), int(stats[1]), int(stats[2]), False)


def run_fasta(query_text, host_text=None, device="cuda:0", out=None, assemble_result: bool = True, kmin: int = 1,
              kmax: int = 8, w: int = 5000, step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False,
              rip: bool = True):
    """FASTA text (bytes / uint8 array, ideally page-locked) in, rows out, through ONE C call (frisk_b200_run_fasta): the
    text is uploaded in chunks and tokenised, packed and counted on the device while it arrives; names and windows are
    derived on the host while the last chunk is still being counted; then tables, IVOM, window kernel, rows.  This is the
    whole of the reference's stages 2+3 (F:1442, F:1478-1494) including its three passes over the file (F:170, F:203,
    F:297).  ``out``: reusable HostOutputs (its row capacity is used; ``out.n_win`` is set)."""
    return _run_fasta_any(query_text, host_text, "text", device, out, assemble_result, kmin, kmax, w, step, mask_host,
                          scaffolds_all, rip)


def run_fasta_bgzf(query_gz, host_gz=None, device="cuda:0", out=None, assemble_result: bool = True, kmin: int = 1,
                   kmax: int = 8, w: int = 5000, step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False,
                   rip: bool = True):
    """``run_fasta`` for BGZF buffers (bgzip, samtools; ideally page-locked): ONE C call (frisk_b200_run_fasta_bgzf) that
    uploads the compressed bytes, inflates every BGZF block on the device straight into the ingest's text buffer and goes
    on exactly as ``run_fasta``.  Same results as ``run_fasta`` on the inflated text."""
    return _run_fasta_any(query_gz, host_gz, "bgzf", device, out, assemble_result, kmin, kmax, w, step, mask_host,
                          scaffolds_all, rip)


def run_fasta_gzip(query_gz, host_gz=None, device="cuda:0", out=None, assemble_result: bool = True, kmin: int = 1,
                   kmax: int = 8, w: int = 5000, step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False,
                   rip: bool = True):
    """``run_fasta`` for single gzip members (gzip, pigz): ONE C call (frisk_b200_run_fasta_gzip) that uploads the
    compressed bytes, inflates them on the device straight into the ingest's text buffer and goes on exactly as
    ``run_fasta``.  Same results as ``run_fasta`` on the inflated text; FriskError E_UNSUPPORTED for a multi-member file."""
    return _run_fasta_any(query_gz, host_gz, "gzip", device, out, assemble_result, kmin, kmax, w, step, mask_host,
                          scaffolds_all, rip)


def run_2bit(query_2bit, host_2bit=None, device="cuda:0", out=None, assemble_result: bool = True, kmin: int = 1,
             kmax: int = 8, w: int = 5000, step: int = 2500, mask_host: bool = False, scaffolds_all: bool = False,
             rip: bool = True):
    """``run_fasta`` for UCSC .2bit files (ideally page-locked): ONE C call (frisk_b200_run_2bit) that uploads the file,
    decodes it on the device straight into the planes and goes on exactly as ``run_fasta``.  Same results as
    ``run_fasta`` on the genome's FASTA."""
    return _run_fasta_any(query_2bit, host_2bit, "2bit", device, out, assemble_result, kmin, kmax, w, step, mask_host,
                          scaffolds_all, rip)


_OPENERS = {"text": "frisk_b200_fasta_open", "bgzf": "frisk_b200_fasta_open_bgzf", "gzip": "frisk_b200_fasta_open_gzip",
            "2bit": "frisk_b200_fasta_open_2bit"}
_RUNNERS = {"text": "frisk_b200_run_fasta", "bgzf": "frisk_b200_run_fasta_bgzf", "gzip": "frisk_b200_run_fasta_gzip",
            "2bit": "frisk_b200_run_2bit"}


def _text_len_hint(buf: np.ndarray, kind: str) -> int:
    """The text's length: exact for text and BGZF; for gzip, ISIZE (the length mod 2^32 -- a guess for sizing rows); for
    .2bit, the number of bases."""
    if kind == "2bit":
        return int(twobit_records(buf)[2].sum())
    if kind == "bgzf":
        return bgzf_text_len(buf)
    if kind == "gzip":
        return int.from_bytes(bytes(buf[-4:]), "little") if buf.shape[0] >= 4 else 0
    return buf.shape[0]


def _run_fasta_any(query_text, host_text, kind, device, out, assemble_result, kmin, kmax, w, step, mask_host, scaffolds_all, rip):
    import torch
    _lib.require_device()
    L = _lib.lib()
    qbuf = _as_u8(query_text)
    hbuf = _as_u8(host_text) if host_text is not None else qbuf
    dev = torch.device(device)
    if out is None:
        # rows: a guess (one window per step of text, one more per 4 KiB for short scaffolds); a text with more windows comes
        # back with FRISK_E_CAPACITY and is scored in a second stage below -- page-locking a far larger buffer "to be safe"
        # would cost more than the run (~0.3 ms per MB)
        n_text = _text_len_hint(qbuf, kind)
        out = HostOutputs(n_text // step + n_text // 4096 + 64, kmax)
    hh, qh = C.c_void_p(), C.c_void_p()
    n_win = C.c_uint64(0)
    what = _RUNNERS[kind]
    fn = getattr(L, what)
    with _device_ctx(dev):
        st = _stream_ptr(dev)
        rc = fn(_ptr(hbuf), hbuf.shape[0], _ptr(qbuf) if host_text is not None else None,
                                    qbuf.shape[0] if host_text is not None else 0, w, step, int(scaffolds_all), kmin, kmax,
                                    int(mask_host), int(rip), out.rows.shape[0], _ptr(out.rows), _ptr(out.status),
                                    _ptr(out.tables), _ptr(out.valid), C.byref(n_win), C.byref(hh), C.byref(qh), st)
        try:
            if rc not in (_lib.OK, _lib.E_CAPACITY):
                _lib.check(rc, what)
            n = int(n_win.value)
            need_genomes = assemble_result or rc == _lib.E_CAPACITY
            host = _genome_from_handle(L, hh, hbuf, kind != "text") if need_genomes else None
            query = (_genome_from_handle(L, qh, qbuf, kind != "text") if qh else host) if need_genomes else None
            if rc == _lib.E_CAPACITY:
                # more windows than the guessed row capacity: the planes are on the device, score them into enough rows
                def planes(h):
                    c, i, l = C.c_void_p(), C.c_void_p(), C.c_void_p()
                    _lib.check(L.frisk_b200_fasta_planes(h, C.byref(c), C.byref(i), C.byref(l)), "frisk_b200_fasta_planes")
                    return (_HandlePlane(c.value), _HandlePlane(i.value), _HandlePlane(l.value) if l.value else None)
                dh = DeviceGenome(host, dev, planes=planes(hh))
                dq = DeviceGenome(query, dev, planes=planes(qh)) if qh else dh
                out = HostOutputs(n, kmax)
                out = run_resident(dq, dh, kmin=kmin, kmax=kmax, w=w, step=step, mask_host=mask_host,
                                   scaffolds_all=scaffolds_all, rip=rip, out=out, assemble_result=False)
        finally:
            if qh:
                L.frisk_b200_fasta_close(qh, st)
            if hh:
                L.frisk_b200_fasta_close(hh, st)
    out.n_win = n
    if not assemble_result:
        return out
    wins = query.windows(w, step, scaffolds_all)
    assert len(wins) == n
    return assemble(query, host, wins, out.tables, int(out.valid[0]), out.rows[:n], out.status[:n], kmin, kmax)


class HostOutputs:
    """Reusable (pinned when possible) host buffers for run_host."""

    def __init__(self, n_win: int, kmax: int, pinned: bool = True):
        self.rows = _alloc((max(n_win, 1), 5), np.float64, pinned)
        self.status = _alloc((max(n_win, 1),), np.uint32, pinned)
        self.tables = _alloc((_lib.table_size(1, kmax),), np.uint64, pinned)
        self.valid = _alloc((1,), np.uint64, pinned)
