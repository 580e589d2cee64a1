"""Pack an on-disk Memdir into the device-resident corpus and keep it in sync (the one-time ingest).

Replaces the per-query walk of utils.list_memories (memdir_tools/utils.py:202-253).  Files are read once, in exactly the
reference's listing order -- folders in os.walk order (utils.py:48), statuses cur/new/tmp, inside a directory os.listdir order
stably sorted by filename timestamp, newest first (utils.py:220,251) -- and decoded like `open(path, "r")` (UTF-8 strict,
universal newlines; undecodable files are reported and skipped, utils.py:247-248).

Who does what:
  * native host code (csrc/memdir_host.cpp): readdir + file-name grammar + stat per directory, multi-threaded file reads;
  * GPU (csrc/ingest.cu, corpus.cu, hdir.cu): UTF-8 validation, newline folding, first-'---' split (utils.py:105), body .strip()
    (utils.py:120), body tiling, header directory / value columns;
  * this module: which directories changed (inotify, directory mtimes), the diff of a re-listed directory against its cached
    listing by (name, inode, size, mtime), and the bookkeeping of listing order.  Per-record state lives in numpy arrays.

Incremental sync.  The packed corpus is a BASE corpus (built once, in listing order) plus a small DELTA corpus: new or rewritten
files are read and appended to the delta (one or a few 4096-record windows re-tiled, not the shard); removed files become
tombstones; a rename -- move_memory / update_memory_flags are renames, utils.py:255-297, :354-388 -- is recognised by
(inode, size, mtime) and carried over without reading the file (its packed text moves from the device into the delta with the
new name, flags and folder).  Listing order is a permutation kept on the host: hits come back as device record ids and are
mapped to listing positions.  When the delta or the tombstones outgrow a fraction of the base, everything is repacked.
"""
from __future__ import annotations

import calendar
import ctypes as C
import errno
import os
import queue
import re
import struct
import threading
import time
from datetime import datetime
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _abi
from .memdir_tools import utils as U

REC_NO_SEPARATOR, REC_NONASCII, REC_HAS_SIGMA, REC_HAS_IDOT = 1, 2, 4, 8
_LIST_RE = re.compile(r"\d+\.[a-z0-9]+\.[^:]+:2,[A-Z]*")          # utils.py:223
MAX_BODY = 32 << 20                                                # packed layout limit per record (corpus.cu)
MAX_RAW_BATCH = 40 << 30                                           # raw bytes packed in one go
COLD_CHUNK_BYTES = 256 << 20                                        # cold pack: bytes per host chunk
COLD_SLOTS = 3                                                      # reused chunk buffers (one being read into, up to two being uploaded)
LIST_CONCURRENCY = 4                                                # directories listed at the same time in a cold pack
READ_THREADS = max(1, min(32, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)))
_KEY_DT = np.dtype([("ino", "u8"), ("size", "u8"), ("mtime", "i8")])


# ----------------------------------------------------------------------------- native directory listing
class DirListing:
    """One cur/new/tmp directory as arrays, in the reference's listing order (fei_dir_list + the entries Python must judge)."""
    __slots__ = ("n", "names", "name_off", "ts", "wall", "flags8", "spans", "ino", "size", "mtime_ns", "bad")

    def name_bytes(self, i: int) -> bytes:
        return self.names[int(self.name_off[i]):int(self.name_off[i + 1])]

    def name(self, i: int) -> str:
        return os.fsdecode(self.name_bytes(i))

    def key(self) -> np.ndarray:
        """Identity of every entry's content: a changed key means the file must be read again."""
        k = np.zeros(self.n, dtype=_KEY_DT)
        k["ino"], k["size"], k["mtime"] = self.ino, self.size, self.mtime_ns
        return k


def _arr(p, dt, k):
    if not k:
        return np.zeros(0, dtype=dt)
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(np.ctypeslib.as_ctypes_type(dt))), shape=(k,)).copy()


def list_dir(path: str, want_stat: bool = True) -> DirListing:
    """want_stat=False: names only (ino from the directory entry, size 0, mtime -1): read_dir_packed fills them from the open files."""
    l = _abi.lib()
    h = C.c_void_p()
    _abi.check((l.fei_dir_list if want_stat else l.fei_dir_list_names)(os.fsencode(path), C.byref(h)))
    try:
        v = _abi.DirlistView()
        _abi.check(l.fei_dirlist_view_get(h, C.byref(v)))
        n = int(v.n)
        name_off = _arr(v.name_off, np.uint64, n + 1)
        blob = C.string_at(v.names, int(name_off[n])) if n else b""
        status = _arr(v.status, np.uint8, n)
        nflags = _arr(v.flags_len, np.int64, n)
        cols = {"ts": _arr(v.ts, np.int64, n), "wall": _arr(v.wall, np.int64, n), "flags8": _arr(v.flags8, np.uint64, n),
                "ino": _arr(v.ino, np.uint64, n), "size": _arr(v.size, np.uint64, n), "mtime_ns": _arr(v.mtime_ns, np.int64, n)}
        spans = _arr(v.spans, np.uint16, 4 * n).reshape(-1, 4)
    finally:
        l.fei_dirlist_free(h)
    d = DirListing()
    d.bad = []
    keep = np.ones(n, dtype=bool)
    extra: List[Tuple[int, int, Dict[str, Any]]] = []                 # entries Python judged: (ts, original index, fields)
    for i in np.nonzero((status != 1) | (nflags > 7) | (cols["size"] > MAX_BODY))[0].tolist():
        keep[i] = False
        name = os.fsdecode(blob[int(name_off[i]):int(name_off[i + 1])])
        try:
            if status[i] == 1:
                raise NotImplementedError("more than 7 flag letters" if nflags[i] > 7 else "a file over 32 MiB does not fit the packed layout")
            if not _LIST_RE.match(name):                              # what the reference does for this name (utils.py:223-233)
                continue
            m = U.FILENAME_RE.match(name)
            if not m:
                raise ValueError(f"Invalid memory filename: {name}")
            ts = int(m.group(1))
            date = datetime.fromtimestamp(ts)
            st = os.stat(os.path.join(path, name))
            if len(m.group(4)) > 7 or st.st_size > MAX_BODY or not -(1 << 62) < ts < (1 << 62):
                raise NotImplementedError("beyond the packed layout (more than 7 flag letters, a file over 32 MiB or a timestamp past int64)")
            sp = [len(os.fsencode(name[:x])) for x in (m.start(2), m.end(2), m.start(3), m.end(3))]
            f8 = len(m.group(4)) << 56
            for k, ch in enumerate(m.group(4)):
                f8 |= ord(ch) << (8 * k)
            extra.append((ts, i, {"name": os.fsencode(name), "ts": ts, "wall": calendar.timegm(date.timetuple()), "flags8": f8,
                                  "spans": (sp[0], sp[1] - sp[0], sp[2], sp[3] - sp[2]), "ino": st.st_ino, "size": st.st_size, "mtime_ns": st.st_mtime_ns}))
        except Exception as e:                                        # reported like the reference reports a bad file (utils.py:247-248)
            d.bad.append(f"Error processing {name}: {e}")
    idx = np.nonzero(keep)[0]
    lens = (name_off[1:] - name_off[:-1]).astype(np.int64)
    if len(idx) == n:
        d.names, d.name_off = blob, name_off
    else:
        d.names = b"".join(blob[int(name_off[i]):int(name_off[i + 1])] for i in idx.tolist())
        d.name_off = np.zeros(len(idx) + 1, dtype=np.uint64)
        np.cumsum(lens[idx], out=d.name_off[1:])
    for k, a in cols.items():
        setattr(d, k, a[idx])
    d.spans = spans[idx]
    d.n = len(idx)
    for ts, _i, f in sorted(extra, key=lambda t: (-t[0], t[1])):       # merge the Python-judged entries at their timestamp position
        pos = int(np.searchsorted(-d.ts, -ts, side="right"))
        a = int(d.name_off[pos])
        d.names = d.names[:a] + f["name"] + d.names[a:]
        d.name_off = np.concatenate([d.name_off[:pos + 1], d.name_off[pos:] + np.uint64(len(f["name"]))])
        for k in ("ts", "wall", "flags8", "ino", "size", "mtime_ns"):
            a_ = getattr(d, k)
            setattr(d, k, np.insert(a_, pos, np.array(f[k]).astype(a_.dtype)))
        d.spans = np.insert(d.spans, pos, np.array(f["spans"], dtype=np.uint16), axis=0)
        d.n += 1
    return d


def read_range_into(path: str, d: DirListing, lo: int, hi: int, out: np.ndarray) -> bool:
    """Entries [lo, hi) of the listing read back to back into out[0 : sum(sizes)] (native threads).  False if any file could not
    be read or no longer has its listed size (the caller then takes the careful path)."""
    k = hi - lo
    if k <= 0:
        return True
    a, b = int(d.name_off[lo]), int(d.name_off[hi])
    nbuf = np.frombuffer(d.names, dtype=np.uint8)[a:b] if b > a else np.zeros(1, dtype=np.uint8)
    name_off = np.ascontiguousarray(d.name_off[lo:hi + 1] - np.uint64(a))
    sizes = d.size[lo:hi]
    off = np.zeros(k + 1, dtype=np.uint64)
    np.cumsum(sizes, out=off[1:])
    got = np.zeros(k, dtype=np.uint64); err = np.zeros(k, dtype=np.int32)
    _abi.check(_abi.lib().fei_read_files(os.fsencode(path), nbuf.ctypes.data, _abi.ptr(name_off), k, out.ctypes.data, _abi.ptr(off), READ_THREADS,
                                        _abi.ptr(got), _abi.ptr(err)))
    return not err.any() and bool((got == sizes).all())


def read_files(path: str, d: DirListing, sel: Optional[np.ndarray] = None, out: Optional[np.ndarray] = None, out_base: int = 0
               ) -> Tuple[np.ndarray, np.ndarray, List[Tuple[int, str]]]:
    """Contents of the selected entries (all when sel is None): (raw blob, offsets[k+1], [(k, error message)]).  With `out`, the
    bytes land in out[out_base : out_base + sum(sizes)] (one buffer for a whole tree, no concatenation afterwards)."""
    if sel is None:
        names, name_off, sizes = d.names, d.name_off, d.size
    else:
        sel = np.asarray(sel, dtype=np.int64)
        names = b"".join(d.name_bytes(i) for i in sel.tolist())
        name_off = np.zeros(len(sel) + 1, dtype=np.uint64)
        np.cumsum((d.name_off[1:] - d.name_off[:-1])[sel], out=name_off[1:])
        sizes = d.size[sel]
    k = len(sizes)
    off = np.zeros(k + 1, dtype=np.uint64)
    np.cumsum(sizes, out=off[1:])
    if out is None:
        raw = np.empty(max(1, int(off[k])), dtype=np.uint8)
    else:
        raw = out[out_base:out_base + max(1, int(off[k]))]
    got = np.zeros(max(1, k), dtype=np.uint64)
    err = np.zeros(max(1, k), dtype=np.int32)
    nbuf = np.frombuffer(names, dtype=np.uint8) if names else np.zeros(1, dtype=np.uint8)
    _abi.check(_abi.lib().fei_read_files(os.fsencode(path), _abi.ptr(nbuf), _abi.ptr(np.ascontiguousarray(name_off)), k, raw.ctypes.data, _abi.ptr(off),
                                        READ_THREADS, _abi.ptr(got), _abi.ptr(err)))
    problems: List[Tuple[int, str]] = []
    short = np.nonzero((err[:k] != 0) | (got[:k] != sizes))[0]
    if len(short):                                                    # shrunk or vanished between stat and read: read those again, one by one
        parts = [raw[int(off[i]):int(off[i + 1])].tobytes() for i in range(k)]
        for i in short.tolist():
            name = os.fsdecode(names[int(name_off[i]):int(name_off[i + 1])])
            try:
                with open(os.path.join(path, name), "rb") as f:
                    parts[i] = f.read()
            except OSError as e:
                parts[i] = b""
                problems.append((i, f"Error processing {name}: {e}"))
        off = np.zeros(k + 1, dtype=np.uint64)
        np.cumsum(np.fromiter(map(len, parts), dtype=np.int64, count=k), out=off[1:])
        raw = np.frombuffer(b"".join(parts), dtype=np.uint8).copy() if off[k] else np.zeros(1, dtype=np.uint8)
        if out is not None and int(off[k]) <= len(out) - out_base:      # keep the one-buffer layout when it still fits
            out[out_base:out_base + int(off[k])] = raw[:int(off[k])]
            raw = out[out_base:out_base + max(1, int(off[k]))]
    return raw, off, problems


class _Arena:
    """Address space for a cold read whose total size is not known in advance (fei_host_arena_alloc: NORESERVE, only what is read
    becomes resident).  Finished stretches are page-locked by a background thread while the next directory is being read, so the
    upload that follows runs at the pinned-memory rate."""
    BLOCK = 64 << 20                                               # = kH2DPiece of csrc/ingest.cu

    def __init__(self, cap: int):
        self.cap = cap
        p = C.c_void_p()
        _abi.check(_abi.lib().fei_host_arena_alloc(cap, 1 if os.environ.get("FEI_ARENA_THP") else 0, C.byref(p)))
        self.addr = p.value
        self.cursor = C.c_uint64(0)
        self.buf = np.ctypeslib.as_array(C.cast(self.addr, C.POINTER(C.c_uint8)), shape=(cap,))
        self._pinned: List[Tuple[int, int]] = []
        self._pin_to = 0
        self._jobs: "queue.Queue[Optional[Tuple[int, int]]]" = queue.Queue()
        self._thread = threading.Thread(target=self._pin_loop, daemon=True)
        self._thread.start()

    def _pin_loop(self):
        l = _abi.lib()
        while True:
            job = self._jobs.get()
            if job is None:
                return
            lo, hi = job
            if l.fei_host_register(self.addr + lo, hi - lo) == 0:
                self._pinned.append((lo, hi))

    def pin_finished(self, final: bool = False) -> None:
        """Everything below the cursor is final once the directory that wrote it has returned.  Registrations are whole BLOCKs at
        BLOCK-aligned offsets (the last one shorter): the upload copies BLOCK by BLOCK (fei_corpus_load_raw), and a copy must not
        straddle two registrations."""
        hi = int(self.cursor.value)
        hi = min(self.cap, -(-hi // 4096) * 4096) if final else (hi // self.BLOCK) * self.BLOCK
        if hi > self._pin_to and os.environ.get("FEI_PIN_COLD", "1") != "0":
            for lo in range(self._pin_to, hi, self.BLOCK):
                self._jobs.put((lo, min(lo + self.BLOCK, hi)))
            self._pin_to = hi
        if final:
            self._jobs.put(None)
            self._thread.join()

    def close(self) -> None:
        if self.addr is None:
            return
        if self._thread.is_alive():
            self._jobs.put(None)
            self._thread.join()
        l = _abi.lib()
        for lo, _hi in self._pinned:
            l.fei_host_unregister(self.addr + lo)
        self.buf = None
        l.fei_host_arena_free(self.addr, self.cap)
        self.addr = None


class _HostText:
    """The exact host buffer of a cold pack: an anonymous mapping advised to use huge pages (where transparent huge pages are in
    "madvise" mode a multi-GB numpy buffer is touched, and later unmapped, 4 KiB at a time: ~1 M page faults for 1 M files)."""

    def __init__(self, n: int):
        self.cap = max(1 << 21, -(-n // (1 << 21)) * (1 << 21))
        p = C.c_void_p()
        _abi.check(_abi.lib().fei_host_arena_alloc(self.cap, 0 if os.environ.get("FEI_HOST_THP", "1") == "0" else 1, C.byref(p)))
        self.addr = p.value
        self.buf = np.ctypeslib.as_array(C.cast(self.addr, C.POINTER(C.c_uint8)), shape=(self.cap,))[:max(1, n)]

    def close(self) -> None:
        if self.addr is not None:
            self.buf = None
            _abi.lib().fei_host_arena_free(self.addr, self.cap)
            self.addr = None


def read_dir_packed(path: str, d: DirListing, arena: _Arena) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Cold read of every listed entry into the arena (open + fstat + read + close: no stat pass).  Fills d.size / d.ino / d.mtime_ns
    from the open files; returns (begin, len, errno) per entry."""
    k = d.n
    begin = np.zeros(max(1, k), dtype=np.uint64); ln = np.zeros(max(1, k), dtype=np.uint64)
    ino = np.zeros(max(1, k), dtype=np.uint64); mt = np.zeros(max(1, k), dtype=np.int64); err = np.zeros(max(1, k), dtype=np.int32)
    nbuf = np.frombuffer(d.names, dtype=np.uint8) if d.names else np.zeros(1, dtype=np.uint8)
    _abi.check(_abi.lib().fei_read_dir_packed(os.fsencode(path), _abi.ptr(nbuf), _abi.ptr(np.ascontiguousarray(d.name_off)), k, arena.addr, arena.cap,
                                             C.byref(arena.cursor), MAX_BODY, READ_THREADS, _abi.ptr(begin), _abi.ptr(ln), _abi.ptr(ino), _abi.ptr(mt), _abi.ptr(err)))
    d.size, d.ino, d.mtime_ns = ln[:k].copy(), ino[:k], mt[:k]
    return begin[:k], ln[:k], err[:k]


# ----------------------------------------------------------------------------- change notification
class _Watcher:
    """inotify on every cur/new/tmp directory: a directory is dirty when something was created, deleted, renamed, or WRITTEN in
    place in it (the reference rewrites memory files in place, folders.py:575, archiver.py:591; a directory's mtime does not see
    that).  Without inotify the packer falls back to directory mtimes plus a periodic native re-listing (FEI_REVALIDATE_S)."""
    _MASK = 0x2 | 0x4 | 0x8 | 0x40 | 0x80 | 0x100 | 0x200 | 0x400 | 0x800       # MODIFY ATTRIB CLOSE_WRITE MOVED_FROM MOVED_TO CREATE DELETE DELETE_SELF MOVE_SELF
    _Q_OVERFLOW, _IGNORED = 0x4000, 0x8000

    def __init__(self):
        self.fd = -1
        self.wd_of: Dict[str, int] = {}
        self.path_of: Dict[int, str] = {}
        if os.environ.get("FEI_INOTIFY", "1") == "0":
            return
        try:
            self.libc = C.CDLL(None, use_errno=True)
            fd = self.libc.inotify_init1(0o4000 | 0o2000000)           # IN_NONBLOCK | IN_CLOEXEC
            if fd >= 0:
                self.fd = fd
        except Exception:
            self.fd = -1

    @property
    def ok(self) -> bool:
        return self.fd >= 0

    def watch(self, path: str) -> bool:
        if not self.ok:
            return False
        if path in self.wd_of:
            return True
        wd = self.libc.inotify_add_watch(self.fd, os.fsencode(path), self._MASK)
        if wd < 0:
            return False
        self.wd_of[path] = wd
        self.path_of[wd] = path
        return True

    def drain(self) -> Optional[set]:
        """Paths with events since the last call; None = 'everything may have changed' (queue overflow / no inotify)."""
        if not self.ok:
            return None
        dirty = set()
        while True:
            try:
                buf = os.read(self.fd, 1 << 16)
            except BlockingIOError:
                break
            except OSError:
                return None
            if not buf:
                break
            o = 0
            while o + 16 <= len(buf):
                wd, mask, _cookie, ln = struct.unpack_from("iIII", buf, o)
                o += 16 + ln
                if mask & self._Q_OVERFLOW:
                    return None
                p = self.path_of.get(wd)
                if p is not None:
                    dirty.add(p)
                    if mask & self._IGNORED:                           # the directory itself went away
                        self.wd_of.pop(p, None); self.path_of.pop(wd, None)
        return dirty

    def close(self) -> None:
        if self.fd >= 0:
            os.close(self.fd)
            self.fd = -1


# ----------------------------------------------------------------------------- packed tree
class _Seg:
    """Cached state of one (folder, status) directory: its listing + the device record id of every entry."""
    __slots__ = ("listing", "dev", "mtime_ns", "bad", "bad_files")      # bad_files: name -> (inode, size, mtime) of files that could not be packed


def _headers_of(text: str) -> Dict[str, str]:
    headers: Dict[str, str] = {}
    for line in text.strip().split("\n"):
        k, colon, v = line.partition(":")
        if colon:
            headers[k.strip()] = v.strip()
    return headers


def _decode_error(data: bytes) -> str:
    try:
        data.decode("utf-8")
        return "invalid UTF-8"
    except UnicodeDecodeError as e:
        return str(e)


class PackedMemdir:
    """Host bookkeeping for one packed tree: listing order as arrays + the device corpora (base + delta)."""

    def __init__(self, base: str):
        self.base = base
        self.lock = threading.RLock()                        # one request at a time syncs / plans aux columns / scans this tree
        self.folders: List[str] = []
        self.folder_ids: Dict[str, int] = {}
        self.segs: Dict[Tuple[str, str], _Seg] = {}
        self.segments: Dict[Tuple[str, str], Tuple[int, int]] = {}       # (folder, status) -> listing positions [a, b)
        self.corpus = None                                   # base corpus (device ids 0 .. n_base)
        self.delta = None                                    # delta corpus (device ids n_base ..)
        self.n_base = 0
        self.n_delta = 0
        self.delta_raw: List[bytes] = []                     # contents of the delta's records (small): the delta is re-packed as a whole
        self.n = 0                                           # listed records
        self.identity = True                                 # device id == listing position (fresh base, no delta, no tombstones)
        self.dev = np.zeros(0, dtype=np.int64)               # listing position -> device record id
        self.pos_of_dev = np.zeros(0, dtype=np.int64)        # device record id -> listing position (-1: tombstone)
        self.arrays: Dict[str, np.ndarray] = {}              # listing-order meta columns: ts, wall, flags8, fsb, rec_bits
        self.files_read = 0                                  # files whose content was read from disk by the last sync
        self.windows_packed = 0                              # 4096-record windows (re)tiled by the last sync
        self.full_packs = 0
        self.snapshot_gbs: Optional[float] = None
        self.timing: Dict[str, float] = {}               # stage times of the last full pack
        self.watcher = _Watcher()
        self.last_full_check = 0.0
        self._field_values: Dict[str, Tuple[np.ndarray, np.ndarray, List[str]]] = {}
        self.parsed_dates: Dict[str, Tuple[Any, bool]] = {}
        self._aux_next = 0
        self._key_error: Optional[BaseException] = None
        self.last_sort_info = None                           # fei_sort_info of the last device sort (sort_page)
        self._seg_index: Optional[Tuple[List[Tuple[str, str]], np.ndarray]] = None
        self._walk_cache: Optional[List[str]] = None
        self._tree_dirty = True
        self._tree_dirs: List[str] = []

    # ---- tree walk
    def _walk(self) -> List[str]:
        """get_memdir_folders (utils.py:43-57): every directory that directly contains a cur / new / tmp child, in os.walk order
        (top-down, children in scandir order).  os.walk would also list the million files inside cur / new / tmp on every call;
        a Maildir status directory without sub-directories (st_nlink == 2) cannot contain a folder and is not descended into.
        With inotify on every directory of the tree, an unchanged tree is not walked at all."""
        if self._walk_cache is not None and self.watcher.ok and not self._tree_dirty:
            return list(self._walk_cache)
        out: List[str] = []
        self._tree_dirs: List[str] = []
        ok_watch = True

        def visit(path: str, rel: str) -> None:
            nonlocal ok_watch
            try:
                with os.scandir(path) as it:
                    entries = list(it)
            except OSError:
                return
            ok_watch = self.watcher.watch(path) and ok_watch
            self._tree_dirs.append(path)
            dirs = []
            for e in entries:
                try:
                    if e.is_dir():                                       # os.walk follows symlinks for the test, not for the descent
                        dirs.append(e)
                except OSError:
                    pass
            names = {e.name for e in dirs}
            if any(st in names for st in U.STANDARD_FOLDERS):
                out.append(rel)
            for e in dirs:
                if e.is_symlink():
                    continue
                if e.name in U.STANDARD_FOLDERS and names & set(U.STANDARD_FOLDERS):
                    try:
                        if os.stat(e.path).st_nlink == 2:                # no sub-directories inside this status directory
                            continue
                    except OSError:
                        continue
                visit(e.path, e.name if rel == "" else os.path.join(rel, e.name))

        visit(self.base, "")
        if len(out) > 65535:
            raise NotImplementedError("more than 65535 folders")
        self._walk_cache = list(out) if ok_watch else None
        self._tree_dirty = False
        return out

    def _tree_dir_set(self) -> set:
        status_dirs = {self._dir(f, st) for f in self.folders for st in U.STANDARD_FOLDERS}
        return set(self._tree_dirs) - status_dirs

    def _dir(self, folder: str, st: str) -> str:
        return os.path.join(self.base, folder, st) if folder else os.path.join(self.base, st)

    def _order(self) -> List[Tuple[str, str]]:
        return [(f, st) for f in self.folders for st in U.STANDARD_FOLDERS]

    # ---- sync
    def sync(self) -> "PackedMemdir":
        """Bring the packed corpus up to date with the tree.  Cheap when nothing changed: one os.walk over the folder tree, one
        stat per cur/new/tmp directory and a drain of the inotify queue."""
        with self.lock:
            dirty_paths = self.watcher.drain()
            if dirty_paths is None or any(p in self._tree_dir_set() for p in dirty_paths):
                self._tree_dirty = True                                # a directory was created / removed / renamed somewhere in the folder tree
            folders = self._walk()
            now = time.monotonic()
            recheck = float(os.environ.get("FEI_REVALIDATE_S", "1.0"))
            full_check = self.corpus is None or (dirty_paths is None and now - self.last_full_check >= recheck)
            changed: List[Tuple[str, str]] = []
            for folder in folders:
                for st in U.STANDARD_FOLDERS:
                    path = self._dir(folder, st)
                    seg = self.segs.get((folder, st))
                    isdir = os.path.isdir(path)
                    watched = self.watcher.watch(path) if isdir else True
                    try:
                        mt = os.stat(path).st_mtime_ns
                    except OSError:
                        mt = -1
                    if (seg is None or seg.mtime_ns != mt or full_check or (dirty_paths is not None and path in dirty_paths)
                            or (isdir and not watched and now - self.last_full_check >= recheck)):
                        changed.append((folder, st))
            if full_check or changed:
                self.last_full_check = now
            if self.corpus is None:
                self._full_pack(folders)
            elif folders != self.folders or changed:
                self._set_folders(folders)
                self._incremental(changed)
            return self

    def _list(self, folder: str, st: str, want_stat: bool = True) -> Tuple[DirListing, int]:
        path = self._dir(folder, st)
        try:
            mt = os.stat(path).st_mtime_ns
        except OSError:
            mt = -1
        return list_dir(path, want_stat), mt

    def _fsb_of(self, key: Tuple[str, str]) -> int:
        return (self.folder_ids[key[0]] & 0xFFFF) | (U.STANDARD_FOLDERS.index(key[1]) << 16)

    def _set_folders(self, folders: List[str]) -> None:
        """The folder list in os.walk order (= listing order); packed folder ids are handed out once and never change, so records
        already on the device keep theirs when folders appear or disappear."""
        for f in folders:
            if f not in self.folder_ids:
                self.folder_ids[f] = len(self.folder_ids)
        if len(self.folder_ids) > 65535:
            raise NotImplementedError("more than 65535 folders")
        gone = [k for k in self.segs if k[0] not in folders]
        for key in gone:                                               # a folder that vanished: its records become tombstones
            del self.segs[key]
        self.folders = folders

    def _full_pack(self, folders: List[str]) -> None:
        from .corpus import Corpus
        self.folder_ids = {}
        self._set_folders(folders)
        order = self._order()
        segs: Dict[Tuple[str, str], _Seg] = {}
        arena: Optional[_Arena] = None
        if os.environ.get("FEI_COLD_ARENA", "0") == "1":              # opt-in: measured slower than the stat listing on the bench box (DESIGN.md 2.3)
            try:
                arena = _Arena(MAX_RAW_BATCH + (1 << 30))
            except _abi.FeiError:
                arena = None                                           # no address space to spare: list with sizes, read into an exact buffer
        corpus = Corpus()
        try:
            staged = False
            if arena is not None:
                raw, begin, ln, err = self._cold_read_packed(order, segs, arena)
            else:
                raw, begin, ln, err, staged = self._cold_read_listed(order, segs, corpus)
            n = len(begin)
            self.files_read = n
            t2 = time.perf_counter()
            keep = err == 0
            pos = 0
            for key in order:                                          # files that could not be read: reported and skipped (utils.py:247-248)
                seg = segs[key]; L = seg.listing
                for i in np.nonzero(err[pos:pos + L.n])[0].tolist():
                    e = int(err[pos + i])
                    why = "a file over 32 MiB does not fit the packed layout" if e == errno.EFBIG else str(OSError(e, os.strerror(e), os.path.join(self._dir(*key), L.name(i))))
                    seg.bad.append(f"Error processing {L.name(i)}: {why}")
                pos += L.n
            while True:
                ta = time.perf_counter()
                arrays = self._raw_arrays(segs, order, keep, raw, begin, ln)
                if staged:
                    arrays["raw"] = None                               # every directory's bytes went up while the next one was being read
                tb = time.perf_counter()
                valid = corpus.load_raw(arrays)
                stage_times = {"pack_host_arrays_s": tb - ta, "pack_load_raw_call_s": time.perf_counter() - tb}
                if valid.all():
                    break
                alive = np.nonzero(keep)[0]
                staged = staged and raw is None                        # with a host buffer the second attempt uploads from it; without, the staged text stays
                for j in alive[~valid].tolist():                       # undecodable files: reported and skipped (utils.py:247-248)
                    keep[j] = False
                    key, i = self._locate(segs, order, j)
                    L = segs[key].listing
                    if raw is not None:
                        blob = raw[int(begin[j]):int(begin[j] + ln[j])].tobytes()
                    else:                                              # the text only exists on the device: read this one file again for the message
                        try:
                            with open(os.path.join(self._dir(*key), L.name(i)), "rb") as f:
                                blob = f.read()
                        except OSError:
                            blob = b"\xff"
                    segs[key].bad.append(f"Error processing {L.name(i)}: {_decode_error(blob)}")
                    segs[key].bad_files[L.name_bytes(i)] = (int(L.ino[i]), int(L.size[i]), int(L.mtime_ns[i]))
            raw_bytes = int(ln.sum())
        finally:
            tf = time.perf_counter()
            raw = None
            if arena is not None:
                arena.close()
            if getattr(self, "_host_text", None) is not None:                 # unmapping ~1 M touched 4 KiB pages takes ~0.5 s: off the query's path
                threading.Thread(target=self._host_text.close, daemon=True).start()
                self._host_text = None
            free_s = time.perf_counter() - tf
        pos = start = 0
        for key in order:                                              # drop the skipped entries from the listings; device id = listing position
            seg = segs[key]
            k = seg.listing.n
            sel = keep[start:start + k]
            if not sel.all():
                seg.listing = _subset(seg.listing, np.nonzero(sel)[0])
            seg.dev = np.arange(pos, pos + seg.listing.n, dtype=np.int64)
            pos += seg.listing.n
            start += k
        old, old_delta = self.corpus, self.delta
        self.segs = segs
        self.corpus, self.delta, self.n_base, self.n_delta = corpus, None, corpus.n, 0
        self.delta_raw = []
        self.windows_packed = (corpus.n + 4095) // 4096
        self.full_packs += 1
        t3 = time.perf_counter()
        self._rebuild_listing()
        self.timing.update({"pack_s": t3 - t2, "listing_arrays_s": time.perf_counter() - t3, "files": n, "raw_bytes": raw_bytes})
        self.timing.update(stage_times)
        self.timing["free_host_text_s"] = free_s
        try:
            st = np.zeros(3, dtype=np.float32)
            _abi.check(_abi.lib().fei_corpus_last_load_timing(corpus.handle, _abi.ptr(st)))
            self.timing.update({"device_text_h2d_ms": float(st[0]), "device_pack_kernels_ms": float(st[1])})
        except _abi.FeiError:
            pass
        for c in (old, old_delta):
            if c is not None:
                c.close()

    def _cold_read_packed(self, order, segs, arena: "_Arena"):
        """Names-only listing + open/fstat/read/close into the arena: no stat pass (see fei_read_dir_packed)."""
        t_list = t_read = 0.0
        begins, lens, errs = [], [], []
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(1) as ex:                              # the next directory is listed while this one is being read
            fut = ex.submit(self._list, *order[0], want_stat=False) if order else None
            for k, key in enumerate(order):
                t = time.perf_counter()
                listing, mt = fut.result()
                fut = ex.submit(self._list, *order[k + 1], want_stat=False) if k + 1 < len(order) else None
                seg = _Seg(); seg.listing = listing; seg.mtime_ns = mt; seg.bad = list(listing.bad); seg.bad_files = {}; seg.dev = np.zeros(listing.n, dtype=np.int64)
                segs[key] = seg
                t1 = time.perf_counter(); t_list += t1 - t
                if listing.n:
                    b, l, e = read_dir_packed(self._dir(*key), listing, arena)
                    arena.pin_finished()
                    begins.append(b); lens.append(l); errs.append(e)
                t_read += time.perf_counter() - t1
        total = int(arena.cursor.value)
        if total > MAX_RAW_BATCH:
            raise NotImplementedError("tree larger than one packing batch; shard it over several corpora")
        t = time.perf_counter()
        arena.pin_finished(final=True)
        cat = lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dtype=dt)
        self.timing = {"list_s": t_list, "read_s": t_read, "pin_tail_s": time.perf_counter() - t, "cold_path": "names-only listing (of the next directory, under the current read), open+fstat+read+close into an arena; list_s = listing time not hidden"}
        return arena.buf[:max(1, total)], cat(begins, np.uint64), cat(lens, np.uint64), cat(errs, np.int32)

    def _cold_read_listed(self, order, segs, corpus=None):
        """The default cold read: a listing with a stat of every entry (sizes known), then the files are read CHUNK by CHUNK into a
        few reused host buffers; a side thread sends each finished chunk to its place in the device text (fei_corpus_stage_text, a
        pageable copy) while the next chunk is being read.  The host never holds the whole text: ~1 GB of pages are touched (and
        unmapped) instead of one page per file.  Any surprise (a file that vanished or changed size since it was listed) falls back
        to the one-buffer path below."""
        t0 = time.perf_counter()
        total = 0
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max(1, min(LIST_CONCURRENCY, len(order)))) as ex:   # 1. list every directory (readdir + parallel stat, native):
            listed = list(ex.map(lambda k: self._list(*k), order))                  #    readdir is serial per directory, so several at a time
        for key, (listing, mt) in zip(order, listed):
            seg = _Seg(); seg.listing = listing; seg.mtime_ns = mt; seg.bad = list(listing.bad); seg.bad_files = {}; seg.dev = np.zeros(listing.n, dtype=np.int64)
            segs[key] = seg
            total += int(listing.size.sum())
        if total > MAX_RAW_BATCH:
            raise NotImplementedError("tree larger than one packing batch; shard it over several corpora")
        t1 = time.perf_counter()
        n = sum(segs[k].listing.n for k in order)
        if corpus is not None and total > 0 and os.environ.get("FEI_STAGE_UPLOAD", "1") != "0" and os.environ.get("FEI_COLD_CHUNKS", "1") != "0":
            got = self._cold_read_chunked(order, segs, corpus, n, total)
            if got is not None:
                self.timing.update({"list_s": t1 - t0})
                return got
        return self._cold_read_one_buffer(order, segs, corpus, n, total, t0, t1)

    def _cold_read_chunked(self, order, segs, corpus, n: int, total: int):
        t1 = time.perf_counter()
        slots: List[_HostText] = []
        try:
            for _ in range(COLD_SLOTS):
                slots.append(_HostText(COLD_CHUNK_BYTES + MAX_BODY))
        except _abi.FeiError:
            for sl in slots:
                sl.close()
            return None
        free: "queue.Queue[int]" = queue.Queue()
        for k in range(COLD_SLOTS):
            free.put(k)
        jobs: "queue.Queue[Optional[Tuple[int, int, int]]]" = queue.Queue()
        failed: List[BaseException] = []

        def uploader():
            while True:
                job = jobs.get()
                if job is None:
                    return
                slot, offset, nbytes = job
                if not failed:
                    try:
                        corpus.stage_text(total, slots[slot].buf[:nbytes], offset)     # returns once the pageable source has been consumed
                    except BaseException as e:                          # noqa: BLE001 -- the caller falls back to the one-buffer path
                        failed.append(e)
                free.put(slot)
        th = threading.Thread(target=uploader, daemon=True)
        th.start()
        ok = True
        base_off = 0
        sizes_all = []
        try:
            for key in order:
                L = segs[key].listing
                if not L.n:
                    continue
                sizes_all.append(L.size)
                cs = np.zeros(L.n + 1, dtype=np.int64)
                np.cumsum(L.size.astype(np.int64), out=cs[1:])
                lo = 0
                while lo < L.n and ok and not failed:
                    hi = int(np.searchsorted(cs, cs[lo] + COLD_CHUNK_BYTES, side="right")) - 1
                    hi = min(L.n, max(hi, lo + 1))
                    slot = free.get()
                    nbytes = int(cs[hi] - cs[lo])
                    ok = read_range_into(self._dir(*key), L, lo, hi, slots[slot].buf)
                    if not ok:
                        free.put(slot)
                        break
                    jobs.put((slot, base_off + int(cs[lo]), nbytes))
                    lo = hi
                if not ok or failed:
                    break
                base_off += int(cs[L.n])
        finally:
            t_reads_done = time.perf_counter()
            jobs.put(None)
            th.join()
            tf = time.perf_counter()
            for sl in slots:
                sl.close()
            t_freed = time.perf_counter()
        if not ok or failed or base_off != total:
            return None
        sizes = np.concatenate(sizes_all).astype(np.uint64) if sizes_all else np.zeros(0, dtype=np.uint64)
        begin = np.zeros(n, dtype=np.uint64)
        if n > 1:
            np.cumsum(sizes[:-1], out=begin[1:])
        self._cold_total = total
        self.timing = {"read_s": t_reads_done - t1, "upload_tail_s": tf - t_reads_done, "free_chunk_buffers_s": t_freed - tf,
                       "cold_path": "listing with stat; files read in %d MiB chunks into %d reused host buffers, each chunk uploaded under the next read" % (COLD_CHUNK_BYTES >> 20, COLD_SLOTS)}
        return None, begin, sizes, np.zeros(n, dtype=np.int32), True

    def _cold_read_one_buffer(self, order, segs, corpus, n: int, total: int, t0: float, t1: float):
        """Reads into one exact buffer (the careful path: per-file re-reads when something changed under the listing)."""
        try:
            self._host_text = _HostText(total)
            raw = self._host_text.buf                                  # 2. read every file into ONE buffer (native threads), directory by directory
        except _abi.FeiError:
            self._host_text = None
            raw = np.empty(max(1, total), dtype=np.uint8)
        raw_off = np.zeros(n + 1, dtype=np.uint64)
        pos = base_off = 0
        exact = True
        stage = corpus is not None and total > 0 and os.environ.get("FEI_STAGE_UPLOAD", "1") != "0"
        jobs: "queue.Queue[Optional[Tuple[int, int]]]" = queue.Queue()
        failed: List[BaseException] = []

        def uploader():
            while True:
                job = jobs.get()
                if job is None:
                    return
                if not failed:
                    try:
                        corpus.stage_text(total, raw[job[0]:job[1]], job[0])
                    except BaseException as e:                          # noqa: BLE001 -- reported by falling back to the plain upload
                        failed.append(e)
        th = threading.Thread(target=uploader, daemon=True) if stage else None
        if th:
            th.start()
        try:
            for key in order:
                L = segs[key].listing
                if not L.n:
                    continue
                r, off, problems = read_files(self._dir(*key), L, out=raw if exact else None, out_base=base_off)
                segs[key].bad.extend(msg for _i, msg in problems)
                if exact and r.base is not raw and r is not raw and int(off[-1]) and not np.shares_memory(r, raw):
                    exact = False                                      # a file changed size under us: fall back to pieces
                    pieces = [raw[:base_off].copy()]
                if not exact:
                    pieces.append(r[:int(off[-1])].copy())
                elif th:
                    jobs.put((base_off, base_off + int(off[-1])))
                raw_off[pos + 1:pos + L.n + 1] = off[1:] + np.uint64(base_off)
                pos += L.n; base_off += int(off[-1])
        finally:
            t_reads_done = time.perf_counter()
            if th:
                jobs.put(None)
                th.join()
        if not exact:
            raw = np.concatenate(pieces) if pieces else np.zeros(1, dtype=np.uint8)
        staged = bool(th) and exact and not failed and base_off == total
        self.timing = {"list_s": t1 - t0, "read_s": t_reads_done - t1, "upload_tail_s": time.perf_counter() - t_reads_done,
                       "cold_path": "listing with stat, reads into one exact buffer" + (", each directory uploaded under the next read" if staged else "")}
        return raw, raw_off[:-1].copy(), (raw_off[1:] - raw_off[:-1]), np.zeros(n, dtype=np.int32), staged

    @staticmethod
    def _locate(segs, order, j):
        for key in order:
            k = segs[key].listing.n
            if j < k:
                return key, j
            j -= k
        raise IndexError(j)

    def _raw_arrays(self, segs, order, keep, raw, begin, ln) -> Dict[str, Any]:
        cols: Dict[str, List[np.ndarray]] = {k: [] for k in ("ts", "wall", "flags8", "spans", "fsb")}
        names, lens = [], []
        for key in order:
            L = segs[key].listing
            if not L.n:
                continue
            cols["ts"].append(L.ts); cols["wall"].append(L.wall); cols["flags8"].append(L.flags8); cols["spans"].append(L.spans)
            cols["fsb"].append(np.full(L.n, self._fsb_of(key), dtype=np.uint32))
            names.append(L.names); lens.append((L.name_off[1:] - L.name_off[:-1]).astype(np.int64))
        n_all = len(keep)
        cat = lambda k, dt: (np.concatenate(cols[k]) if cols[k] else np.zeros(0, dtype=dt))
        ts, wall, f8, fsb = cat("ts", np.int64), cat("wall", np.int64), cat("flags8", np.uint64), cat("fsb", np.uint32)
        spans = np.concatenate(cols["spans"]) if cols["spans"] else np.zeros((0, 4), dtype=np.uint16)
        nlen = np.concatenate(lens) if lens else np.zeros(0, dtype=np.int64)
        nblob = b"".join(names)
        if keep.all():
            sel_begin, sel_len = begin, ln
            name = np.frombuffer(nblob, dtype=np.uint8).copy() if nblob else np.zeros(1, dtype=np.uint8)
            name_off = np.zeros(n_all + 1, dtype=np.uint64); np.cumsum(nlen, out=name_off[1:])
        else:
            idx = np.nonzero(keep)[0]
            noff = np.zeros(n_all + 1, dtype=np.int64); np.cumsum(nlen, out=noff[1:])
            sel_begin, sel_len = begin[idx], ln[idx]
            nm = b"".join(nblob[int(noff[j]):int(noff[j + 1])] for j in idx.tolist())
            name = np.frombuffer(nm, dtype=np.uint8).copy() if nm else np.zeros(1, dtype=np.uint8)
            name_off = np.zeros(len(idx) + 1, dtype=np.uint64); np.cumsum(nlen[idx], out=name_off[1:])
            ts, wall, f8, fsb, spans = ts[idx], wall[idx], f8[idx], fsb[idx], spans[idx]
        n = len(ts)
        return {"n": n, "global_base": 0, "raw": raw, "raw_bytes": len(raw) if raw is not None else int(self._cold_total), "raw_begin": np.ascontiguousarray(sel_begin, dtype=np.uint64),
                "raw_len": np.ascontiguousarray(sel_len, dtype=np.uint64), "name": name if n else None,
                "name_off": name_off if n else None, "name_spans": np.ascontiguousarray(spans.reshape(-1)) if n else None,
                "ts": np.ascontiguousarray(ts), "wall": np.ascontiguousarray(wall), "flags8": np.ascontiguousarray(f8), "fsb": np.ascontiguousarray(fsb)}

    # ---- incremental
    def _incremental(self, changed: List[Tuple[str, str]]) -> None:
        """Re-list the changed directories, diff them against their cached listings, and apply the difference to the device."""
        fresh: Dict[Tuple[str, str], _Seg] = {}
        rem_dev: List[int] = []
        rem_key: List[Tuple[int, int, int]] = []
        new_entries: List[Tuple[Tuple[str, str], np.ndarray]] = []
        any_change = False
        if len(changed) > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(min(LIST_CONCURRENCY, len(changed))) as ex:
                listed = list(ex.map(lambda k: self._list(*k), changed))
        else:
            listed = [self._list(*k) for k in changed]
        for key, (listing, mt) in zip(changed, listed):
            old = self.segs.get(key)
            seg = _Seg(); seg.listing = listing; seg.mtime_ns = mt; seg.bad = list(listing.bad); seg.bad_files = {}; seg.dev = np.full(listing.n, -1, dtype=np.int64)
            fresh[key] = seg
            if (old is not None and old.listing.n == listing.n and old.listing.names == listing.names
                    and np.array_equal(old.listing.key(), listing.key())):
                seg.dev = old.dev                                      # same names, same (inode, size, mtime): nothing to do here
                if old.bad:
                    seg.bad.extend(m for m in old.bad if m not in seg.bad and self._bad_still_there(key, m, listing))
            elif old is not None and old.listing.n:
                old_names = {old.listing.name_bytes(i): i for i in range(old.listing.n)}
                ok_, nk_ = old.listing.key(), listing.key()
                used = np.zeros(old.listing.n, dtype=bool)
                for i in range(listing.n):                             # same name + same (inode, size, mtime) = same packed record
                    j = old_names.get(listing.name_bytes(i))
                    if j is not None and ok_[j] == nk_[i]:
                        seg.dev[i] = old.dev[j]; used[j] = True
                for i in np.nonzero(seg.dev < 0)[0].tolist():          # a file already known to be unpackable, unchanged: stays out, stays reported
                    nb = listing.name_bytes(i)
                    if old.bad_files.get(nb) == (int(nk_[i]["ino"]), int(nk_[i]["size"]), int(nk_[i]["mtime"])):
                        seg.dev[i] = -2; seg.bad_files[nb] = old.bad_files[nb]
                for j in np.nonzero(~used)[0].tolist():
                    rem_dev.append(int(old.dev[j])); rem_key.append((int(ok_[j]["ino"]), int(ok_[j]["size"]), int(ok_[j]["mtime"])))
                if old.bad:                                            # undecodable files that did not change stay reported without being read again
                    seg.bad.extend(m for m in old.bad if m not in seg.bad and self._bad_still_there(key, m, listing))
                if not used.all() or (seg.dev == -1).any() or not np.array_equal(old.dev, seg.dev[seg.dev != -2]):
                    any_change = True
            elif listing.n:
                any_change = True
            todo = np.nonzero(seg.dev == -1)[0]
            if len(todo):
                new_entries.append((key, todo))
        if not any_change:                                             # only directory timestamps moved (or empty directories appeared)
            for key, seg in fresh.items():
                if key in self.segs:
                    self.segs[key].mtime_ns = seg.mtime_ns
                    self.segs[key].bad = seg.bad
                else:
                    if (seg.dev < 0).any():
                        sel = np.nonzero(seg.dev >= 0)[0]
                        seg.listing = _subset(seg.listing, sel); seg.dev = seg.dev[sel]
                    self.segs[key] = seg
            self.files_read = 0
            self.windows_packed = 0
            if list(self.segments) != self._order() or self.n != sum(s_.listing.n for s_ in self.segs.values()):
                self._rebuild_listing()                                # the folder set changed
            return
        # renames: a new entry whose (inode, size, mtime) equals a removed record's is that record under a new name (move_memory /
        # update_memory_flags, utils.py:255-297, :354-388): its packed text is taken from the device, the file is not read
        rem_map = {k: d for k, d in zip(rem_key, rem_dev) if d >= 0}
        moved_from: List[int] = []
        moved_to: List[Tuple[Tuple[str, str], int]] = []
        to_read: List[Tuple[Tuple[str, str], np.ndarray]] = []
        for key, todo in new_entries:
            L = fresh[key].listing
            nk_ = L.key()
            still = []
            for i in todo.tolist():
                d = rem_map.pop((int(nk_[i]["ino"]), int(nk_[i]["size"]), int(nk_[i]["mtime"])), None)
                if d is not None:
                    moved_from.append(d); moved_to.append((key, i))
                else:
                    still.append(i)
            if still:
                to_read.append((key, np.array(still, dtype=np.int64)))
        # contents of the delta after this sync: surviving delta records + moved records + newly read files
        seg_of = lambda key: fresh.get(key) or self.segs[key]
        raws: List[bytes] = []
        metas: List[Tuple] = []
        place: List[Tuple[Tuple[str, str], int]] = []                  # where each delta record is listed
        for key in self._order():
            seg = fresh.get(key) or self.segs.get(key)
            if seg is None:
                continue
            for i in np.nonzero(seg.dev >= self.n_base)[0].tolist():   # records already in the delta keep their text
                raws.append(self.delta_raw[int(seg.dev[i]) - self.n_base]); metas.append(self._meta_of(seg.listing, i, key)); place.append((key, i))
        if moved_from:
            for (key, i), text in zip(moved_to, self._device_texts(np.array(moved_from, dtype=np.int64))):
                raws.append(text); metas.append(self._meta_of(fresh[key].listing, i, key)); place.append((key, i))
        files = 0
        for key, sel in to_read:
            L = fresh[key].listing
            raw, off, problems = read_files(self._dir(*key), L, sel)
            bad_k = {k for k, _m in problems}
            fresh[key].bad.extend(m for _k, m in problems)
            for k, i in enumerate(sel.tolist()):
                if k in bad_k:
                    fresh[key].dev[i] = -2
                    continue
                raws.append(raw[int(off[k]):int(off[k + 1])].tobytes()); metas.append(self._meta_of(L, i, key)); place.append((key, i))
                files += 1
        self.files_read = files
        delta, keep = self._pack_delta(raws, metas)                    # validates the new files; undecodable ones are reported and dropped
        kept = []
        for j, ok in enumerate(keep):
            key, i = place[j]
            seg = seg_of(key)
            if ok:
                seg.dev[i] = self.n_base + len(kept)
                kept.append(j)
            else:
                seg.bad.append(f"Error processing {seg.listing.name(i)}: {_decode_error(raws[j])}")
                seg.bad_files[seg.listing.name_bytes(i)] = (int(seg.listing.ino[i]), int(seg.listing.size[i]), int(seg.listing.mtime_ns[i]))
                seg.dev[i] = -2
        for key in self._order():                                      # entries that could not be packed leave the listing
            seg = fresh.get(key) or self.segs.get(key)
            if seg is not None and (seg.dev < 0).any():
                sel = np.nonzero(seg.dev >= 0)[0]
                seg.listing = _subset(seg.listing, sel); seg.dev = seg.dev[sel]
            if key in fresh:
                self.segs[key] = fresh[key]
        old_delta = self.delta
        self.delta, self.n_delta = delta, (delta.n if delta is not None else 0)
        self.delta_raw = [raws[j] for j in kept]
        self.windows_packed = (self.n_delta + 4095) // 4096
        if old_delta is not None:
            old_delta.close()
        self._rebuild_listing()
        n_dead = self.n_base - int((self.dev < self.n_base).sum())
        if self.n_delta > max(8192, self.n_base // 16) or n_dead > max(8192, self.n_base // 4):
            self._full_pack(self.folders)                              # the delta / the tombstones outgrew their welcome: repack

    def _bad_still_there(self, key, msg: str, listing: DirListing) -> bool:
        m = re.match(r"Error processing (.*?): ", msg)
        return bool(m) and os.path.exists(os.path.join(self._dir(*key), m.group(1)))

    def _meta_of(self, L: DirListing, i: int, key) -> Tuple:
        return (L.name_bytes(i), int(L.ts[i]), int(L.wall[i]), int(L.flags8[i]), tuple(int(x) for x in L.spans[i]), self._fsb_of(key))

    def _device_texts(self, dev: np.ndarray) -> List[bytes]:
        """The packed text of device records as file contents that pack to the same record again (header + '---' + body)."""
        out: List[bytes] = [b""] * len(dev)
        for corpus, lo in self._corpora():
            sel = np.nonzero((dev >= lo) & (dev < lo + corpus.n))[0]
            if not len(sel):
                continue
            hdr, ho, body, bo = corpus.fetch_records(dev[sel] - lo)
            bits = corpus.fetch_meta()["fsb"] >> 24
            for k, j in enumerate(sel.tolist()):
                h, b = hdr[int(ho[k]):int(ho[k + 1])], body[int(bo[k]):int(bo[k + 1])]
                out[j] = b if int(bits[int(dev[j]) - lo]) & REC_NO_SEPARATOR else h + b"---" + b
        return out

    def _pack_delta(self, raws: List[bytes], metas: List[Tuple]):
        from .corpus import Corpus
        keep = [True] * len(raws)
        delta = None
        while any(keep):
            idx = [j for j, k in enumerate(keep) if k]
            off = np.zeros(len(idx) + 1, dtype=np.uint64)
            np.cumsum([len(raws[j]) for j in idx], out=off[1:])
            raw = np.frombuffer(b"".join(raws[j] for j in idx), dtype=np.uint8).copy() if off[-1] else np.zeros(1, dtype=np.uint8)
            names = [metas[j][0] for j in idx]
            name_off = np.zeros(len(idx) + 1, dtype=np.uint64); np.cumsum([len(x) for x in names], out=name_off[1:])
            arrays = {"n": len(idx), "global_base": 0, "raw": raw, "raw_off": off,
                      "name": np.frombuffer(b"".join(names), dtype=np.uint8).copy(), "name_off": name_off,
                      "name_spans": np.array([metas[j][4] for j in idx], dtype=np.uint16).reshape(-1),
                      "ts": np.array([metas[j][1] for j in idx], dtype=np.int64), "wall": np.array([metas[j][2] for j in idx], dtype=np.int64),
                      "flags8": np.array([metas[j][3] for j in idx], dtype=np.uint64), "fsb": np.array([metas[j][5] for j in idx], dtype=np.uint32)}
            if delta is None:
                delta = Corpus()
            valid = delta.load_raw(arrays)
            if valid.all():
                return delta, keep
            for j, ok in zip(idx, valid.tolist()):
                if not ok:
                    keep[j] = False
        if delta is not None:
            delta.close()
        return None, keep

    # ---- listing order
    def _rebuild_listing(self) -> None:
        self.segments = {}
        pos = 0
        devs: List[np.ndarray] = []
        cols: Dict[str, List[np.ndarray]] = {k: [] for k in ("ts", "wall", "flags8", "fsb")}
        for key in self._order():
            seg = self.segs[key]
            k = seg.listing.n
            self.segments[key] = (pos, pos + k)
            pos += k
            if k:
                devs.append(seg.dev)
                cols["ts"].append(seg.listing.ts); cols["wall"].append(seg.listing.wall); cols["flags8"].append(seg.listing.flags8)
                cols["fsb"].append(np.full(k, self._fsb_of(key), dtype=np.uint32))
        self.n = pos
        self.dev = np.concatenate(devs) if devs else np.zeros(0, dtype=np.int64)
        self.pos_of_dev = np.full(self.n_base + self.n_delta, -1, dtype=np.int64)
        self.pos_of_dev[self.dev] = np.arange(self.n, dtype=np.int64)
        self.identity = self.n == self.n_base and self.n_delta == 0 and bool((self.dev == np.arange(self.n)).all())
        dts = {"ts": np.int64, "wall": np.int64, "flags8": np.uint64, "fsb": np.uint32}
        self.arrays = {k: (np.concatenate(v) if v else np.zeros(0, dtype=dts[k])) for k, v in cols.items()}
        bits = np.zeros(self.n_base + self.n_delta, dtype=np.uint8)
        for corpus, lo in self._corpora():
            if corpus.n:
                bits[lo:lo + corpus.n] = (corpus.fetch_meta()["fsb"] >> 24).astype(np.uint8)
        self.arrays["rec_bits"] = bits[self.dev] if self.n else np.zeros(0, dtype=np.uint8)
        if self.n:
            self.arrays["fsb"] = self.arrays["fsb"] | (self.arrays["rec_bits"].astype(np.uint32) << 24)
        self._field_values = {}
        self._seg_index = None

    @property
    def bad(self) -> Dict[Tuple[str, str], List[str]]:
        return {k: s.bad for k, s in self.segs.items() if s.bad}

    # ---- scanning in listing order
    def _corpora(self):
        out = []
        if self.corpus is not None:
            out.append((self.corpus, 0))
        if self.delta is not None and self.delta.n:
            out.append((self.delta, self.n_base))
        return out

    def scan_hits(self, prog: bytes, nq: int) -> List[np.ndarray]:
        """Per query, the listing positions of the hits, ascending (= the reference's result order inside the tree)."""
        per: List[List[np.ndarray]] = [[] for _ in range(nq)]
        for corpus, lo in self._corpora():
            for q, h in enumerate(corpus.scan_hits(prog, nq)):
                per[q].append(h.astype(np.int64) + lo)
        out = []
        for q in range(nq):
            ids = np.concatenate(per[q]) if per[q] else np.zeros(0, dtype=np.int64)
            if not self.identity:
                ids = self.pos_of_dev[ids]
                ids = ids[ids >= 0]
                ids.sort()
            out.append(ids)
        return out

    def scan_masks(self, prog: bytes) -> np.ndarray:
        """mask[p] bit q = the record at listing position p satisfies query q."""
        if self.identity:
            return self.corpus.scan_masks(prog)
        dev_masks = np.zeros(self.n_base + self.n_delta, dtype=np.uint32)
        for corpus, lo in self._corpora():
            dev_masks[lo:lo + corpus.n] = corpus.scan_masks(prog)
        return dev_masks[self.dev]

    def compact(self) -> None:
        """Fold delta and tombstones back into one base corpus in listing order (whole-corpus passes such as the tag statistics want that)."""
        if not self.identity:
            self._full_pack(self.folders)

    def _segment_index(self):
        if self._seg_index is None:
            keys = [k for k in self._order() if self.segments[k][1] > self.segments[k][0]]
            self._seg_index = (keys, np.array([self.segments[k][0] for k in keys], dtype=np.int64))
        return self._seg_index

    def materialize(self, positions: Sequence[int], include_content: bool) -> List[Dict[str, Any]]:
        """The dicts list_memories yields (utils.py:234-243) for these listing positions; header text and body come from the device."""
        positions = np.asarray(positions, dtype=np.int64)
        m = len(positions)
        if m == 0:
            return []
        dev = self.dev[positions]
        hdr_text: List[str] = [""] * m
        body_text: List[str] = [""] * m
        for corpus, lo in self._corpora():
            sel = np.nonzero((dev >= lo) & (dev < lo + corpus.n))[0]
            if not len(sel):
                continue
            hdr, ho, body, bo = corpus.fetch_records(dev[sel] - lo, want_body=include_content)
            ho_l = ho.tolist()
            bo_l = bo.tolist() if include_content else None
            for k, j in enumerate(sel.tolist()):
                hdr_text[j] = hdr[ho_l[k]:ho_l[k + 1]].decode("utf-8")
                if include_content:
                    body_text[j] = body[bo_l[k]:bo_l[k + 1]].decode("utf-8")
        keys, starts = self._segment_index()
        which = np.searchsorted(starts, positions, side="right") - 1
        out: List[Optional[Dict[str, Any]]] = [None] * m
        fromts = datetime.fromtimestamp
        for w in np.unique(which).tolist():                             # per directory: pull the columns of its hits out as Python lists once
            key = keys[w]
            L = self.segs[key].listing
            js = np.nonzero(which == w)[0]
            idx = positions[js] - self.segments[key][0]
            no = L.name_off
            a_l, b_l = no[idx].tolist(), no[idx + 1].tolist()
            sp_l = L.spans[idx].tolist()
            ts_l = L.ts[idx].tolist()
            f8_l = L.flags8[idx].tolist()
            names = L.names
            folder, status = key
            for t, j in enumerate(js.tolist()):
                nb = names[a_l[t]:b_l[t]]
                s0, l0, s1, l1 = sp_l[t]
                flags = f8_l[t]
                ts = ts_l[t]
                mem = {"filename": os.fsdecode(nb), "folder": folder, "status": status, "headers": _headers_of(hdr_text[j]),
                       "metadata": {"timestamp": ts, "unique_id": os.fsdecode(nb[s0:s0 + l0]), "hostname": os.fsdecode(nb[s1:s1 + l1]),
                                    "flags": [chr((flags >> (8 * k)) & 0xFF) for k in range(flags >> 56)], "date": fromts(ts)}}
                if include_content:
                    mem["content"] = body_text[j]
                out[j] = mem
        return out  # type: ignore[return-value]

    # ---- per-record header values for conditions only Python can judge (search.py:126-130)
    def header_values(self, field: str) -> Tuple[np.ndarray, np.ndarray, List[str]]:
        """(present[n], inv[n], distinct), listing order: the value _get_field_value would read for `field` (first key whose lower()
        equals field.lower(), last line of that exact key) as an index into the list of distinct values (len(distinct) = absent)."""
        key = field.lower()
        got = self._field_values.get(key)
        if got is None:
            from .program import C_SLOT, Cond, ProgramBuilder
            from .regexc import Pattern
            pb = ProgramBuilder()
            pb.add_query([Cond(C_SLOT, pattern=Pattern("regex", "", re.IGNORECASE), field=field, mode=0)])
            prog = pb.build()
            index: Dict[bytes, int] = {}
            inv_dev = np.full(self.n_base + self.n_delta, -1, dtype=np.int64)
            for corpus, lo in self._corpora():
                present, off, blob = corpus.slot_values(prog)
                raw = blob.tobytes()
                o = off.astype(np.int64)
                for i in np.nonzero(present)[0].tolist():
                    inv_dev[lo + i] = index.setdefault(raw[o[i]:o[i + 1]], len(index))
            distinct = [b.decode("utf-8") for b in index]
            inv = inv_dev[self.dev] if self.n else np.zeros(0, dtype=np.int64)
            present = inv >= 0
            inv = np.where(present, inv, len(distinct))
            got = self._field_values[key] = (present, inv, distinct)
        return got

    # ---- result order (search.py:370-388)
    def sort_page(self, positions: np.ndarray, field: str, reverse: bool, include_content: bool, first: int, count: int) -> np.ndarray:
        """The listing positions of the hits (in hit order) ordered as the reference orders their dicts,
        results.sort(key=lambda x: _get_field_value(x, field) or "", reverse=reverse) with its warning and newest-first
        fallback (search.py:97-139, :370-382), then sliced to [first, first + count).  Keys the device can order go to
        fei_sort_rows; the sort runs on the host only where CPython's own comparisons define the outcome: keys of more than
        one class (str / int / naive / aware datetime), which make list.sort raise and leave a partial order, or a key that
        raises."""
        positions = np.asarray(positions, dtype=np.int64)
        m = len(positions)
        if m == 0:
            return positions
        low = field.lower()
        kw: Dict[str, Any] = {}
        if low == "content":
            if not include_content:                                   # memory.get("content", "") == "" for every hit: order unchanged
                return positions[first:first + count]
            kw["source"] = _abi.SORT_BODY
        elif low == "flags":
            kw["source"] = _abi.SORT_FLAGS
        elif low == "date":
            kw["source"] = _abi.SORT_WALL                             # naive datetime.fromtimestamp: the wall clock, not ts (DST)
        elif low == "id":
            kw["source"] = _abi.SORT_NAME_UID
        elif low == "filename":
            kw["source"] = _abi.SORT_NAME
        elif low in ("folder", "status", "maildir_status"):
            fsb = self.arrays["fsb"][positions]
            if low == "folder":
                ids, names = fsb & 0xFFFF, {i: f for f, i in self.folder_ids.items()}
            else:
                ids, names = (fsb >> 16) & 0xFF, dict(enumerate(U.STANDARD_FOLDERS))
            uniq, back = np.unique(ids, return_inverse=True)
            kw.update(source=_abi.SORT_KEYS, keys=np.asarray(_ranks([names[int(u)] for u in uniq]), dtype=np.uint64)[back])
        elif low in ("status_value", "state"):                        # headers.get("Status", ""): the exact key
            kw.update(source=_abi.SORT_SLOT, prog=_slot_prog("Status", 1))
        elif low in ("due", "created", "modified", "deleteddate", "timestamp"):
            keys = self._host_keys(positions, field, low)
            if keys is None or isinstance(keys, list):                # a key raised, or classes mix: CPython decides
                ts = self.arrays["ts"][positions].tolist()
                order = python_order(keys if keys is not None else [], ts, reverse, self._key_error)
                return positions[np.asarray(order, dtype=np.int64)][first:first + count]
            kw.update(source=_abi.SORT_KEYS, keys=keys)
        else:
            kw.update(source=_abi.SORT_SLOT, prog=_slot_prog(field, 0),
                      fallback={"unique_id": _abi.SORT_NAME_UID, "hostname": _abi.SORT_NAME_HOST}.get(low, _abi.SORT_NONE))
        if count <= 0:
            return positions[:0]
        corpora = self._corpora()
        dev = self.dev[positions]
        los = np.array([lo for _, lo in corpora], dtype=np.int64)
        rc = np.searchsorted(los, dev, side="right") - 1
        rows, self.last_sort_info = _abi.sort_rows([c for c, _ in corpora], rc, dev - los[rc], descending=reverse, first=first, count=count, **kw)
        return positions[rows]

    def _host_keys(self, positions: np.ndarray, field: str, low: str):
        """Keys of a date header (dateutil.parser.parse of the value, the raw value when that fails, search.py:124-131) or of
        `timestamp` (a header string, else the int metadata), `or ""` applied.  Returns uint64 ranks when every hit's key is of
        one class, the list of key objects when classes mix, None when computing a key raises (self._key_error)."""
        from .memdir_tools.search import _parse_dt
        import dateutil.parser
        self._key_error = None
        present, inv, distinct = self.header_values(field)
        inv_h = inv[positions]
        if low == "timestamp":
            ts_h = self.arrays["ts"][positions]
            hdr = present[positions]
            meta_str = ~hdr & (ts_h == 0)                             # int 0 or "" -> ""
            classes = (bool(hdr.any() or meta_str.any())) + bool((~hdr & (ts_h != 0)).any())
            if classes > 1 and len(positions) > 1:
                d = distinct + [""]
                return [d[u] if h else (t or "") for u, h, t in zip(inv_h.tolist(), hdr.tolist(), ts_h.tolist())]
            if not hdr.any() and not meta_str.any():
                return np.unique(ts_h, return_inverse=True)[1].astype(np.uint64)
            texts = np.array(distinct + [""], dtype=object)
            vals = np.where(hdr, inv_h, len(distinct))
            uniq, back = np.unique(vals, return_inverse=True)
            return np.asarray(_ranks([texts[u] for u in uniq]), dtype=np.uint64)[back]
        uniq, back = np.unique(inv_h, return_inverse=True)
        objs: List[Any] = []
        errs: Dict[int, BaseException] = {}
        for k, u in enumerate(uniq.tolist()):
            if u == len(distinct):
                objs.append("")                                       # no such header: None or "" -> ""
                continue
            text = distinct[u]
            parsed = self.parsed_dates.get(text)
            if parsed is None:
                parsed = self.parsed_dates[text] = _parse_dt(text)
            dt, today_dependent = parsed
            if dt is None or today_dependent:                         # parse as the reference does: default = today
                try:
                    dt = dateutil.parser.parse(text)
                except (ValueError, TypeError):
                    dt = None
                except Exception as e:                                # escapes _get_field_value and aborts the sort
                    errs[k] = e
            objs.append(dt if dt is not None else (text or ""))
        if errs:
            first_bad = int(np.nonzero(np.isin(back, list(errs)))[0][0])
            self._key_error = errs[int(back[first_bad])]
            return None
        kinds = {_key_class(o) for o in objs}
        if len(kinds) > 1 and len(positions) > 1:
            return [objs[b] for b in back.tolist()]
        return np.asarray(_ranks(objs), dtype=np.uint64)[back]

    def begin_query(self) -> None:
        self._aux_next = 0

    def new_aux(self, verdicts: np.ndarray) -> int:
        """Uploads one per-record verdict column (listing order) for the query being compiled; returns its index (C_RECBITS.which)."""
        from .program import MAX_AUX
        if self._aux_next >= MAX_AUX:
            raise NotImplementedError(f"more than {MAX_AUX} host-judged header conditions in one query")
        k = self._aux_next
        self._aux_next += 1
        dev_v = np.zeros(self.n_base + self.n_delta, dtype=np.uint8)
        dev_v[self.dev] = np.asarray(verdicts, dtype=np.uint8)
        for corpus, lo in self._corpora():
            corpus.set_aux(k, dev_v[lo:lo + corpus.n])
        return k

    def sigma_in(self, ranges: Sequence[Tuple[int, int]]) -> bool:
        """Does a record of these listing ranges hold U+03A3 (the one character whose str.lower() the automata do not model)?"""
        bits = self.arrays.get("rec_bits")
        if bits is None or not len(bits):
            return False
        return any(bool((bits[a:b] & REC_HAS_SIGMA).any()) for a, b in ranges)

    def report_skipped(self, folders: Optional[Sequence[str]], statuses: Optional[Sequence[str]]) -> None:
        """The reference prints `Error processing <file>: <error>` each time a directory is listed (utils.py:247-248)."""
        for f in (self.folders if folders is None else folders):
            for st in (U.STANDARD_FOLDERS if statuses is None else statuses):
                seg = self.segs.get((f, st))
                if seg is not None:
                    for msg in seg.bad:
                        print(msg)

    def ranges(self, folders: Optional[Sequence[str]], statuses: Optional[Sequence[str]]) -> List[Tuple[int, int]]:
        """Listing ranges of the requested (folder, status) pairs in the caller's order (search.py:361-363)."""
        if folders is None:
            folders = self.folders
        if statuses is None:
            statuses = U.STANDARD_FOLDERS
        out = []
        for f in folders:
            for st in statuses:
                if st not in U.STANDARD_FOLDERS:
                    raise ValueError(f"Invalid status: {st}. Must be one of {U.STANDARD_FOLDERS}")
                r = self.segments.get((f, st))
                if r and r[1] > r[0]:
                    out.append(r)
        return out

    # ---- snapshot
    def save_snapshot(self, path: str) -> None:
        """The packed corpus (device buffers) + the listings, so a restart restores instead of re-packing; the next sync() diffs
        the tree against the restored listings and reads only what changed since."""
        with self.lock:
            self.compact()
            self.corpus.save(path + ".corpus")
            blob: Dict[str, Any] = {"folders": np.array(self.folders, dtype=object)}
            for k, key in enumerate(self._order()):
                seg = self.segs[key]
                L = seg.listing
                blob[f"s{k}_names"] = np.frombuffer(L.names, dtype=np.uint8) if L.names else np.zeros(0, dtype=np.uint8)
                for a in ("name_off", "ts", "wall", "flags8", "spans", "ino", "size", "mtime_ns"):
                    blob[f"s{k}_{a}"] = getattr(L, a)
                blob[f"s{k}_mt"] = np.array([seg.mtime_ns], dtype=np.int64)
                blob[f"s{k}_bad"] = np.array(seg.bad, dtype=object)
            np.savez(path + ".dirs.npz", **blob)

    @classmethod
    def from_snapshot(cls, base: str, path: str) -> "PackedMemdir":
        from .corpus import Corpus
        z = np.load(path + ".dirs.npz", allow_pickle=True)
        pm = cls(base)
        pm.folders = [str(x) for x in z["folders"]]
        pm.folder_ids = {f: i for i, f in enumerate(pm.folders)}
        pos = 0
        for k, key in enumerate(pm._order()):
            L = DirListing()
            L.names = z[f"s{k}_names"].tobytes()
            for a in ("name_off", "ts", "wall", "flags8", "spans", "ino", "size", "mtime_ns"):
                setattr(L, a, z[f"s{k}_{a}"])
            L.n = len(L.ts); L.bad = []
            seg = _Seg(); seg.listing = L; seg.dev = np.arange(pos, pos + L.n, dtype=np.int64); seg.mtime_ns = -2; seg.bad = [str(x) for x in z[f"s{k}_bad"]]; seg.bad_files = {}
            pos += L.n
            pm.segs[key] = seg
        pm.corpus = Corpus()
        pm.snapshot_gbs = pm.corpus.load_snapshot(path + ".corpus")
        pm.n_base = pm.corpus.n
        pm._rebuild_listing()
        return pm

    def close(self) -> None:
        with self.lock:
            for c in (self.corpus, self.delta):
                if c is not None:
                    c.close()
            self.corpus = self.delta = None
            self.watcher.close()


def python_order(keys: Sequence[Any], ts: Sequence[int], reverse: bool, key_error: Optional[BaseException] = None) -> List[int]:
    """What search.py:370-382 does to a result list, on indices: list.sort by the keys (a failed sort leaves CPython's partial
    order, the same for indices as for the dicts), then on any exception the warning and a stable newest-first sort.
    key_error: the exception computing a key raised (the list is then left as it was)."""
    idx = list(range(len(ts)))
    try:
        if key_error is not None:
            raise key_error
        idx.sort(key=keys.__getitem__, reverse=reverse)
    except Exception as e:
        print(f"Warning: Unable to sort results: {e}")
        idx.sort(key=ts.__getitem__, reverse=True)
    return idx


def _key_class(o: Any) -> str:
    if isinstance(o, datetime):
        return "aware" if o.tzinfo is not None and o.utcoffset() is not None else "naive"
    return type(o).__name__


def _ranks(objs: Sequence[Any]) -> List[int]:
    """Dense ranks under Python's comparison (objects of one class); equal objects share a rank."""
    order = sorted(range(len(objs)), key=objs.__getitem__)
    out = [0] * len(objs)
    r = 0
    for t, i in enumerate(order):
        if t and objs[order[t - 1]] < objs[i]:
            r += 1
        out[i] = r
    return out


def _slot_prog(field: str, mode: int) -> bytes:
    """A program whose slot 0 names one header (mode 0: first key whose lower() equals the field; 1: the exact key)."""
    from .program import C_SLOT, Cond, ProgramBuilder
    from .regexc import Pattern
    pb = ProgramBuilder()
    pb.add_query([Cond(C_SLOT, pattern=Pattern("regex", "", re.IGNORECASE), field=field, mode=mode)])
    return pb.build()


def _subset(L: DirListing, sel: np.ndarray) -> DirListing:
    d = DirListing()
    d.names = b"".join(L.name_bytes(i) for i in sel.tolist())
    d.name_off = np.zeros(len(sel) + 1, dtype=np.uint64)
    np.cumsum((L.name_off[1:] - L.name_off[:-1])[sel], out=d.name_off[1:])
    for k in ("ts", "wall", "flags8", "spans", "ino", "size", "mtime_ns"):
        setattr(d, k, getattr(L, k)[sel])
    d.n = len(sel)
    d.bad = L.bad
    return d


# ----------------------------------------------------------------------------- host-side listing of one directory (no GPU)
def read_segment(base: str, folder: str, status: str) -> List[Dict[str, Any]]:
    """utils.list_memories for callers that want plain dicts of one directory (host only: the reference-shaped helper, and the
    one-record corpora of MemoryFilter.matches)."""
    path = os.path.join(base, folder, status) if folder else os.path.join(base, status)
    if not os.path.exists(path):
        return []
    out = []
    for name in os.listdir(path):
        try:
            if not _LIST_RE.match(name):
                continue
            m = U.FILENAME_RE.match(name)
            if not m:
                raise ValueError(f"Invalid memory filename: {name}")
            with open(os.path.join(path, name), "r") as f:
                text = f.read()
            head, sep, rest = text.partition("---")
            ts = int(m.group(1))
            out.append({"filename": name, "folder": folder, "status": status, "ts": ts, "uid": m.group(2), "host": m.group(3), "flags": m.group(4),
                        "uid_span": (m.start(2), m.end(2)), "host_span": (m.start(3), m.end(3)),
                        "hdr_text": head if sep else "", "body_text": (rest if sep else text).strip(), "has_sep": bool(sep),
                        "date": datetime.fromtimestamp(ts)})
        except Exception as e:
            print(f"Error processing {name}: {e}")
    out.sort(key=lambda r: r["ts"], reverse=True)
    return out


def memory_dict(rec: Dict[str, Any], include_content: bool) -> Dict[str, Any]:
    """The dict list_memories yields (utils.py:234-243) from a read_segment record."""
    headers = _headers_of(rec["hdr_text"]) if rec["has_sep"] else {}
    mem = {"filename": rec["filename"], "folder": rec["folder"], "status": rec["status"], "headers": headers,
           "metadata": {"timestamp": rec["ts"], "unique_id": rec["uid"], "hostname": rec["host"], "flags": list(rec["flags"]), "date": rec["date"]}}
    if include_content:
        mem["content"] = rec["body_text"]
    return mem


def arrays_from_segments(recs: Sequence[Dict[str, Any]], folder_ids: Dict[str, int], global_base: int = 0) -> Dict[str, Any]:
    """Canonical host arrays (fei_corpus_load) from read_segment records: the host-text path, used for one-record corpora
    (MemoryFilter.matches) and tests."""
    n = len(recs)
    hdr_parts = [r["hdr_text"].encode("utf-8") for r in recs]
    body_parts = [r["body_text"].encode("utf-8") for r in recs]
    name_parts = [os.fsencode(r["filename"]) for r in recs]

    def blob(parts):
        off = np.zeros(n + 1, dtype=np.uint64)
        if n:
            np.cumsum(np.fromiter(map(len, parts), dtype=np.int64, count=n), out=off[1:])
        data = np.frombuffer(b"".join(parts), dtype=np.uint8).copy() if n and off[n] else np.zeros(1, dtype=np.uint8)
        return data, off

    hdr, hdr_off = blob(hdr_parts)
    body, body_off = blob(body_parts)
    name, name_off = blob(name_parts)
    spans = np.zeros((max(n, 1), 4), dtype=np.uint16)
    bits = np.zeros(max(n, 1), dtype=np.uint32)
    for i, r in enumerate(recs):
        fname = r["filename"]
        (a0, a1), (b0, b1) = r["uid_span"], r["host_span"]
        if len(name_parts[i]) != len(fname):
            a0, a1, b0, b1 = (len(os.fsencode(fname[:x])) for x in (a0, a1, b0, b1))
        spans[i] = (a0, a1 - a0, b0, b1 - b0)
        b = 0 if r["has_sep"] else REC_NO_SEPARATOR
        text = r["hdr_text"] + r["body_text"]
        if not text.isascii():
            b |= REC_NONASCII
            if "Σ" in text:
                b |= REC_HAS_SIGMA
            if "İ" in text:
                b |= REC_HAS_IDOT
        bits[i] = b
    ts = np.array([r["ts"] for r in recs], dtype=np.int64)
    wall = np.array([calendar.timegm(r["date"].timetuple()) for r in recs], dtype=np.int64)
    f8 = np.array([_flags8(r["flags"], r["filename"]) for r in recs], dtype=np.uint64)
    fsb = np.array([(folder_ids[r["folder"]] & 0xFFFF) | (U.STANDARD_FOLDERS.index(r["status"]) << 16) | (int(bits[i]) << 24)
                    for i, r in enumerate(recs)], dtype=np.uint32)
    return {"n": n, "global_base": global_base, "hdr": hdr, "hdr_off": hdr_off, "body": body, "body_off": body_off,
            "name": name, "name_off": name_off, "name_spans": spans.reshape(-1), "ts": ts, "wall": wall, "flags8": f8, "fsb": fsb,
            "rec_bits": bits[:n].astype(np.uint8)}


def _flags8(flags: str, name: str) -> int:
    if len(flags) > 7:
        raise NotImplementedError(f"{name}: more than 7 flag letters are not supported by the packed layout")
    v = len(flags) << 56
    for k, ch in enumerate(flags):
        v |= ord(ch) << (8 * k)
    return v


# ----------------------------------------------------------------------------- process-wide cache
_cache: Dict[str, PackedMemdir] = {}
_cache_lock = threading.Lock()


def packed(base: Optional[str] = None) -> PackedMemdir:
    """The packed corpus for a tree, synced with the tree (see PackedMemdir.sync).  Callers hold `pm.lock` while they compile
    conditions against it and scan, so a request sees one consistent state."""
    base = base or U.MEMDIR_BASE
    with _cache_lock:
        pm = _cache.get(base)
        if pm is None:
            pm = _cache[base] = PackedMemdir(base)
    return pm.sync()


def drop(base: Optional[str] = None) -> None:
    """Forget (and free) the packed corpus of a tree, or of every tree."""
    with _cache_lock:
        keys = [base] if base else list(_cache)
        for k in keys:
            pm = _cache.pop(k, None)
            if pm is not None:
                pm.close()
