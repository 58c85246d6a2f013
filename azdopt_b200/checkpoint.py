"""Reader of the checkpoint blobs azb_checkpoint_save writes (format and digest defined in include/azb.h).

Plain numpy, no library call: it parses the header, restates the digest, and splits the tree section into records, so
that a blob can be inspected, and checked independently of the code that wrote it.
"""
from __future__ import annotations

import dataclasses

import numpy as np

MAGIC = 0x3154504B43425A41  # "AZBCKPT1"
FORMAT = 1
HEADER_WORDS = 96
HEADER_BYTES = 8 * HEADER_WORDS
BLK_PAD = 64   # block-arena units kept free in front of each tree's blocks (not saved)
WK_HDR = 80    # walker words before the state part
WK_NNODES, WK_NBLK, WK_INTOP, WK_STEP = 2, 3, 5, 7

_M64 = (1 << 64) - 1
_K = 0x9E3779B97F4A7C15


def mix64(z):
    """azb_mix64 on numpy uint64 arrays (wrapping arithmetic) or Python ints."""
    if isinstance(z, int):
        z = (z + _K) & _M64
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
        return z ^ (z >> 31)
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(_K)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def digest(data) -> int:
    """mix64(S ^ n), S = sum_i mix64(w_i ^ (i * 0x9E3779B97F4A7C15)) mod 2^64 over the n little-endian uint64 words."""
    w = np.frombuffer(memoryview(data), dtype="<u8") if not isinstance(data, np.ndarray) else data.view("<u8").reshape(-1)
    n = w.size
    with np.errstate(over="ignore"):
        i = np.arange(n, dtype=np.uint64) * np.uint64(_K)
        s = int(mix64(w.astype(np.uint64) ^ i).sum(dtype=np.uint64)) if n else 0
    return mix64(s ^ n)


def _f32(word: int) -> float:
    return float(np.array([word & 0xFFFFFFFF], dtype=np.uint32).view(np.float32)[0])


@dataclasses.dataclass
class Header:
    words: np.ndarray  # the 96 header words

    def __getitem__(self, i):
        return int(self.words[i])

    magic = property(lambda s: s[0])
    format = property(lambda s: s[1])
    version = property(lambda s: s[2])
    blob_bytes = property(lambda s: s[3])
    n_vertices = property(lambda s: s[4])
    c_lower = property(lambda s: _f32(s[5]))
    c_upper = property(lambda s: _f32(s[6]))
    n_as_tol = property(lambda s: [s[7 + i] for i in range(s[15])])
    n_as_tol_default = property(lambda s: s[16])
    mlp_hidden = property(lambda s: (s[17], s[18], s[19]))
    mlp_mode = property(lambda s: s[20])
    prior_mode = property(lambda s: s[21])
    prior_seed = property(lambda s: s[22])
    selection = property(lambda s: s[23])
    puct_c = property(lambda s: _f32(s[24]))
    first_root = property(lambda s: s[25])
    n_roots = property(lambda s: s[26])
    steps_done = property(lambda s: s[27])
    resets = property(lambda s: s[28])
    adam_t = property(lambda s: s[29])
    adam = property(lambda s: tuple(_f32(s[30 + i]) for i in range(5)))  # lr, beta1, beta2, eps, l2
    params_set = property(lambda s: bool(s[35] & 1))
    best_ord = property(lambda s: s[36])
    best_root = property(lambda s: s[37])
    best_node = property(lambda s: s[38])
    n_params = property(lambda s: s[78])
    model = property(lambda s: (s[79], s[80]))
    table = property(lambda s: (s[81], s[82]))
    trees = property(lambda s: (s[83], s[84]))
    model_digest = property(lambda s: s[85])
    table_digest = property(lambda s: s[86])
    header_digest = property(lambda s: s[95])

    @property
    def best_eval(self) -> np.float32:
        o = self.best_ord
        u = (o & 0x7FFFFFFF) if o & 0x80000000 else (~o & 0xFFFFFFFF)
        return np.array([u], dtype=np.uint32).view(np.float32)[0]

    @property
    def best_state(self):
        """(parents u8[N], permitted u32[W]) of the running best."""
        st = self.words[39:78].view(np.uint32)[:77]
        n = self.n_vertices
        a = (n - 1) * (n - 2) // 2 - 1
        return st[:16].view(np.uint8)[:n].copy(), st[16:16 + (a + 31) // 32].copy()


def _u8(blob) -> np.ndarray:
    return blob.view(np.uint8).reshape(-1) if isinstance(blob, np.ndarray) else np.frombuffer(memoryview(blob), dtype=np.uint8)


def read_header(blob) -> Header:
    """The header of a blob (bytes, numpy array or np.memmap); raises ValueError on a bad magic, format or digest."""
    b = _u8(blob)
    if b.size < HEADER_BYTES:
        raise ValueError("shorter than a checkpoint header")
    w = b[:HEADER_BYTES].view("<u8").astype(np.uint64)
    h = Header(w)
    if h.magic != MAGIC:
        raise ValueError("bad magic")
    if h.format != FORMAT:
        raise ValueError(f"format {h.format}, this reader knows {FORMAT}")
    if digest(b[:HEADER_BYTES - 8]) != h.header_digest:
        raise ValueError("header digest")
    return h


def tree_offsets(blob, h: Header = None) -> np.ndarray:
    b = _u8(blob)
    h = h or read_header(b)
    off, size = h.table
    return b[off:off + size].view("<u8").astype(np.uint64)


def tree_record(blob, i: int, h: Header = None) -> np.ndarray:
    """Record of the blob's i-th root as uint32 words (its last two words are the digest)."""
    b = _u8(blob)
    h = h or read_header(b)
    t = tree_offsets(b, h)
    base = h.trees[0]
    return b[base + int(t[i]):base + int(t[i + 1])].view("<u4")


def record_sizes(rec: np.ndarray, n_vertices: int):
    """(n_nodes, nblk, intop, data words) of a record, from its walker words."""
    a = (n_vertices - 1) * (n_vertices - 2) // 2 - 1
    w = (a + 31) // 32
    ws = WK_HDR + 2 * ((n_vertices + 3) // 4) + 3 * w
    nn, nblk, intop = int(rec[WK_NNODES]), int(rec[WK_NBLK]), int(rec[WK_INTOP])
    data = ws + nn * (16 + w) + 2 * max(nblk - BLK_PAD, 0) + 2 * intop
    return nn, nblk, intop, (data + 1) & ~1


def verify(blob) -> Header:
    """Every digest and every length of a blob, restated here; raises ValueError naming the first mismatch."""
    b = _u8(blob)
    h = read_header(b)
    if h.blob_bytes != b.size:
        raise ValueError(f"{b.size} bytes, the header says {h.blob_bytes}")
    mo, ms = h.model
    if ms != (12 * h.n_params + 7) & ~7 or digest(b[mo:mo + ms]) != h.model_digest:
        raise ValueError("model section")
    to, ts = h.table
    if ts != 8 * (h.n_roots + 1) or digest(b[to:to + ts]) != h.table_digest:
        raise ValueError("tree offset table")
    t = tree_offsets(b, h)
    if int(t[0]) != 0 or int(t[-1]) != h.trees[1] or h.trees[0] + h.trees[1] != b.size:
        raise ValueError("tree section size")
    for i in range(h.n_roots):
        rec = tree_record(b, i, h)
        *_, data = record_sizes(rec, h.n_vertices)
        if data + 2 != rec.size:
            raise ValueError(f"root {h.first_root + i}: record length")
        if digest(rec[:data]) != int(rec[data:].view("<u8")[0]):
            raise ValueError(f"root {h.first_root + i}: record digest")
    return h
