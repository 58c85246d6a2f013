"""On-disk outputs the reference's example and its `pics` tooling expect (SURVEY.md §8f row 4), host side only:

* graph6 of a state's tree (graph-state/src/simple_graph/connected_bitset_graph/graph6.rs:11-39; the g6 standard);
* a Graphviz DOT description of one search DAG with the reference's node labels and attributes
  (az-discrete-opt/src/nabla/tree/graphviz.rs:9-51; the reference pipes it through `dot -Tpng`);
* a TensorBoard event file with the scalars the example writes: `cost/cost`, `cost/lambda_1`, `cost/mu`
  (connected_bitset_graph/mod.rs:355-365) and `loss` (nabla/model/mod.rs:25-32), framed as TFRecords
  (length, masked CRC-32C of the length, payload, masked CRC-32C of the payload) around `Event` protos — what the
  `tensorboard_writer` crate emits (04-c21-tree.rs:77-84,121,163-170).
No dependency on tensorflow / protobuf: the few messages are encoded by hand.
"""
from __future__ import annotations

import struct
import time
from typing import Iterable, Sequence, Tuple


# ---- graph6 --------------------------------------------------------------------------------------------------------
def graph6_from_edges(n: int, edges: Iterable[Tuple[int, int]]) -> bytes:
    """g6 string of the simple graph on `n` <= 62 vertices (graph6.rs:11-39: upper triangle column by column, six bits
    per byte, big-endian within the byte, zero padded, each byte + 63)."""
    if not 0 <= n <= 62:
        raise ValueError("graph6: at most 62 vertices (graph6.rs:17-23 leaves the long form unimplemented)")
    adj = [[False] * n for _ in range(n)]
    for u, v in edges:
        if u == v or not (0 <= u < n and 0 <= v < n):
            raise ValueError(f"bad edge ({u}, {v})")
        adj[u][v] = adj[v][u] = True
    bits = [adj[u][v] for v in range(n) for u in range(v)]  # edge_bools (mod.rs:123-132): for v, for u < v
    bits += [False] * ((6 - len(bits) % 6) % 6)
    out = bytearray([n + 63])
    for i in range(0, len(bits), 6):
        byte = 0
        for b in bits[i:i + 6]:
            byte = (byte << 1) | int(b)
        out.append(byte + 63)
    return bytes(out)


def tree_edges(parents: Sequence[int]) -> list:
    """Edges of a RootedOrderedTree given as its parent array (rooted_tree/mod.rs:8-10): (v, parents[v]) for v >= 1."""
    return [(v, int(parents[v])) for v in range(1, len(parents))]


def graph6_of_state(parents: Sequence[int]) -> bytes:
    return graph6_from_edges(len(parents), tree_edges(parents))


# ---- canonical code of a tree (include/azb.h: azb_tree_codes) -------------------------------------------------------
def tree_code(parents: Sequence[int]) -> Tuple[int, int]:
    """The canonical code of the tree with edges {v, parents[v]} (parents[v] < v), as two 64-bit words: the maximum over
    the centres r of enc(r) = 1 . enc(c_1) ... enc(c_d) . 0 with the children's codes in descending order, string bit i
    at bit 63 - i % 64 of word i // 64.  Equal codes <=> isomorphic trees.  The plain statement azb_tree_codes is
    checked against."""
    n = len(parents)
    adj = [[] for _ in range(n)]
    for v in range(1, n):
        p = int(parents[v])
        if not 0 <= p < v:
            raise ValueError(f"parents[{v}] = {p} is not < {v}")
        adj[v].append(p)
        adj[p].append(v)
    alive = set(range(n))
    while len(alive) > 2:  # the centres: strip every leaf at once
        alive -= {v for v in alive if sum(u in alive for u in adj[v]) <= 1}

    def enc(v, up):
        return "1" + "".join(sorted((enc(u, v) for u in adj[v] if u != up), reverse=True)) + "0"

    bits = int(max(enc(r, -1) for r in alive).ljust(128, "0"), 2)
    return bits >> 64, bits & ((1 << 64) - 1)


# ---- Graphviz ------------------------------------------------------------------------------------------------------
def search_tree_dot(dump: dict) -> str:
    """DOT text of one SearchTree from its canonical dump (capi.Handle.dump_tree / the oracle's dump): node label
    s{index}n{n_t}x{exhausted_children}, inactive nodes drawn as double circles, arcs into active nodes carry
    dir=forward (graphviz.rs:11-45).  Out-arcs are listed newest first like petgraph's neighbors_directed."""
    nodes, arcs = dump["nodes"], dump["arcs"]

    def label(i):
        return f"s{i}n{int(nodes[i][2])}x{int(nodes[i][3])}"

    def active(i):  # StateWeight::is_active (state_weight.rs:31-33)
        return int(nodes[i][4]) + int(nodes[i][3]) < int(nodes[i][5])

    lines = ["graph search_tree {"]
    for i in range(len(nodes)):
        lines.append(f"  {label(i)}" + ("" if active(i) else " [shape=doublecircle]"))
    out = {}
    for src, dst, _ in arcs:
        out.setdefault(int(src), []).append(int(dst))
    for u in range(len(nodes)):
        for v in reversed(out.get(u, [])):
            lines.append(f"  {label(u)} -- {label(v)}" + (" [dir=forward]" if active(v) else ""))
    lines.append("}")
    return "\n".join(lines) + "\n"


# ---- TensorBoard event files -----------------------------------------------------------------------------------------
_CRC_TABLE = []


def _crc_table():
    if not _CRC_TABLE:
        for i in range(256):
            c = i
            for _ in range(8):
                c = (c >> 1) ^ (0x82F63B78 if c & 1 else 0)  # CRC-32C (Castagnoli), reflected
            _CRC_TABLE.append(c)
    return _CRC_TABLE


def crc32c(data: bytes) -> int:
    t, c = _crc_table(), 0xFFFFFFFF
    for b in data:
        c = t[(c ^ b) & 0xFF] ^ (c >> 8)
    return c ^ 0xFFFFFFFF


def masked_crc32c(data: bytes) -> int:  # TFRecord's mask
    c = crc32c(data)
    return ((((c >> 15) | (c << 17)) & 0xFFFFFFFF) + 0xA282EAD8) & 0xFFFFFFFF


def _varint(x: int) -> bytes:
    out = bytearray()
    while True:
        b = x & 0x7F
        x >>= 7
        out.append(b | (0x80 if x else 0))
        if not x:
            return bytes(out)


def _field(num: int, wire: int, payload: bytes) -> bytes:
    return _varint((num << 3) | wire) + payload


def _event(wall_time: float, step: int, *, file_version: str = None, scalars: dict = None) -> bytes:
    # Event { double wall_time = 1; int64 step = 2; string file_version = 3; Summary summary = 5; }
    ev = _field(1, 1, struct.pack("<d", wall_time)) + _field(2, 0, _varint(step & 0xFFFFFFFFFFFFFFFF))
    if file_version is not None:
        fv = file_version.encode()
        ev += _field(3, 2, _varint(len(fv)) + fv)
    if scalars:
        summ = b""
        for tag, value in scalars.items():  # Summary { repeated Value value = 1; }  Value { string tag = 1; float simple_value = 2; }
            t = tag.encode()
            val = _field(1, 2, _varint(len(t)) + t) + _field(2, 5, struct.pack("<f", float(value)))
            summ += _field(1, 2, _varint(len(val)) + val)
        ev += _field(5, 2, _varint(len(summ)) + summ)
    return ev


class TensorboardWriter:
    """tensorboard_writer::TensorboardWriter as the example uses it: write_file_version, then write_summary(time,
    step, summary) per logged point (04-c21-tree.rs:81-84,121,163-170)."""

    def __init__(self, fileobj):
        self.f = fileobj

    def _record(self, payload: bytes):
        head = struct.pack("<Q", len(payload))
        self.f.write(head + struct.pack("<I", masked_crc32c(head)) + payload + struct.pack("<I", masked_crc32c(payload)))

    def write_file_version(self):
        self._record(_event(time.time(), 0, file_version="brain.Event:2"))

    def write_summary(self, step: int, scalars: dict, wall_time: float = None):
        self._record(_event(time.time() if wall_time is None else wall_time, step, scalars=scalars))

    def write_cost(self, step: int, lambda_1: float, mu: int):
        """Conjecture2Dot1Cost::summary (connected_bitset_graph/mod.rs:355-365)."""
        self.write_summary(step, {"cost/cost": lambda_1 + mu, "cost/lambda_1": lambda_1, "cost/mu": mu})

    def write_loss(self, step: int, loss: float):
        """impl Summarize for f32 (nabla/model/mod.rs:25-32)."""
        self.write_summary(step, {"loss": loss})

    def flush(self):
        self.f.flush()


def read_events(data: bytes):
    """Parse an event file back into (step, {tag: value}) pairs, checking every CRC (used by the tests)."""
    def rd_varint(buf, i):
        x = s = 0
        while True:
            b = buf[i]
            i += 1
            x |= (b & 0x7F) << s
            s += 7
            if not b & 0x80:
                return x, i

    def fields(buf):
        i = 0
        while i < len(buf):
            key, i = rd_varint(buf, i)
            num, wire = key >> 3, key & 7
            if wire == 0:
                v, i = rd_varint(buf, i)
            elif wire == 1:
                v, i = buf[i:i + 8], i + 8
            elif wire == 5:
                v, i = buf[i:i + 4], i + 4
            elif wire == 2:
                n, i = rd_varint(buf, i)
                v, i = buf[i:i + n], i + n
            else:
                raise ValueError("wire type")
            yield num, wire, v

    out, i = [], 0
    while i < len(data):
        head = data[i:i + 8]
        (n,) = struct.unpack("<Q", head)
        assert struct.unpack("<I", data[i + 8:i + 12])[0] == masked_crc32c(head), "length CRC"
        payload = data[i + 12:i + 12 + n]
        assert struct.unpack("<I", data[i + 12 + n:i + 16 + n])[0] == masked_crc32c(payload), "payload CRC"
        i += 16 + n
        step, scalars, version = 0, {}, None
        for num, _, v in fields(payload):
            if num == 2:
                step = v
            elif num == 3:
                version = v.decode()
            elif num == 5:
                for n2, _, val in fields(v):
                    tag = value = None
                    for n3, _, x in fields(val):
                        if n3 == 1:
                            tag = x.decode()
                        elif n3 == 2:
                            (value,) = struct.unpack("<f", x)
                    scalars[tag] = value
        out.append((step, scalars, version))
    return out
