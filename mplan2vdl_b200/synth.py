"""Synthetic TPC-H-shaped columns drawn to the reference's bounds metadata.

The reference ships metadata but no data, so throughput is reported on columns generated to
``tests/tpch10noorder/bounds.csv`` (min, max, trailing zeros, count; Config.hs:57, 114-120).
The recipe is *counter based*: a value depends only on (seed, stream, global row), so every
GPU shard generates its own row range in place (``vdl_column_fill_synthetic``) and the CPU
oracle generates identical data on the host -- nothing crosses PCIe.

    base = splitmix64(seed ^ (stream * 0x9E3779B97F4A7C15));  h = splitmix64(base + row)
    UNIFORM : vmin + stride * mulhi64(h, p0)         p0 = number of distinct values
    SEQ     : vmin + stride * row
    FKDENSE : vmin + stride * ((row * p0) // p1)     nondecreasing FK; p0 = dim rows, p1 = fact rows

Columns that must agree row by row (an FK index column and the key column it was built from,
e.g. lineitem_orders / l_orderkey) share one ``stream``.
"""
from __future__ import annotations

from dataclasses import dataclass

from .meta import Catalog

UNIFORM, SEQ, FKDENSE = 0, 1, 2

# lineitem cardinalities per TPC-H scale factor (SF10 is the fixture's own count, bounds.csv:59-79).
_LINEITEM_ROWS = {1: 6_001_215, 10: 59_986_052, 100: 600_037_902}
_FIXED_ROWS = {"nation": 25, "region": 5}


@dataclass(frozen=True)
class ColumnSpec:
    name: str       # "table.column"
    width: int      # 4 or 8 bytes
    kind: int
    vmin: int
    stride: int
    p0: int
    p1: int
    stream: int     # RNG stream id (64-bit)


def seed_for(sf: float) -> int:
    return 0x5EED ^ int(round(sf * 1000))


def _fnv1a(s: str) -> int:
    h = 0xCBF29CE484222325
    for b in s.encode():
        h = ((h ^ b) * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return h


def table_rows(cat: Catalog, table: str, sf: float) -> int:
    if table in _FIXED_ROWS:
        return _FIXED_ROWS[table]
    if table == "lineitem" and sf in _LINEITEM_ROWS:
        return _LINEITEM_ROWS[int(sf)]
    return max(1, int(round(cat.tables[table].rows * sf / 10.0)))


# columns whose values are dictionary codes with a non-power-of-two spacing, or whose real
# distribution is a sequence: (kind, vmin, stride, number of values or None = table rows)
_SPECIAL = {
    "lineitem.l_returnflag": (UNIFORM, 16, 24, 3),     # 16, 40, 64   (dictionary.csv:80-82)
    "lineitem.l_linestatus": (UNIFORM, 16, 24, 2),     # 16, 40
    "customer.c_mktsegment": (UNIFORM, -112, 32, 5),   # 5 codes, includes 16 = 'BUILDING' (dictionary.csv:74)
    "nation.n_name": (SEQ, 16, 24, None),              # distinct per nation, inside [16, 640]
    "region.r_name": (SEQ, 16, 24, None),              # 16, 40 'AMERICA', 64 'ASIA', 88, 112
    "region.r_regionkey": (SEQ, 0, 1, None),
    "nation.n_nationkey": (SEQ, 0, 1, None),
    "customer.c_custkey": (SEQ, 1, 1, None),
    "supplier.s_suppkey": (SEQ, 1, 1, None),
    "part.p_partkey": (SEQ, 1, 1, None),
    "orders.o_orderkey": (SEQ, 1, 4, None),
}

# key column -> (FK index column it mirrors, vmin, stride): value = vmin + stride * fk_index
_MIRRORS = {
    "lineitem.l_orderkey": ("lineitem_orders", 1, 4),
    "lineitem.l_suppkey": ("lineitem_supplier", 1, 1),
    "lineitem.l_partkey": ("lineitem_part", 1, 1),
    "orders.o_custkey": ("orders_customer", 1, 1),
    "customer.c_nationkey": ("customer_nation", 0, 1),
    "supplier.s_nationkey": ("supplier_nation", 0, 1),
    "nation.n_regionkey": ("nation_region", 0, 1),
    "partsupp.ps_partkey": ("partsupp_part", 1, 1),
    "partsupp.ps_suppkey": ("partsupp_supplier", 1, 1),
}


def column_spec(cat: Catalog, qualified: str, sf: float) -> ColumnSpec:
    table, cname = qualified.split(".", 1)
    tab = cat.tables[table]
    col = tab.columns[cname]
    rows = table_rows(cat, table, sf)
    fk = {f.name: f for f in tab.fkeys}
    stream = _fnv1a(qualified)

    def fk_spec(fkname: str, vmin: int, stride: int) -> ColumnSpec:
        dim_rows = table_rows(cat, fk[fkname].ref_table, sf)
        s = _fnv1a(f"{table}.{fkname}")
        if fkname == "lineitem_orders":   # clustered: lineitem is stored in l_orderkey order (storage.csv:188)
            return ColumnSpec(qualified, col.width, FKDENSE, vmin, stride, dim_rows, rows, s)
        return ColumnSpec(qualified, col.width, UNIFORM, vmin, stride, dim_rows, 0, s)

    if cname in fk:
        return fk_spec(cname, 0, 1)
    if qualified in _MIRRORS:
        fkname, vmin, stride = _MIRRORS[qualified]
        return fk_spec(fkname, vmin, stride)
    if qualified in _SPECIAL:
        kind, vmin, stride, n = _SPECIAL[qualified]
        return ColumnSpec(qualified, col.width, kind, vmin, stride, n if n is not None else rows, 0, stream)
    if col.vmin == -(1 << 63):            # pkey pseudo-columns carry nil bounds (bounds.csv:4): row ids
        return ColumnSpec(qualified, col.width, SEQ, 0, 1, rows, 0, stream)
    tz = col.trailing_zeros if col.vmax > col.vmin else 0
    nvals = ((col.vmax - col.vmin) >> tz) + 1
    return ColumnSpec(qualified, col.width, UNIFORM, col.vmin, 1 << tz, nvals, 0, stream)


# ------------------------------------------------------------------------------------------ string heaps
# `Like` reads the strings of a char / varchar column from its heap, `Load,<table>.<col>.heap` (Vdl.hs:244-247): a byte
# vector in which every string is NUL-terminated; the column itself holds byte offsets into it (MonetDB's layout; the
# offsets of bounds.csv are multiples of 8, trailing_zeros = 3).  The synthetic heap of a column is a POOL of distinct
# strings built from the TPC-H word lists (dbgen's grammar, reduced), laid out from the column's minimum offset on, each
# padded to the next multiple of 8; a row draws a pool entry with the same counter-based hash as the UNIFORM kind, so
# shards and the host agree.  Returns numpy arrays; the heap is small (<= a few MB), the offsets are per row.
_SYLL1 = ["STANDARD", "SMALL", "MEDIUM", "LARGE", "ECONOMY", "PROMO"]
_SYLL2 = ["ANODIZED", "BURNISHED", "PLATED", "POLISHED", "BRUSHED"]
_SYLL3 = ["TIN", "NICKEL", "BRASS", "STEEL", "COPPER"]
_COLORS = ("almond antique aquamarine azure beige bisque black blanched blue blush brown burlywood burnished chartreuse chiffon "
           "chocolate coral cornflower cornsilk cream cyan dark deep dim dodger drab firebrick floral forest frosted gainsboro "
           "ghost goldenrod green grey honeydew hot indian ivory khaki lace lavender lawn lemon light lime linen magenta maroon "
           "medium metallic midnight mint misty moccasin navajo navy olive orange orchid pale papaya peach peru pink plum powder "
           "puff purple red rose rosy royal saddle salmon sandy seashell sienna sky slate smoke snow spring steel tan thistle "
           "tomato turquoise violet wheat white yellow").split()
_FILLER = ("furiously carefully quickly slyly blithely final ironic regular express bold pending even silent unusual special "
           "Customer Complaints Recommends requests deposits packages accounts foxes ideas theodolites pinto beans instructions "
           "dependencies excuses platelets asymptotes courts dolphins multipliers sauternes warthogs frets dinos attainments "
           "somas Tiresias patterns forges braids hockey players frays warhorses dugouts notornis epitaphs pearls tithes "
           "waters orbits gifts sheaves depths sentiments decoys realms pains grouches escapades").split()


def _sm64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    z = x
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)


def string_pool(qualified: str) -> list:
    """The distinct strings of a column's synthetic heap, in heap order."""
    col = qualified.split(".", 1)[1]
    if col == "p_type":
        return [f"{a} {b} {c}" for a in _SYLL1 for b in _SYLL2 for c in _SYLL3]
    h0 = _fnv1a(qualified + ".heap")
    words, n, k = (_COLORS, 16384, 5) if col == "p_name" else (_FILLER, 4096, 9)
    out = []
    for i in range(n):
        h = _sm64(h0 + i)
        ws = []
        for j in range(k):
            h = _sm64(h + j)
            ws.append(words[h % len(words)])
        out.append(" ".join(ws))
    return out


def is_heap(qualified: str) -> bool:
    return qualified.endswith(".heap")


def string_heap(cat: Catalog, qualified: str):
    """(heap bytes as numpy uint8, offsets of the pool entries as numpy int64) of column `qualified` (no `.heap` suffix)."""
    import numpy as np
    c = cat.column(qualified)
    start = max(16, (c.vmin + 7) // 8 * 8) if c.vmin > -(1 << 62) else 16
    pool = string_pool(qualified)
    offs, parts, at = [], [bytes(start)], start
    for s in pool:
        b = s.encode() + b"\0"
        b += bytes(-len(b) % 8)
        offs.append(at)
        parts.append(b)
        at += len(b)
    return np.frombuffer(b"".join(parts), dtype=np.uint8).copy(), np.asarray(offs, dtype=np.int64)


def string_offsets(cat: Catalog, qualified: str, rows: int, row_offset: int, seed: int):
    """Offsets column of `rows` rows from global row `row_offset`: pool entry mulhi64(splitmix64(base + row), |pool|)."""
    import numpy as np
    _heap, offs = string_heap(cat, qualified)
    base = _sm64((seed ^ (_fnv1a(qualified) * 0x9E3779B97F4A7C15)) & 0xFFFFFFFFFFFFFFFF)
    with np.errstate(over="ignore"):
        x = (np.arange(rows, dtype=np.uint64) + np.uint64(row_offset) + np.uint64(base)) + np.uint64(0x9E3779B97F4A7C15)
        z = x
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    idx = ((z >> np.uint64(32)) * np.uint64(len(offs)) >> np.uint64(32)).astype(np.int64)      # mulhi on the high word: uniform enough
    return offs[idx]


# ------------------------------------------------------------------------------------------ code heaps
# A char column that is not Loaded with its heap holds dictionary codes drawn at a fixed stride (UNIFORM / SEQ above:
# l_returnflag 16, 40, 64; o_orderpriority -128, -120, ..., 104).  To order such a column by its strings the executor
# needs strings behind the codes: the code heap puts a NUL-terminated string of at most stride - 1 bytes at byte
# code - origin of every code the recipe can draw, origin being the smallest.  A code dictionary.csv names holds that
# string (cut to fit: '1-URGENT' at stride 8 is '1-URGEN'); every other code a string of the TPC-H filler words, of a
# length and content fixed by the column's name and the code.  The column's values are untouched.
def _sm64_np(x):
    import numpy as np
    with np.errstate(over="ignore"):
        z = x + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def code_heap(cat: Catalog, qualified: str):
    """(heap bytes as numpy uint8, origin) of the dictionary codes of char column `qualified`: the string of code c starts
    at heap byte c - origin.  ValueError for a column whose codes are not drawn at a fixed stride."""
    import numpy as np
    col = cat.column(qualified)
    spec = column_spec(cat, qualified, 10)
    if spec.kind not in (UNIFORM, SEQ) or spec.stride < 2 or col.mtype not in ("char", "varchar"):
        raise ValueError(f"{qualified}: no code heap (a {col.mtype} column whose synthetic values are not codes at a fixed stride)")
    count = spec.p0 if spec.kind == UNIFORM else (col.vmax - spec.vmin) // spec.stride + 1
    width = spec.stride - 1
    named = {code: s for s, code in cat.dictionary.get(qualified, {}).items()}
    h = _sm64_np(np.arange(count, dtype=np.uint64) + np.uint64(_fnv1a(qualified + ".codes")))
    words = [h]
    for _ in range(3):
        words.append(_sm64_np(words[-1]))
    lens = (1 + (h >> np.uint64(32)) % np.uint64(width)).tolist()
    idx = [(w % np.uint64(len(_FILLER))).tolist() for w in words[1:]]
    out = []
    for k in range(count):
        s = named.get(spec.vmin + k * spec.stride)
        b = s.encode() if s is not None else " ".join(_FILLER[ix[k]] for ix in idx).encode()[:lens[k]]
        out.append(b[:width].ljust(spec.stride, b"\0"))
    return np.frombuffer(b"".join(out), dtype=np.uint8).copy(), spec.vmin
