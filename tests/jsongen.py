"""A seeded generator of valid JSON with known answers, for differential tests of stage 2 and the pointer lookups.

The generator has its own serializer (it never calls json.dumps), so the bytes it writes are not limited to what Python's
json writes: every escape in both hex cases, surrogate pairs, raw UTF-8 of 1 to 4 bytes, empty, escaped, numeric-looking and
repeated keys, strings past 64 B and 2 KiB, integers of 1 to 19 digits and the int64 limits, doubles on and off the exact
fast path, wide and deep containers, and any whitespace between tokens.  For every document it returns

    data    the bytes (no framing around them)
    value   the Python value in the shape oracle.decode_tape returns: objects as ("object", [(key, value), ...]) so that member
            order and repeated keys survive, arrays as lists; a double is a Float, a float that remembers its token
    paths   every location in the document as a list of reference tokens (str keys, int indexes); the root is []
    tokens  the number of structurals stage 1 gives the document

`stream()` frames documents as NDJSON (LF or CRLF, blank lines) or as concatenated JSON and records where each starts.
`Gen.counts` counts the features written, so that tests can assert the coverage they claim."""
from __future__ import annotations

import random
from collections import Counter
from dataclasses import dataclass, field

INT64_MIN, INT64_MAX = -(1 << 63), (1 << 63) - 1
MAX_ARRAY_LEVEL = 99    # the deepest level an array may open at (the document's root is level 1)
MAX_OBJECT_LEVEL = 100  # objects go one level deeper than arrays
WIDE = 2049             # more elements than one 2048-token block of the tape kernels holds
WS = b" \t\n\r"


class Float(float):
    """A double with the token it was written as: the device's payload is a function of the token, not of the value."""

    tok: bytes

    def __new__(cls, tok: bytes):
        f = super().__new__(cls, float(tok))
        f.tok = tok
        return f


@dataclass
class Doc:
    data: bytes
    value: object
    paths: list = field(default_factory=list)
    tokens: int = 0


SHORT_ESCAPES = {b'\\"': '"', b"\\\\": "\\", b"\\/": "/", b"\\b": "\b", b"\\f": "\f", b"\\n": "\n", b"\\r": "\r", b"\\t": "\t"}
U_EDGES = [0x0000, 0x001F, 0x007F, 0x0080, 0x07FF, 0x0800, 0xFFFF, 0xD7FF, 0xE000, 0xFFFD]
RAW_CHARS = ["a", "Z", "~", "/", "0", " ", "é", "ß", "ߴ", "中", "€", "ࠀ", "￿", "😀", "\U00010000", "\U0010ffff"]
KEY_WORDS = ["", "a", "b", "id", "0", "1", "10", "-", "a/b", "~", "~0", "~1", "/", "//", "a~b", "é", "中文", "😀", " ", "key", "x.y", "\\"]


class Gen:
    def __init__(self, seed: int, ws: float = 0.3, deep: float = 0.01, wide: float = 0.004, long: float = 0.01, ws_bytes: bytes = WS):
        """ws: how often whitespace goes between two tokens, drawn from ws_bytes (leave out '\\n' for one document per line);
        deep, wide, long: how often a document is a chain to the deepest level, a container is wide, a string is long."""
        self.r = random.Random(seed)
        self.counts: Counter = Counter()
        self.ws, self.p_deep, self.p_wide, self.p_long, self.ws_bytes = ws, deep, wide, long, ws_bytes

    # ---- whitespace ---------------------------------------------------------------------------------------------------------
    def space(self, force: bool = False) -> bytes:
        r = self.r
        if not force and r.random() >= self.ws:
            return b""
        out = bytes(r.choice(self.ws_bytes) for _ in range(r.choice((1, 1, 1, 2, 3, 6))))
        for c, name in zip(WS, ("ws_space", "ws_tab", "ws_lf", "ws_cr")):
            if c in out:
                self.counts[name] += 1
        return out

    # ---- strings ------------------------------------------------------------------------------------------------------------
    def _u(self, cp: int) -> bytes:
        upper = self.r.random() < 0.5
        self.counts["u_upper" if upper else "u_lower"] += 1
        h = b"%04X" % cp if upper else b"%04x" % cp
        return b"\\u" + h

    def char(self) -> tuple[bytes, str]:
        r, c = self.r, self.r.random()
        if c < 0.45:
            ch = r.choice(RAW_CHARS)
            self.counts["utf8_%d" % len(ch.encode())] += 1
            return ch.encode(), ch
        if c < 0.6:
            esc = r.choice(list(SHORT_ESCAPES))
            self.counts["esc_" + esc[1:].decode()] += 1
            return esc, SHORT_ESCAPES[esc]
        if c < 0.72:
            cp = r.choice(U_EDGES)
            self.counts["u_%04x" % cp] += 1
            return self._u(cp), chr(cp)
        if c < 0.84:
            cp = r.choice((r.randrange(0x80), r.randrange(0x80, 0x800), r.randrange(0x800, 0xD800), r.randrange(0xE000, 0x10000)))
            self.counts["u_bmp"] += 1
            return self._u(cp), chr(cp)
        if c < 0.94:
            cp = r.choice((0x10000, 0x10FFFF, 0x1F600, r.randrange(0x10000, 0x110000)))
            v = cp - 0x10000
            self.counts["surrogate_pair"] += 1
            if cp == 0x10FFFF:
                self.counts["surrogate_pair_max"] += 1
            return self._u(0xD800 + (v >> 10)) + self._u(0xDC00 + (v & 0x3FF)), chr(cp)
        ch = chr(r.choice((0x7F, 0x20, 0x41)))   # raw bytes JSON lets through unescaped (DEL is one; those below 0x20 are not)
        return ch.encode(), ch

    def text(self, n: int) -> tuple[bytes, str]:
        raw, val = [], []
        for _ in range(n):
            b, s = self.char()
            raw.append(b)
            val.append(s)
        return b"".join(raw), "".join(val)

    def string(self, key: bool = False) -> tuple[bytes, str]:
        r = self.r
        if key and r.random() < 0.5:
            word = r.choice(KEY_WORDS)
            raw = word.encode().replace(b"\\", b"\\\\")
            return b'"' + raw + b'"', word
        if not key and r.random() < self.p_long:
            n = r.choice((r.randint(65, 200), r.randint(2049, 3000)))
            b, s = self.text(n)
        else:
            b, s = self.text(r.choice((0, 1, 2, 3, 5, 8, 16, 31, 33)))
        n = len(s.encode("utf-8", "surrogatepass"))
        if n > 64:
            self.counts["str_gt64"] += 1
        if n > 2048:
            self.counts["str_gt2k"] += 1
        return b'"' + b + b'"', s

    # ---- numbers ------------------------------------------------------------------------------------------------------------
    def integer(self) -> tuple[bytes, int]:
        r, c = self.r, self.r.random()
        if c < 0.08:
            v = r.choice((INT64_MIN, INT64_MAX, 0))
            self.counts[{INT64_MIN: "int64_min", INT64_MAX: "int64_max", 0: "int_zero"}[v]] += 1
            return b"%d" % v, v
        if c < 0.12:
            self.counts["int_neg_zero"] += 1
            return b"-0", 0
        nd = r.randint(1, 19)
        v = r.randrange(10 ** (nd - 1) if nd > 1 else 0, min(10**nd, INT64_MAX + 1))
        if r.random() < 0.4:
            v = -v
        self.counts["int_digits_%d" % len(str(abs(v)))] += 1
        return b"%d" % v, v

    def double(self) -> tuple[bytes, Float]:
        r = self.r
        if r.random() < 0.04:
            self.counts["float_neg_zero"] += 1
            tok = r.choice((b"-0.0", b"-0e0", b"-0.0E+5"))
            return tok, Float(tok)
        nd = r.choice((1, 2, 3, 5, 8, 15, 16, 17, 18, 19, 20, r.randint(1, 20)))
        digits = "".join(r.choice("0123456789") for _ in range(nd))
        digits = digits if digits[0] != "0" else "1" + digits[1:]
        self.counts["mant_%d" % nd] += 1
        point = r.randint(0, nd)   # digits before the point; 0: "0.ddd"
        ip, fp = (digits[:point] or "0"), digits[point:]
        tok = ("-" if r.random() < 0.4 else "") + ip + ("." + fp if fp else "")
        if not fp or r.random() < 0.6:
            e = r.choice((r.randint(-5, 5), r.randint(20, 24), -r.randint(20, 24), r.randint(300, 310), -r.randint(300, 310),
                          r.randint(320, 400), -r.randint(320, 400)))
            mark = r.choice("eE")
            sign = "-" if e < 0 else r.choice(("", "+"))
            self.counts["exp_" + mark] += 1
            self.counts["exp_sign_" + (sign or "none")] += 1
            a = abs(e)
            self.counts["exp_near22" if 20 <= a <= 24 else "exp_near308" if 300 <= a <= 310 else "exp_beyond" if a > 310 else "exp_small"] += 1
            tok += mark + sign + str(a)
        tok = tok.encode()
        return tok, Float(tok)

    # ---- values -------------------------------------------------------------------------------------------------------------
    def scalar(self) -> tuple[bytes, object, int]:
        c = self.r.random()
        if c < 0.3:
            b, v = self.string()
        elif c < 0.55:
            b, v = self.integer()
        elif c < 0.8:
            b, v = self.double()
        else:
            b, v = self.r.choice(((b"true", True), (b"false", False), (b"null", None)))
            self.counts[b.decode()] += 1
        return b, v, 1

    def array(self, items: list) -> tuple[bytes, list, int]:
        """items: (bytes, value, tokens) of the elements."""
        if not items:
            self.counts["empty_array"] += 1
        if len(items) >= WIDE:
            self.counts["wide_array"] += 1
        sep = [self.space() + b"," + self.space() for _ in range(len(items) - 1)]
        body = b"".join(x[0] + (sep[i] if i < len(sep) else b"") for i, x in enumerate(items))
        return b"[" + self.space() + body + self.space() + b"]", [x[1] for x in items], 2 + sum(x[2] for x in items) + max(len(items) - 1, 0)

    def obj(self, members: list) -> tuple[bytes, tuple, int]:
        """members: (key bytes, key str, (bytes, value, tokens)) of the members."""
        if not members:
            self.counts["empty_object"] += 1
        if len(members) >= WIDE:
            self.counts["wide_object"] += 1
        keys = [k for _, k, _ in members]
        for name, hit in (("key_empty", ""), ("key_numeric", "0")):
            if hit in keys:
                self.counts[name] += 1
        if any("/" in k for k in keys):
            self.counts["key_slash"] += 1
        if any("~" in k for k in keys):
            self.counts["key_tilde"] += 1
        if len(set(keys)) < len(keys):
            self.counts["key_dup"] += 1
        parts = [kb + self.space() + b":" + self.space() + x[0] for kb, _, x in members]
        body = b"".join(p + (self.space() + b"," + self.space() if i + 1 < len(parts) else b"") for i, p in enumerate(parts))
        toks = 2 + sum(2 + x[2] for _, _, x in members) + max(len(members) - 1, 0)
        return b"{" + self.space() + body + self.space() + b"}", ("object", [(k, x[1]) for _, k, x in members]), toks

    def member_key(self, keys: list) -> tuple[bytes, str]:
        """keys: the (bytes, str) keys of the object so far; now and then one of them again."""
        kk = self.r.choice(keys) if keys and self.r.random() < 0.08 else self.string(key=True)
        keys.append(kk)
        return kk

    def value(self, level: int, budget: list) -> tuple[bytes, object, int]:
        """A random value that opens its containers at `level` (the root is 1); budget[0] bounds the elements left."""
        r = self.r
        c = r.random()
        if budget[0] > 0 and level <= MAX_ARRAY_LEVEL and r.random() < self.p_wide / level:
            n = r.randint(WIDE, WIDE + 200)
            budget[0] -= n
            if r.random() < 0.5:
                return self.array([self.scalar() for _ in range(n)])
            keys = []
            return self.obj([(*self.member_key(keys), self.scalar()) for _ in range(n)])
        if budget[0] <= 0 or c < 0.45 or level > MAX_OBJECT_LEVEL:
            return self.scalar()
        if c < 0.72 and level <= MAX_ARRAY_LEVEL:
            n = r.choice((0, 1, 1, 2, 3, 4, 6))
            budget[0] -= n
            return self.array([self.value(level + 1, budget) for _ in range(n)])
        n = r.choice((0, 1, 1, 2, 3, 4, 6))
        budget[0] -= n
        members, keys = [], []
        for _ in range(n):
            members.append((*self.member_key(keys), self.value(level + 1, budget)))
        return self.obj(members)

    def deep(self, level: int, limit_array: bool) -> tuple[bytes, object, int]:
        """A chain of containers down to the deepest level the walk accepts, with small siblings on the way."""
        r = self.r
        last = MAX_ARRAY_LEVEL if limit_array else MAX_OBJECT_LEVEL
        if level == last:
            self.counts["max_depth_array" if limit_array else "max_depth_object"] += 1
            inner = [self.scalar()]
            return self.array(inner) if limit_array else self.obj([(*self.string(key=True), inner[0])])
        child = self.deep(level + 1, limit_array)
        sib = [self.scalar()] if r.random() < 0.2 else []
        if level >= MAX_ARRAY_LEVEL or r.random() < 0.5:   # only objects may sit at level 100
            mem = [(*self.string(key=True), child)] + [(*self.string(key=True), s) for s in sib]
            r.shuffle(mem)
            return self.obj(mem)
        items = [child] + sib
        r.shuffle(items)
        return self.array(items)

    def root(self, budget: int = 60) -> tuple[bytes, object, int]:
        r = self.r
        if r.random() < self.p_deep:
            return self.deep(1, r.random() < 0.5)
        while True:
            b, v, t = self.value(1, [budget])
            if b[:1] in b"{[" and t == 2:   # a root-level empty container is a TAPE_ERROR document
                continue
            if t == 1 and r.random() < 0.7:   # root scalars: about one document in five
                continue
            return b, v, t

    def document(self, budget: int = 60) -> Doc:
        b, v, t = self.root(budget)
        self.counts["documents"] += 1
        if not isinstance(v, (list, tuple)):
            self.counts["root_scalar"] += 1
        return Doc(b, v, list(paths(v)), t)

    # ---- templated documents: a few shapes with optional keys and varying value types ----------------------------------------
    def template(self, level: int = 1):
        r = self.r
        if level > 3 or (level > 1 and r.random() < 0.4):
            return ("leaf", r.sample(["str", "int", "float", "bool", "null", "arr"], r.randint(1, 3)))
        if level > 1 and r.random() < 0.2:
            return ("array", self.template(level + 1))
        keys = list(dict.fromkeys(r.choice(KEY_WORDS) for _ in range(r.randint(1, 6))))
        return ("object", [(k, r.random() < 0.7, self.template(level + 1)) for k in keys])

    def instance(self, t) -> tuple[bytes, object, int]:
        r = self.r
        if t[0] == "leaf":
            kind = r.choice(t[1])
            if kind == "str":
                return (*self.string(), 1)
            if kind == "int":
                return (*self.integer(), 1)
            if kind == "float":
                return (*self.double(), 1)
            if kind == "arr":
                return self.array([self.scalar() for _ in range(r.randint(0, 4))])
            if kind == "null":
                return b"null", None, 1
            return (b"true", True, 1) if r.random() < 0.5 else (b"false", False, 1)
        if t[0] == "array":
            return self.array([self.instance(t[1]) for _ in range(r.randint(0, 4))])
        members = [(b'"' + k.encode().replace(b"\\", b"\\\\") + b'"', k, self.instance(sub)) for k, required, sub in t[1] if required or r.random() < 0.6]
        return self.obj(members)

    def templated(self, n_docs: int, n_shapes: int = 4) -> list[Doc]:
        shapes = [self.template() for _ in range(n_shapes)]
        out = []
        while len(out) < n_docs:
            b, v, t = self.instance(self.r.choice(shapes))
            if t == 2:
                continue
            self.counts["templated"] += 1
            out.append(Doc(b, v, list(paths(v)), t))
        return out


def paths(v, prefix=()):
    """Every location of a value as a list of reference tokens (str for a member, int for an element).  Of repeated keys only
    the first is a location: a pointer names the first member with its key."""
    yield list(prefix)
    if isinstance(v, tuple):
        seen = set()
        for k, x in v[1]:
            if k not in seen:
                seen.add(k)
                yield from paths(x, prefix + (k,))
    elif isinstance(v, list):
        for i, x in enumerate(v):
            yield from paths(x, prefix + (i,))


def pointer(path) -> bytes:
    """The JSON Pointer (RFC 6901) of a path: '~' as '~0', '/' as '~1', keys as raw UTF-8."""
    return b"".join(b"/" + (str(t).encode("utf-8", "surrogatepass").replace(b"~", b"~0").replace(b"/", b"~1")) for t in path)


def stream(docs: list[Doc], r: random.Random, mode: str, counts: Counter | None = None) -> tuple[bytes, list[int]]:
    """The documents framed as one stream; returns (bytes, offset of every document's first byte).  mode: 'lf', 'crlf' (NDJSON,
    with blank lines now and then) or 'concat' (no separator where the grammar needs none: after '}', ']' or '"' before a
    document that starts with '{', '[' or '"'; otherwise whitespace).  A root scalar is always followed by whitespace."""
    counts = Counter() if counts is None else counts
    out, starts, pos = [], [], 0
    for i, d in enumerate(docs):
        if mode == "concat" and i == 0 and r.random() < 0.5:
            lead = bytes(r.choice(WS) for _ in range(r.randint(1, 3)))
            out.append(lead)
            pos += len(lead)
        starts.append(pos)
        out.append(d.data)
        pos += len(d.data)
        nxt, last = (docs[i + 1].data[:1] if i + 1 < len(docs) else b""), d.data[-1:]
        if mode in ("lf", "crlf"):
            nl = b"\n" if mode == "lf" else b"\r\n"
            sep = nl * (2 if r.random() < 0.05 else 1)
            counts["sep_" + mode] += 1
            if len(sep) > len(nl):
                counts["blank_line"] += 1
        elif nxt and last in (b"}", b"]", b'"') and nxt in (b"{", b"[", b'"') and r.random() < 0.7:
            sep = b""
            counts["concat_after_" + {b"}": "brace", b"]": "bracket", b'"': "quote"}[last]] += 1
        elif not nxt and last in (b"}", b"]") and r.random() < 0.5:
            sep = b""
        else:
            sep = bytes(r.choice(WS) for _ in range(r.randint(1, 3)))
        out.append(sep)
        pos += len(sep)
    return b"".join(out), starts
