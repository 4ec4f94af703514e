"""Character n-gram language model for the LM-fused CTC prefix beam search (csrc/prefix_beam.cu, LM instantiation).

`CharNGramLM.from_arpa(path, converter, space_token="<space>")` reads a standard ARPA file (the text format KenLM's
`lmplz` and SRILM write) whose tokens are the characters of `converter.character`, the space written as `space_token`
(ARPA tokens are whitespace-separated), and builds the device table the kernel queries once, on the current device.

Query semantics (ARPA backoff): log10 p(w | h) is the listed prob of (h, w) if listed, else bow(h) + log10 p(w | h[1:])
with bow(h) = 0 for an unlisted context; at the unigram level an unlisted w takes <unk>'s prob (-100, KenLM's default,
when the file lists no <unk>).  Alphabet characters the LM does not list as unigrams, and class ids beyond the
alphabet, are <unk>, as predicted tokens and in the context.  An n-gram with a token outside the alphabet and the
specials can never be queried and is dropped.  Sentences start in context <s>; <s> itself is never scored.

Table: open addressing with linear probing, 32-byte slots {u64 lo, u64 hi, f32 log10 p, f32 log10 bow, u64 pad}.  The
key holds the n-gram exactly - its tokens, LAST token first, as 16-bit fields (token id + 1) - so a hash collision
never produces a false match; lo == 0 marks an empty slot; the slot count is a power of two at least twice the number
of n-grams.  Values are float32, as KenLM stores them.
"""
import math

import numpy as np
import torch

from ._lib import HtrvtError

MAX_ORDER = 8
UNK, BOS, EOS = 0, 1, 2                     # token ids of <unk>, <s>, </s> (the kernel's constants)
UNK_LOG10P = -100.0                         # <unk>'s log10 prob when the file lists none (KenLM's default)
_SPECIAL = {"<unk>": UNK, "<s>": BOS, "</s>": EOS}


def parse_arpa(path):
    """-> (order, counts, grams): grams[k - 1] = list of (token tuple, log10 p, log10 bow) of the k-grams, values as
    float64 parsed from the text.  ValueError on a malformed file: no \\data\\ section or counts, an order above 8, a
    missing or misplaced \\k-grams: section, counts that do not match, a line with the wrong number of fields or a value
    that is not a finite number, or no \\end\\."""
    with open(path, "r", encoding="utf-8") as fh:
        lines = fh.read().splitlines()
    i, n = 0, len(lines)
    while i < n and lines[i].strip() != "\\data\\":
        i += 1
    if i == n:
        raise ValueError("ARPA: no \\data\\ section")
    i += 1
    counts = {}
    while i < n:
        s = lines[i].strip()
        if s.startswith("ngram "):
            k, _, v = s[6:].partition("=")
            try:
                counts[int(k)] = int(v)
            except ValueError:
                raise ValueError("ARPA: bad count line %r" % s)
        elif s:
            break
        i += 1
    if not counts:
        raise ValueError("ARPA: no n-gram counts")
    order = max(counts)
    if sorted(counts) != list(range(1, order + 1)) or min(counts.values()) < 0:
        raise ValueError("ARPA: counts must list orders 1..N once each")
    if order > MAX_ORDER:
        raise ValueError("ARPA: order %d is above the supported %d" % (order, MAX_ORDER))
    grams = []
    for k in range(1, order + 1):
        while i < n and not lines[i].strip():
            i += 1
        if i == n or lines[i].strip() != "\\%d-grams:" % k:
            raise ValueError("ARPA: missing \\%d-grams: section" % k)
        i += 1
        out = []
        while i < n:
            s = lines[i].strip()
            if not s:
                i += 1
                continue
            if s.startswith("\\"):
                break
            f = s.split()
            if len(f) not in (k + 1, k + 2):
                raise ValueError("ARPA: line %d has %d fields for a %d-gram" % (i + 1, len(f), k))
            try:
                p = float(f[0])
                b = float(f[k + 1]) if len(f) == k + 2 else 0.0
            except ValueError:
                raise ValueError("ARPA: line %d holds a value that is not a number" % (i + 1))
            toks = tuple(f[1:k + 1])
            if not math.isfinite(p) and toks == ("<s>",):
                p = -99.0                   # <s> is never predicted; some writers give it -inf
            if not (math.isfinite(p) and math.isfinite(b)):
                raise ValueError("ARPA: line %d holds a non-finite value" % (i + 1))
            out.append((toks, p, b))
            i += 1
        if len(out) != counts[k]:
            raise ValueError("ARPA: \\data\\ announces %d %d-grams, the section holds %d" % (counts[k], k, len(out)))
        grams.append(out)
    while i < n and not lines[i].strip():
        i += 1
    if i == n or lines[i].strip() != "\\end\\":
        raise ValueError("ARPA: missing \\end\\")
    return order, [counts[k] for k in range(1, order + 1)], grams


def lm_hash(lo, hi):
    """The kernel's slot hash (csrc/prefix_beam.cu::lm_hash) on uint64 arrays."""
    with np.errstate(over="ignore"):
        h = lo * np.uint64(0x9E3779B97F4A7C15) + hi * np.uint64(0xC2B2AE3D27D4EB4F)
        h ^= h >> np.uint64(31)
        h *= np.uint64(0xBF58476D1CE4E5B9)
        return h ^ (h >> np.uint64(29))


def pack_keys(tokens, bits=16):
    """tokens int [N, k] (token ids, first to last) -> (lo, hi) uint64 [N]: last token first, bits-wide fields of
    id + 1, 64 // bits of them per word (16: the character LM's 4 + 4 fields; 21: the word LM's 3 + 3)."""
    tokens = np.asarray(tokens, dtype=np.int64)
    N, k = tokens.shape
    per = 64 // bits
    if k > 2 * per or (tokens.size and (tokens.min() < 0 or tokens.max() > (1 << bits) - 2)):
        raise ValueError("n-gram keys hold at most %d token ids in 0..%d" % (2 * per, (1 << bits) - 2))
    lo = np.zeros(N, dtype=np.uint64)
    hi = np.zeros(N, dtype=np.uint64)
    for f in range(k):
        v = (tokens[:, k - 1 - f] + 1).astype(np.uint64) << np.uint64(bits * (f % per))
        if f < per:
            lo |= v
        else:
            hi |= v
    return lo, hi


def pack_table(lo, hi, logp, bow):
    """Open-addressing table of the (distinct) keys: uint64 [slots, 4] rows (lo, hi, (f32 p, f32 bow), 0)."""
    n = len(lo)
    slots = 2
    while slots < 2 * n:
        slots *= 2
    mask = np.uint64(slots - 1)
    owner = np.full(slots, -1, dtype=np.int64)
    pos = (lm_hash(lo, hi) & mask).astype(np.int64)
    pending = np.arange(n)
    while pending.size:                                   # every pending key tries its slot; per free slot the lowest
        p = pos[pending]                                  # key index wins, everyone else moves one slot on
        free = owner[p] < 0
        cand, cp = pending[free], p[free]
        won = np.zeros(pending.size, dtype=bool)
        if cand.size:
            slot_u, first = np.unique(cp, return_index=True)
            owner[slot_u] = cand[first]
            won[np.flatnonzero(free)[first]] = True
        pending = pending[~won]
        pos[pending] = (pos[pending] + 1) & (slots - 1)
    table = np.zeros((slots, 4), dtype=np.uint64)
    used = owner >= 0
    o = owner[used]
    table[used, 0] = lo[o]
    table[used, 1] = hi[o]
    vals = np.zeros((slots, 2), dtype=np.float32)
    vals[used, 0] = np.asarray(logp, dtype=np.float64)[o].astype(np.float32)
    vals[used, 1] = np.asarray(bow, dtype=np.float64)[o].astype(np.float32)
    table[:, 2] = vals.view(np.uint64)[:, 0]
    return table


def table_find(table, lo, hi):
    """Host lookup in a packed table (the kernel's probe): slot index per key, -1 when absent."""
    slots = table.shape[0]
    mask = np.uint64(slots - 1)
    lo = np.asarray(lo, dtype=np.uint64)
    hi = np.asarray(hi, dtype=np.uint64)
    pos = (lm_hash(lo, hi) & mask).astype(np.int64)
    res = np.full(lo.shape, -1, dtype=np.int64)
    todo = np.arange(lo.size)
    for _ in range(slots):
        if not todo.size:
            break
        p = pos[todo]
        hit = (table[p, 0] == lo[todo]) & (table[p, 1] == hi[todo])
        res[todo[hit]] = p[hit]
        empty = table[p, 0] == 0
        todo = todo[~(hit | empty)]
        pos[todo] = (pos[todo] + 1) % slots
    return res


def table_values(table, idx):
    """(log10 p, log10 bow) float32 of the slots idx."""
    v = table[idx, 2].view(np.float32).reshape(-1, 2)
    return v[:, 0], v[:, 1]


class CharNGramLM(object):
    """A character n-gram LM on the device.  Attributes: order, counts (the file's n-gram counts per order), slots,
    table (int64 [slots, 4] device tensor, the packed slots), token_map (int32 device tensor: class id -> token id),
    kept (n-grams in the table), device."""

    def __init__(self, order, counts, table, token_map, kept, device):
        self.order = order
        self.counts = counts
        self.slots = int(table.shape[0])
        self.kept = kept
        self.device = device
        self.table = torch.from_numpy(table.view(np.int64)).to(device)
        self.token_map = torch.from_numpy(np.asarray(token_map, dtype=np.int32)).to(device)

    @staticmethod
    def host_tables(path, converter, space_token="<space>"):
        """Parse and pack on the host: -> (order, counts, packed table, token map, n-grams kept)."""
        order, counts, grams = parse_arpa(path)
        chars = list(converter.character[1:])             # class id c >= 1 <-> chars[c - 1]
        listed = set(t[0] for t, _, _ in grams[0])
        tok_of = dict(_SPECIAL)                           # ARPA token -> token id
        tmap = [UNK] * len(converter.character)
        for c, ch in enumerate(chars, start=1):
            word = space_token if ch == " " else ch
            if word in _SPECIAL or word not in listed:
                continue                                  # not in the LM: scored as <unk>
            if word not in tok_of:
                tok_of[word] = len(tok_of)
            tmap[c] = tok_of[word]
        entries = {}                                      # token-id tuple -> (log10 p, log10 bow); a repeat wins
        for gk in grams:
            for toks, p, b in gk:
                ids = tuple(tok_of.get(t, -1) for t in toks)
                if min(ids) >= 0:                         # else: a token outside the alphabet, never queried
                    entries[ids] = (p, b)
        entries.setdefault((UNK,), (UNK_LOG10P, 0.0))
        lo, hi, ps, bs = [], [], [], []
        for k in range(1, order + 1):
            kk = [key for key in entries if len(key) == k]
            l, h = pack_keys(np.array(kk, dtype=np.int64).reshape(-1, k))
            lo.append(l)
            hi.append(h)
            ps.extend(entries[key][0] for key in kk)
            bs.extend(entries[key][1] for key in kk)
        lo, hi = np.concatenate(lo), np.concatenate(hi)
        table = pack_table(lo, hi, np.array(ps, dtype=np.float64), np.array(bs, dtype=np.float64))
        return order, counts, table, tmap, len(lo)

    @classmethod
    def from_arpa(cls, path, converter, space_token="<space>"):
        """Load an ARPA file over converter.character (see the module doc) onto the current CUDA device.  ValueError
        for a malformed file; HtrvtError without a CUDA device (there is no CPU fallback)."""
        order, counts, table, tmap, kept = cls.host_tables(path, converter, space_token)
        if not torch.cuda.is_available():
            raise HtrvtError("CharNGramLM lives on a CUDA device (there is no CPU fallback)")
        return cls(order, counts, table, tmap, kept, torch.device("cuda", torch.cuda.current_device()))
