"""Word n-gram language model for the lexicon-constrained CTC prefix beam search (csrc/prefix_beam.cu, word-LM
instantiation; Scheidl et al. 2018, "Word Beam Search", "NGrams" mode).

`WordNGramLM.from_arpa(path, lexicon)` reads a standard ARPA file (lm.parse_arpa) whose tokens are words - what KenLM
builds from plain text, which it splits on whitespace - and packs it against a `Lexicon`, on the lexicon's device.

Tokens of a labelling are its words: the maximal runs of word characters, as the lexicon defines them; free classes
are no tokens.  With words w1 .. wm the search ranks and returns

    fused = ctc + sum_i [alpha ln10 log10 p(w_i | <s> w_1 .. w_i-1) + beta] + alpha ln10 log10 p(</s> | <s> w_1 .. w_m)

with ARPA backoff exactly as lm.py (float32 values summed in float64).  While an entry is inside a word whose spelled
part is s, its ranking adds alpha ln10 smear(s), the largest unigram log10 prob of the lexicon words that start with s
(flashlight's "max" smearing), so that a half-spelled word does not rank as if it cost nothing.

Token ids: <unk> = 0, <s> = 1, </s> = 2, lexicon word i (lexicon.words order) = 3 + i.  A lexicon word the file does
not list as a unigram is <unk>; an n-gram with a token that is neither a listed lexicon word nor a special can never be
queried and is dropped.  Table: lm.py's 32-byte slots and hash with 21-bit key fields (lm.pack_keys(..., bits=21)), so
keys hold up to 6 tokens of ids below 2^21 - 1.  Per trie node: node_tok (int32, the token of the word ending there,
-1 where none ends) and smear (float32).
"""
import numpy as np
import torch

from .lm import UNK, UNK_LOG10P, _SPECIAL, pack_keys, pack_table, parse_arpa

MAX_ORDER = 6
KEY_BITS = 21
MAX_WORDS = (1 << KEY_BITS) - 1 - 3          # token ids 3 + i stay below 2^21 - 1


def node_smear(first, child, node_p):
    """smear float32 [n_nodes]: node_p (the unigram log10 prob of the word ending at a node, -inf elsewhere) maxed
    over each node's subtree.  Breadth-first numbering gives every trie level a contiguous id range after its parent
    level's, so one pass over the levels, deepest first, carries every maximum up to the root."""
    n = len(first) - 1
    parent = np.zeros(n, dtype=np.int64)
    parent[child] = np.repeat(np.arange(n, dtype=np.int64), np.diff(first))
    levels, a, b = [], 0, 1                                   # nodes a .. b - 1 form one level
    while first[b] > first[a]:
        kids = child[first[a]:first[b]]
        levels.append(kids)
        a, b = int(kids.min()), int(kids.max()) + 1
    s = np.asarray(node_p, dtype=np.float32).copy()
    for kids in reversed(levels):
        np.maximum.at(s, parent[kids], s[kids])
    return s


class WordNGramLM(object):
    """A word n-gram LM bound to one Lexicon.  Attributes: order, counts (the file's n-gram counts per order), slots,
    kept (n-grams in the table), n_dropped (n-grams dropped), n_unk_words (lexicon words scored as <unk>), lexicon,
    device, and the tensors table (int64 [slots, 4]), node_tok (int32 [n_nodes]), smear (float32 [n_nodes])."""

    def __init__(self, order, counts, table, node_tok, smear, kept, n_dropped, n_unk_words, lexicon):
        self.order = order
        self.counts = counts
        self.slots = int(table.shape[0])
        self.kept = kept
        self.n_dropped = n_dropped
        self.n_unk_words = n_unk_words
        self.lexicon = lexicon
        self.device = lexicon.device
        self.table = torch.from_numpy(table.view(np.int64)).to(self.device)
        self.node_tok = torch.from_numpy(np.ascontiguousarray(node_tok, dtype=np.int32)).to(self.device)
        self.smear = torch.from_numpy(np.ascontiguousarray(smear, dtype=np.float32)).to(self.device)

    @staticmethod
    def host_tables(path, lexicon):
        """Parse and pack on the host: -> (order, counts, packed table, node_tok, smear, n-grams kept, n_dropped,
        n_unk_words).  ValueError for a malformed file, an order outside 1..6 or a lexicon of more than 2^21 - 4
        words."""
        order, counts, grams = parse_arpa(path)
        if not 1 <= order <= MAX_ORDER:
            raise ValueError("word LM: order %d is outside 1..%d" % (order, MAX_ORDER))
        if lexicon.n_words > MAX_WORDS:
            raise ValueError("word LM: %d lexicon words, the 21-bit keys hold %d" % (lexicon.n_words, MAX_WORDS))
        listed = set(t[0] for t, _, _ in grams[0])
        tok_of = dict(_SPECIAL)                                   # ARPA token -> token id
        word_tok = np.full(len(lexicon.words), UNK, dtype=np.int64)
        for i, w in enumerate(lexicon.words):
            if w in listed and w not in _SPECIAL:
                tok_of[w] = word_tok[i] = 3 + i
        entries, n_dropped = {}, 0                                # token-id tuple -> (log10 p, log10 bow); repeat wins
        for gk in grams:
            for toks, p, b in gk:
                ids = tuple(tok_of.get(t, -1) for t in toks)
                if min(ids) >= 0:
                    entries[ids] = (p, b)
                else:
                    n_dropped += 1
        entries.setdefault((UNK,), (UNK_LOG10P, 0.0))
        lo, hi, ps, bs = [], [], [], []
        for k in range(1, order + 1):
            kk = [key for key in entries if len(key) == k]
            l, h = pack_keys(np.array(kk, dtype=np.int64).reshape(-1, k), bits=KEY_BITS)
            lo.append(l)
            hi.append(h)
            ps.extend(entries[key][0] for key in kk)
            bs.extend(entries[key][1] for key in kk)
        lo, hi = np.concatenate(lo), np.concatenate(hi)
        table = pack_table(lo, hi, np.array(ps, dtype=np.float64), np.array(bs, dtype=np.float64))
        first, _, child, word_end = lexicon.trie
        node_tok = np.full(len(word_end), -1, dtype=np.int32)
        node_tok[lexicon.word_node] = word_tok
        unigram = np.array([entries[(t,)][0] for t in word_tok.tolist()], dtype=np.float64).astype(np.float32)
        node_p = np.full(len(word_end), -np.inf, dtype=np.float32)
        node_p[lexicon.word_node] = unigram
        smear = node_smear(first, child, node_p)
        n_unk = int((word_tok == UNK).sum())
        return order, counts, table, node_tok, smear, len(lo), n_dropped, n_unk

    @classmethod
    def from_arpa(cls, path, lexicon):
        """Load an ARPA file of words (see the module doc) against lexicon, onto the lexicon's device."""
        return cls(*cls.host_tables(path, lexicon), lexicon=lexicon)
