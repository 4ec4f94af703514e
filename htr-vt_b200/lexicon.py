"""Word lexicon for the lexicon-constrained CTC prefix beam search (csrc/prefix_beam.cu, LEX instantiation).

`Lexicon.from_words(words, converter, word_chars=None)` / `Lexicon.from_file(path, converter, word_chars=None)` pack a
word list over `converter.character` into a trie the kernel walks, on the current device.  Every word of a decoded
line then comes from the list (Scheidl et al. 2018, "Word Beam Search", "Words" mode).

Word characters are the characters of the kept words by default (`word_chars=` overrides, "" included); every other
class - the space, punctuation, ids beyond the alphabet - is free.  A labelling is accepted when every maximal run of
word characters in it is a lexicon word.  Words are stripped of surrounding whitespace; blank ones are ignored and
duplicates merged.  A word with a character outside the alphabet, or with a free character (only possible with an
explicit `word_chars`), is skipped and counted in `n_skipped`.

`Lexicon.on_host(words, converter, word_chars=None)` builds the same object with its tensors left on the host: a word
LM (wordlm.py) can then be packed against it and inspected on a machine without a GPU; the kernels refuse it.  Every
lexicon also keeps its host-side trie, its kept words and the node each word ends at, which a word LM numbers its
tokens and builds its per-node tables from (one vectorised walk: about a tenth of the packing time for 10^5 words).

Trie (CSR): node 0 = root, nodes numbered breadth first; first int32 [n_nodes + 1], the edges of node n are
first[n] .. first[n + 1] - 1 with label int32 (class id) sorted ascending and child int32; word_end uint8 [n_nodes].
"""
import numpy as np
import torch

from ._lib import HtrvtError


def pack_trie(words):
    """words: iterable of non-empty class-id tuples -> (first int32 [N + 1], label int32 [E], child int32 [E],
    word_end uint8 [N]), N nodes (root 0, breadth-first order), E = N - 1 edges, labels sorted within a node."""
    kids = [{}]                                           # node -> {label: child}
    end = [False]
    for w in words:
        n = 0
        for c in w:
            nxt = kids[n].get(c)
            if nxt is None:
                nxt = len(kids)
                kids[n][c] = nxt
                kids.append({})
                end.append(False)
            n = nxt
        end[n] = True
    order, new_id = [0], {0: 0}                           # breadth first, children by label
    for n in order:
        for c in sorted(kids[n]):
            new_id[kids[n][c]] = len(order)
            order.append(kids[n][c])
    first = np.zeros(len(order) + 1, dtype=np.int32)
    label, child = [], []
    for i, n in enumerate(order):
        for c in sorted(kids[n]):
            label.append(c)
            child.append(new_id[kids[n][c]])
        first[i + 1] = len(label)
    word_end = np.array([end[n] for n in order], dtype=np.uint8)
    return first, np.array(label, dtype=np.int32), np.array(child, dtype=np.int32), word_end


def check_trie(first, label, child, word_end):
    """The kernel's contract on a packed trie; ValueError when it does not hold."""
    N, E = len(word_end), len(label)
    if N < 1 or len(first) != N + 1 or first[0] != 0 or first[-1] != E or len(child) != E:
        raise ValueError("trie: array sizes do not match")
    if (np.diff(first) < 0).any():
        raise ValueError("trie: first[] is not monotone")
    if E and (child.min() < 1 or child.max() >= N or label.min() < 1):
        raise ValueError("trie: child or label out of range")
    starts = np.zeros(E + 1, dtype=bool)
    starts[first] = True
    if (~starts[np.flatnonzero(np.diff(label) <= 0) + 1]).any():
        raise ValueError("trie: the labels of a node are not strictly ascending")


def trie_nodes(first, label, child, seqs):
    """The node each class-id sequence of seqs (every one spelled by the trie) ends at, int64 [len(seqs)]: one
    vectorised walk, a character position at a time; edges are found by their (parent, label) key, which the CSR
    layout keeps in ascending order."""
    n = len(seqs)
    lens = np.array([len(q) for q in seqs], dtype=np.int64)
    cur = np.zeros(n, dtype=np.int64)
    if not n or not len(label):
        return cur
    width = int(label.max()) + 1
    key = np.repeat(np.arange(len(first) - 1, dtype=np.int64), np.diff(first)) * width + label
    pad = np.zeros((n, int(lens.max())), dtype=np.int64)
    for i, q in enumerate(seqs):
        pad[i, : len(q)] = q
    for k in range(pad.shape[1]):
        m = lens > k
        cur[m] = child[np.searchsorted(key, cur[m] * width + pad[m, k])]
    return cur


class Lexicon(object):
    """A word lexicon on the device.  Attributes: n_words, n_nodes, n_skipped, word_chars (the word characters in
    class order), device, and the device tensors first, label, child (int32), word_end, is_word (uint8; is_word has
    one entry per class of converter.character).  On the host: words (the kept words, sorted: a word LM numbers them
    in this order), word_node (int64 [n_words]: the trie node each of them ends at) and trie (first, label, child,
    word_end as numpy arrays)."""

    def __init__(self, first, label, child, word_end, is_word, n_words, n_skipped, word_chars, device, words=(),
                 word_node=()):
        self.n_words = n_words
        self.n_nodes = int(len(word_end))
        self.n_skipped = n_skipped
        self.word_chars = word_chars
        self.device = device
        self.words = list(words)
        self.word_node = np.asarray(word_node, dtype=np.int64)
        self.trie = (np.asarray(first, dtype=np.int32), np.asarray(label, dtype=np.int32),
                     np.asarray(child, dtype=np.int32), np.asarray(word_end, dtype=np.uint8))
        # label / child keep at least one element: an empty tensor has no data pointer, and the kernel never reads it
        pad = lambda a: a if len(a) else np.zeros(1, dtype=a.dtype)   # noqa: E731
        self.first = torch.from_numpy(np.ascontiguousarray(first, dtype=np.int32)).to(device)
        self.label = torch.from_numpy(pad(np.ascontiguousarray(label, dtype=np.int32))).to(device)
        self.child = torch.from_numpy(pad(np.ascontiguousarray(child, dtype=np.int32))).to(device)
        self.word_end = torch.from_numpy(np.ascontiguousarray(word_end, dtype=np.uint8)).to(device)
        self.is_word = torch.from_numpy(np.ascontiguousarray(is_word, dtype=np.uint8)).to(device)

    @staticmethod
    def _pack(words, converter, word_chars):
        """-> (host_tables' tuple, kept words, the node each kept word ends at)"""
        cls_of = {ch: c for c, ch in enumerate(converter.character) if c >= 1}
        uniq = sorted(set(w.strip() for w in words) - {""})
        in_alpha = [w for w in uniq if all(ch in cls_of for ch in w)]
        wc = set("".join(in_alpha)) if word_chars is None else set(word_chars)
        is_word = np.zeros(len(converter.character), dtype=np.uint8)
        for ch, c in cls_of.items():
            is_word[c] = ch in wc
        kept = [w for w in in_alpha if all(ch in wc for ch in w)]
        seqs = [tuple(cls_of[ch] for ch in w) for w in kept]
        first, label, child, word_end = pack_trie(seqs)
        check_trie(first, label, child, word_end)
        chars = "".join(converter.character[c] for c in range(1, len(converter.character)) if is_word[c])
        tables = (first, label, child, word_end, is_word, len(kept), len(uniq) - len(kept), chars)
        return tables, kept, trie_nodes(first, label, child, seqs)

    @staticmethod
    def host_tables(words, converter, word_chars=None):
        """Pack on the host: -> (first, label, child, word_end, is_word, n_words, n_skipped, word_chars)."""
        return Lexicon._pack(words, converter, word_chars)[0]

    @staticmethod
    def _file_pack(path, converter, word_chars):
        with open(path, "r", encoding="utf-8") as fh:
            p = Lexicon._pack(fh.read().splitlines(), converter, word_chars)
        if not p[0][5]:
            raise ValueError("lexicon %s: no usable word (every line blank, or every word skipped)" % path)
        return p

    @classmethod
    def _on_device(cls, packed):
        if not torch.cuda.is_available():
            raise HtrvtError("Lexicon lives on a CUDA device (there is no CPU fallback)")
        tables, kept, nodes = packed
        return cls(*tables, device=torch.device("cuda", torch.cuda.current_device()), words=kept, word_node=nodes)

    @classmethod
    def on_host(cls, words, converter, word_chars=None):
        """from_words with every tensor left on the host: for building a word LM's tables without a GPU (the kernels
        refuse a lexicon that does not live on the log-probs' device)."""
        tables, kept, nodes = cls._pack(words, converter, word_chars)
        return cls(*tables, device=torch.device("cpu"), words=kept, word_node=nodes)

    @classmethod
    def from_words(cls, words, converter, word_chars=None):
        """Pack a list of words over converter.character (see the module doc) onto the current CUDA device.
        HtrvtError without a CUDA device (there is no CPU fallback)."""
        return cls._on_device(cls._pack(words, converter, word_chars))

    @staticmethod
    def file_tables(path, converter, word_chars=None):
        """host_tables of a UTF-8 file, one word per line; ValueError when no usable word remains."""
        return Lexicon._file_pack(path, converter, word_chars)[0]

    @classmethod
    def from_file(cls, path, converter, word_chars=None):
        """from_words on the lines of a UTF-8 file; ValueError when no usable word remains."""
        return cls._on_device(cls._file_pack(path, converter, word_chars))
