"""A word n-gram language model in ARPA format, uploaded once to the GPU for the prefix beam search
(``CTCDecoder.decode(..., lm=)`` / ``decode_nbest(..., lm=)``; include/e2e_ctc.h, e2e_ctc_ngram).

The n-grams go into one open-addressing table on the device, keyed by the whole n-gram and built by the library's insert
kernel, so a lookup costs a few probes of a table that stays in L2 for small models and its result does not depend on
the order the n-grams were inserted in.  The lexicon (a trie over the characters of the vocabulary's spellings) depends on
the decoder's labels, case folding and word marker; it is built on first use for each and kept with the model.

Labels are either characters (``" "`` separates words) or sub-word units with a word marker (SentencePiece's ``"\u2581"``):
:func:`label_kinds` sorts the latter into continuations, word starts and boundaries (include/e2e_ctc.h,
e2e_ctc_ngram_tokens).
"""
import ctypes
import math

import torch

from .. import _lib

#: the reference builds KenLM with KENLM_MAX_ORDER = 6
MAX_ORDER = 6
#: what KenLM substitutes when a model has no <unk>
UNK_LOG10_PROB = -100.0
_SPECIAL = ("<s>", "</s>", "<unk>")
# first bytes of a KenLM binary model
_KENLM_MAGIC = b"mmap lm "


def _value(field, path, lineno):
    try:
        v = float(field)
    except ValueError:
        raise ValueError("%s:%d: %r is not a number" % (path, lineno, field)) from None
    if not math.isfinite(v):
        raise ValueError("%s:%d: non-finite value %r" % (path, lineno, field))
    return v


def parse_arpa(path):
    """``(vocab, ngrams)`` of a text ARPA file: ``vocab`` the unigrams' words in file order, ``ngrams`` a list over orders
    1..N of dicts ``{tuple of words: (log10 prob, log10 backoff)}``.  Raises ``ValueError`` on a malformed file."""
    with open(path, "rb") as f:
        raw = f.read()
    if raw.startswith(_KENLM_MAGIC):
        raise ValueError("%s is a binary KenLM model; only text ARPA files are read" % path)
    try:
        lines = raw.decode("utf-8").splitlines()
    except UnicodeDecodeError:
        raise ValueError("%s is not a UTF-8 text ARPA file" % path) from None
    i, n = 0, len(lines)
    while i < n and lines[i].strip() != "\\data\\":
        i += 1
    if i == n:
        raise ValueError("%s: no \\data\\ section" % path)
    i += 1
    counts = {}
    while i < n:
        s = lines[i].strip()
        if s.startswith("ngram "):
            k, _, c = s[6:].partition("=")
            try:
                counts[int(k)] = int(c)
            except ValueError:
                raise ValueError("%s:%d: malformed count line %r" % (path, i + 1, s)) from None
        elif s:
            break
        i += 1
    if not counts:
        raise ValueError("%s: no n-gram counts in \\data\\" % path)
    order = max(counts)
    if order > MAX_ORDER:
        raise ValueError("%s: order %d above %d" % (path, order, MAX_ORDER))
    if sorted(counts) != list(range(1, order + 1)):
        raise ValueError("%s: counts for orders %s" % (path, sorted(counts)))
    ngrams = [dict() for _ in range(order)]
    vocab = []
    seen = set()
    ended = False
    while i < n:
        s = lines[i].strip()
        i += 1
        if not s:
            continue
        if s == "\\end\\":
            ended = True
            break
        if not (s.startswith("\\") and s.endswith("-grams:")):
            raise ValueError("%s:%d: expected a \\k-grams: header, got %r" % (path, i, s))
        try:
            k = int(s[1:-7])
        except ValueError:
            raise ValueError("%s:%d: malformed section header %r" % (path, i, s)) from None
        if k not in counts or k in seen:
            raise ValueError("%s:%d: unexpected section %r" % (path, i, s))
        seen.add(k)
        table = ngrams[k - 1]
        while i < n:
            s = lines[i].strip()
            if not s:
                i += 1
                continue
            if s.startswith("\\"):
                break
            f = s.split()
            if len(f) not in (k + 1, k + 2):
                raise ValueError("%s:%d: a %d-gram line needs %d or %d fields, got %d" % (path, i + 1, k, k + 1, k + 2, len(f)))
            words = tuple(f[1:k + 1])
            prob = _value(f[0], path, i + 1)
            bow = _value(f[k + 1], path, i + 1) if len(f) == k + 2 else 0.0
            if words in table:
                raise ValueError("%s:%d: duplicate n-gram %r" % (path, i + 1, " ".join(words)))
            if k > 1 and words[:-1] not in ngrams[k - 2]:
                raise ValueError("%s:%d: the context of %r is not in the model" % (path, i + 1, " ".join(words)))
            table[words] = (prob, bow)
            if k == 1:
                vocab.append(words[0])
            i += 1
        if len(table) != counts[k]:
            raise ValueError("%s: \\data\\ announces %d %d-grams, the section holds %d" % (path, counts[k], k, len(table)))
    if not ended:
        raise ValueError("%s: no \\end\\" % path)
    if seen != set(counts):
        raise ValueError("%s: missing sections for orders %s" % (path, sorted(set(counts) - seen)))
    for w in ("<s>", "</s>"):
        if (w,) not in ngrams[0]:
            raise ValueError("%s: the model has no %s" % (path, w))
    if ("<unk>",) not in ngrams[0]:
        ngrams[0][("<unk>",)] = (UNK_LOG10_PROB, 0.0)
        vocab.append("<unk>")
    return vocab, ngrams


#: the kinds of sub-word labels (include/e2e_ctc.h, e2e_ctc_ngram_tokens)
CONTINUATION, WORD_START, BOUNDARY = 0, 1, 2


def label_kinds(labels, blank_idx, word_marker, case_sensitive=True):
    """``(kinds, texts)`` of sub-word ``labels`` with the word marker ``word_marker``: for every label its kind
    (``CONTINUATION``: does not start with the marker; ``WORD_START``: the marker and at least one character;
    ``BOUNDARY``: exactly the marker) and the characters it adds to a word's spelling (the marker stripped, lowercased
    when ``case_sensitive`` is false).  The blank is ``(CONTINUATION, "")`` and never read.  Raises ``ValueError`` for an
    empty marker, an empty label, a label containing ``" "`` and a label containing the marker anywhere but at its
    start."""
    if not isinstance(word_marker, str) or not word_marker:
        raise ValueError("the word marker must be a non-empty string, got %r" % (word_marker,))
    m = word_marker
    kinds, texts = [], []
    for i, lab in enumerate(labels):
        if i == blank_idx:
            kinds.append(CONTINUATION)
            texts.append("")
            continue
        if not isinstance(lab, str) or not lab:
            raise ValueError("label %d is empty or no string: %r" % (i, lab))
        if " " in lab:
            raise ValueError("label %d %r contains \" \"; words are separated by the marker %r" % (i, lab, m))
        if lab.find(m, 1) >= 0:
            raise ValueError("label %d %r contains the marker %r other than at its start" % (i, lab, m))
        if lab.startswith(m):
            rest = lab[len(m):]
            kinds.append(WORD_START if rest else BOUNDARY)
        else:
            rest = lab
            kinds.append(CONTINUATION)
        texts.append(rest if case_sensitive else rest.lower())
    return kinds, texts


class NGramLM:
    """A word n-gram model on one CUDA device.  Build it with :meth:`from_arpa`; pass it to ``CTCDecoder.decode`` /
    ``decode_nbest`` as ``lm=``.  ``order``, ``vocab`` (word id -> word) and ``n_ngrams`` describe it."""

    def __init__(self, vocab, ngrams, device=None):
        _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("an NGramLM lives on a CUDA device, got %s" % self.device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.order = len(ngrams)
        self.vocab = list(vocab)
        self.word_id = {w: i for i, w in enumerate(self.vocab)}
        self.bos_id, self.eos_id, self.unk_id = (self.word_id[w] for w in _SPECIAL)
        count = sum(len(t) for t in ngrams)
        self.n_ngrams = count
        slots = 2
        while slots < 2 * count:
            slots *= 2
        self.table_slots = slots
        ids = torch.full((count, MAX_ORDER), -1, dtype=torch.int32)
        orders = torch.empty(count, dtype=torch.int32)
        probs = torch.empty(count, dtype=torch.float64)
        bows = torch.empty(count, dtype=torch.float64)
        r, wid = 0, self.word_id
        for k, table in enumerate(ngrams, 1):
            m = len(table)
            if not m:
                continue
            ids[r:r + m, :k] = torch.tensor([[wid[w] for w in words] for words in table], dtype=torch.int32)
            orders[r:r + m] = k
            pb = torch.tensor(list(table.values()), dtype=torch.float64)
            probs[r:r + m], bows[r:r + m] = pb[:, 0], pb[:, 1]
            r += m
        L = _lib.load()
        nbytes = L.e2e_ctc_ngram_table_bytes(slots)
        with torch.cuda.device(self.device):
            dev = [t.to(self.device) for t in (ids, orders, probs, bows)]
            self.table = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            stream = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            p = lambda t: ctypes.c_void_p(t.data_ptr()) if t.numel() else ctypes.c_void_p(0)   # noqa: E731
            _lib.check(L.e2e_ctc_ngram_build_device(p(self.table), slots, count, *map(p, dev), stream))
            torch.cuda.current_stream(self.device).synchronize()   # the inputs of the insert kernel go out of scope
        self._lexicons = {}

    @classmethod
    def from_arpa(cls, path, device=None):
        """Read a text ARPA file (orders 1-6) and upload its n-grams to ``device`` (default: the current CUDA device).
        A model without ``<unk>`` gets it with log10 probability -100 and backoff 0, as KenLM does.  Raises
        ``ValueError`` on a malformed file, an order above 6 or a binary KenLM model."""
        vocab, ngrams = parse_arpa(path)
        return cls(vocab, ngrams, device)

    def lexicon(self, labels, blank_idx, case_sensitive=True, word_marker=None):
        """The ``e2e_ctc_ngram`` descriptor of this model for the decoder's ``labels`` (built on first use and kept).
        Without ``word_marker`` every label except the blank must be one character and ``" "`` must be a label; with it
        the labels are sub-word units classified by :func:`label_kinds`, and the result is the pair ``(e2e_ctc_ngram,
        e2e_ctc_ngram_tokens)``.  Labels are lowercased when ``case_sensitive`` is false.  Words with a character no
        label spells are unreachable and left out."""
        labels = list(labels)
        key = (tuple(labels), int(blank_idx), bool(case_sensitive), word_marker)
        hit = self._lexicons.get(key)
        if hit is not None:
            return hit[0]
        if word_marker is not None:
            return self._token_lexicon(key, labels, blank_idx, case_sensitive, word_marker)
        if " " not in labels:
            raise ValueError("a language model needs the label \" \" between words")
        char_id, label_char = {}, []
        for i, lab in enumerate(labels):
            if i == blank_idx:
                label_char.append(-1)
                continue
            if not isinstance(lab, str) or len(lab) != 1:
                raise ValueError("with a language model every label but the blank is one character, got %r" % (lab,))
            if lab == " ":
                label_char.append(-1)
                continue
            ch = lab if case_sensitive else lab.lower()
            label_char.append(char_id.setdefault(ch, len(char_id)))
        d, kept = self._trie(char_id)
        lc_t = torch.tensor(label_char, dtype=torch.int32).to(self.device)
        d.label_char = lc_t.data_ptr()
        self._lexicons[key] = (d, kept, lc_t)
        return d

    def _token_lexicon(self, key, labels, blank_idx, case_sensitive, word_marker):
        kinds, texts = label_kinds(labels, blank_idx, word_marker, case_sensitive)
        char_id, off, chars = {}, [0], []
        for t in texts:
            chars.extend(char_id.setdefault(ch, len(char_id)) for ch in t)
            off.append(len(chars))
        d, kept = self._trie(char_id)
        dev = self.device
        kind_t = torch.tensor(kinds, dtype=torch.int8).to(dev)
        off_t = torch.tensor(off, dtype=torch.int32).to(dev)
        chars_t = torch.tensor(chars or [0], dtype=torch.int32).to(dev)
        tok = _lib.NGramTokensDesc()
        tok.label_kind, tok.label_off, tok.label_chars = kind_t.data_ptr(), off_t.data_ptr(), chars_t.data_ptr()
        self._lexicons[key] = ((d, tok), kept, kind_t, off_t, chars_t)
        return d, tok

    def _trie(self, char_id):
        """The e2e_ctc_ngram descriptor (without label_char) of the lexicon over the characters ``char_id`` and the
        device tensors it points into."""
        n_chars = len(char_id)
        child, word = [[-1] * n_chars], [-1]        # node 0: the empty spelling
        for wid, w in enumerate(self.vocab):
            if w in _SPECIAL or any(ch not in char_id for ch in w):
                continue
            node = 0
            for ch in w:
                c = char_id[ch]
                nxt = child[node][c]
                if nxt < 0:
                    nxt = child[node][c] = len(child)
                    child.append([-1] * n_chars)
                    word.append(-1)
                node = nxt
            word[node] = wid
        dev = self.device
        tensors = (torch.tensor(child, dtype=torch.int32).reshape(-1) if n_chars else torch.full((1,), -1, dtype=torch.int32),
                   torch.tensor(word, dtype=torch.int32))
        child_t, word_t = (t.to(dev) for t in tensors)
        d = _lib.NGramDesc()
        d.table, d.table_slots = self.table.data_ptr(), self.table_slots
        d.lex_child, d.lex_word = child_t.data_ptr(), word_t.data_ptr()
        d.lex_nodes, d.n_chars, d.order = len(word), n_chars, self.order
        d.bos_id, d.eos_id, d.unk_id = self.bos_id, self.eos_id, self.unk_id
        return d, (child_t, word_t)
