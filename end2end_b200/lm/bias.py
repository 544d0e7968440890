"""Phrase biasing (contextual biasing, hot words) for the GPU prefix beam search (``CTCDecoder.decode(..., bias=)`` /
``decode_nbest(..., bias=)``; include/e2e_ctc.h, e2e_ctc_bias, has the definition).

A :class:`PhraseBias` holds caller-given phrases of labels with a per-token weight.  The search adds the bonus of the
phrases a prefix has completed (``committed``) and partial credit for a phrase being spelled (``phi``) to every score it
ranks and prunes with, and withdraws the partial credit at the end.  The phrases are compiled once, on the host, into an
Aho-Corasick automaton over labels (full transition table over the labels that occur in some phrase) and uploaded once.
"""
import math

import torch

from .. import _lib

#: the largest transition table (automaton nodes x distinct phrase labels, int32 entries: 256 MB)
MAX_TRANSITIONS = 1 << 26


class PhraseBias:
    """Phrases to boost inside the prefix beam search, on one CUDA device.

    :param phrases: a sequence of phrases, each a non-empty sequence of label ids (not the blank), or a string when
        ``labels`` is given and every label but the blank is one character (each character is the label spelling it;
        no case folding).  No two phrases may be equal.
    :param weight: the per-token weight (natural log, finite, > 0): one float for every phrase or one per phrase.  A
        completed phrase of k labels adds ``weight * k`` to the score of every prefix that contains it, once per
        occurrence.
    :param labels: the decoder's labels (optional): fixes the alphabet size and lets phrases be strings.
    :param blank_idx: the blank label, which no phrase may contain.
    :param device: the CUDA device (default: the current one).  The automaton is uploaded there once, with the first
        search.

    Raises ``ValueError`` for an empty phrase list or phrase, the blank or an out-of-range label in a phrase, a
    duplicate phrase, a character with no label, a weight that is not finite and positive, and an automaton whose
    transition table exceeds ``MAX_TRANSITIONS`` entries (checked before the table is allocated).
    ``nodes`` and ``n_cols`` describe the automaton."""

    def __init__(self, phrases, weight, *, labels=None, blank_idx=0, device=None):
        self.blank_idx = int(blank_idx)
        self.alphabet = None if labels is None else len(labels)
        self.phrases = [self._phrase(p, labels) for p in phrases]
        if not self.phrases:
            raise ValueError("no phrases")
        if len(set(self.phrases)) != len(self.phrases):
            raise ValueError("duplicate phrase")
        if isinstance(weight, (int, float)):
            weights = [float(weight)] * len(self.phrases)
        else:
            weights = [float(w) for w in weight]
            if len(weights) != len(self.phrases):
                raise ValueError("%d weights for %d phrases" % (len(weights), len(self.phrases)))
        if not all(math.isfinite(w) and w > 0 for w in weights):
            raise ValueError("phrase weights must be finite and > 0")
        self.weights = weights
        label_col, nxt, partial, complete = build_automaton(self.phrases, weights)
        self.nodes, self.n_cols = len(partial), len(label_col)
        self._label_col = label_col                 # phrase label -> column
        device = torch.device("cuda") if device is None else torch.device(device)
        if device.type != "cuda":
            raise ValueError("a PhraseBias lives on a CUDA device, got %s" % device)
        if device.index is None:
            _lib.load()
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        # uploaded with the first search (a host-only object can be built and checked without a device)
        self._host = (torch.tensor(nxt, dtype=torch.int32).reshape(-1), torch.tensor(partial, dtype=torch.float64),
                      torch.tensor(complete, dtype=torch.float64))
        self._dev = None
        self._cols = {}                             # alphabet size -> device label_col

    def _phrase(self, p, labels):
        if isinstance(p, str):
            if labels is None:
                raise ValueError("a phrase given as a string needs labels")
            if any(i != self.blank_idx and (not isinstance(lab, str) or len(lab) != 1) for i, lab in enumerate(labels)):
                raise ValueError("string phrases need labels of one character each")
            index = {lab: i for i, lab in enumerate(labels) if i != self.blank_idx}
            try:
                p = [index[ch] for ch in p]
            except KeyError as e:
                raise ValueError("no label spells %r" % e.args[0]) from None
        p = tuple(int(c) for c in p)
        if not p:
            raise ValueError("empty phrase")
        for c in p:
            if c == self.blank_idx:
                raise ValueError("phrase %r contains the blank" % (p,))
            if c < 0 or (self.alphabet is not None and c >= self.alphabet):
                raise ValueError("phrase %r has a label outside the alphabet" % (p,))
        return p

    def descriptor(self, alphabet):
        """The ``e2e_ctc_bias`` descriptor for logits of ``alphabet`` labels (the label-to-column table is built on
        first use and kept).  Raises ``ValueError`` when the bias was built for another alphabet size or a phrase
        label is outside it."""
        alphabet = int(alphabet)
        if self.alphabet is not None and self.alphabet != alphabet:
            raise ValueError("a PhraseBias for %d labels, logits of %d" % (self.alphabet, alphabet))
        if max(self._label_col) >= alphabet:
            raise ValueError("phrase label %d outside an alphabet of %d" % (max(self._label_col), alphabet))
        if self._dev is None:
            self._dev = tuple(t.to(self.device) for t in self._host)
        col = self._cols.get(alphabet)
        if col is None:
            host = [-1] * alphabet
            for c, j in self._label_col.items():
                host[c] = j
            col = self._cols[alphabet] = torch.tensor(host, dtype=torch.int32).to(self.device)
        nxt, partial, complete = self._dev
        d = _lib.BiasDesc()
        d.label_col, d.next = col.data_ptr(), nxt.data_ptr()
        d.partial, d.complete = partial.data_ptr(), complete.data_ptr()
        d.nodes, d.n_cols = self.nodes, self.n_cols
        return d


def build_automaton(phrases, weights):
    """``(label_col, next, partial, complete)`` of the Aho-Corasick automaton over ``phrases`` (tuples of labels) with
    per-token ``weights`` (include/e2e_ctc.h, e2e_ctc_bias): ``label_col`` maps each phrase label to its column,
    ``next`` is a list of rows (one per node, node 0 the root), ``partial`` and ``complete`` are lists of floats."""
    labels = sorted({c for p in phrases for c in p})
    label_col = {c: j for j, c in enumerate(labels)}
    children, own, depth = [{}], [-1], [0]          # the trie; own: the phrase ending at the node
    for i, p in enumerate(phrases):
        node = 0
        for c in p:
            nxt = children[node].get(c)
            if nxt is None:
                nxt = len(children)
                children[node][c] = nxt
                children.append({})
                own.append(-1)
                depth.append(depth[node] + 1)
            node = nxt
        own[node] = i
    n = len(children)
    if n * len(labels) > MAX_TRANSITIONS:
        raise ValueError("the phrases make an automaton of %d nodes x %d labels, above %d transitions"
                         % (n, len(labels), MAX_TRANSITIONS))
    fail, order = [0] * n, [0]                      # breadth-first: every shallower node comes first
    nxt = [None] * n
    for u in order:
        row = list(nxt[fail[u]]) if u else [0] * len(labels)
        for c, v in children[u].items():
            row[label_col[c]] = v
            fail[v] = nxt[fail[u]][label_col[c]] if u else 0
            order.append(v)
        nxt[u] = row
    # the phrases ending at each node (its own and along the fail chain), summed in ascending phrase index
    ends = [()] * n
    complete = [0.0] * n
    for u in order[1:]:
        e = ends[fail[u]]
        if own[u] >= 0:
            e = tuple(sorted(e + (own[u],)))
        ends[u] = e
        acc = 0.0
        for i in e:
            acc = acc + weights[i] * len(phrases[i])
        complete[u] = acc
    # phi: the longest suffix that is a proper phrase prefix (a node with children) times the largest weight of the
    # phrases it is a proper prefix of
    below = [-math.inf] * n                          # largest weight of a phrase ending strictly below the node
    for u in reversed(order):
        for v in children[u].values():
            w = max(below[v], weights[own[v]] if own[v] >= 0 else -math.inf)
            below[u] = max(below[u], w)
    grow = [0] * n                                   # the longest suffix with children
    partial = [0.0] * n
    for u in order[1:]:
        g = u if children[u] else grow[fail[u]]
        grow[u] = g
        partial[u] = depth[g] * below[g] if g else 0.0
    return label_col, nxt, partial, complete
