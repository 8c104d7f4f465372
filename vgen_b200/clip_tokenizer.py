"""CLIP byte-pair tokenizer (host side of the text conditioning, SURVEY.md section 8f-4).

The reference calls `open_clip.tokenize(text)` (tools/modules/clip_embedder.py:186): lower-cased, whitespace-collapsed
text is split by a regex into words / digits / punctuation runs, every UTF-8 byte is mapped to a printable code point,
and adjacent symbols are merged greedily by the rank of the pair in the published merge list
(`bpe_simple_vocab_16e6.txt.gz`, OpenAI CLIP, MIT licence); ids = [<start_of_text>] + pieces + [<end_of_text>], zero
padded / truncated to 77.  This file implements that published algorithm; ids are index work, so the bar is bit-exact
(tests/test_host_logic.py compares with ids the reference's vendored tokenizer produced, stored under tests/golden/).

The merge list is data, not code: it is looked up (a) at `VGEN_CLIP_BPE`, (b) inside an installed `open_clip` package,
(c) in the reference tree on `sys.path` (`utils/reward/open_clip/`), the way the engines' own import finds it.
"""
from __future__ import annotations

import gzip
import html
import os
import sys
from functools import lru_cache

import regex
import torch

CONTEXT_LENGTH = 77
_N_MERGES = 49152 - 256 - 2          # vocabulary = 256 bytes + 256 end-of-word bytes + merges + 2 specials
_SPLIT = regex.compile(r"<start_of_text>|<end_of_text>|'s|'t|'re|'ve|'m|'ll|'d|[\p{L}]+|[\p{N}]|[^\s\p{L}\p{N}]+", regex.IGNORECASE)


def find_bpe_file():
    cands = []
    if os.environ.get("VGEN_CLIP_BPE"):
        cands.append(os.environ["VGEN_CLIP_BPE"])
    try:
        import importlib.util
        spec = importlib.util.find_spec("open_clip")
        if spec and spec.submodule_search_locations:
            cands += [os.path.join(p, "bpe_simple_vocab_16e6.txt.gz") for p in spec.submodule_search_locations]
    except Exception:  # noqa: BLE001 - a broken optional package must not hide the other locations
        pass
    for root in list(sys.path) + [os.getcwd()]:
        cands.append(os.path.join(root, "utils", "reward", "open_clip", "bpe_simple_vocab_16e6.txt.gz"))
    for c in cands:
        if c and os.path.exists(c):
            return c
    raise FileNotFoundError("CLIP merge list bpe_simple_vocab_16e6.txt.gz not found: set VGEN_CLIP_BPE, install open_clip, "
                            "or run from the reference tree (utils/reward/open_clip/)")


@lru_cache()
def _byte_symbols():
    """byte value -> printable unicode character (bytes that already are printable map to themselves)."""
    keep = list(range(33, 127)) + list(range(161, 173)) + list(range(174, 256))
    table, extra = {}, 0
    for b in range(256):
        if b in keep:
            table[b] = chr(b)
        else:
            table[b] = chr(256 + extra)
            extra += 1
    return table


class ClipTokenizer:
    def __init__(self, bpe_path=None):
        path = bpe_path or find_bpe_file()
        lines = gzip.open(path).read().decode("utf-8").split("\n")
        merges = [tuple(ln.split()) for ln in lines[1:1 + _N_MERGES]]
        sym = _byte_symbols()
        # vocabulary order: printable-first byte order of the published table, then the same with </w>, then merges
        order = list(range(33, 127)) + list(range(161, 173)) + list(range(174, 256))
        order += [b for b in range(256) if b not in order]
        base = [sym[b] for b in order]
        vocab = base + [s + "</w>" for s in base] + ["".join(m) for m in merges] + ["<start_of_text>", "<end_of_text>"]
        self.ids = {tok: i for i, tok in enumerate(vocab)}
        self.rank = {m: i for i, m in enumerate(merges)}
        self.sot, self.eot = self.ids["<start_of_text>"], self.ids["<end_of_text>"]
        self._cache = {}

    def _merge_word(self, word):
        """word: string of byte symbols -> list of sub-word pieces after greedy lowest-rank merging."""
        if word in self._cache:
            return self._cache[word]
        parts = list(word[:-1]) + [word[-1] + "</w>"]
        while len(parts) > 1:
            best, best_rank = None, None
            for a, b in zip(parts, parts[1:]):
                r = self.rank.get((a, b))
                if r is not None and (best_rank is None or r < best_rank):
                    best, best_rank = (a, b), r
            if best is None:
                break
            out, i = [], 0
            while i < len(parts):
                if i + 1 < len(parts) and parts[i] == best[0] and parts[i + 1] == best[1]:
                    out.append(parts[i] + parts[i + 1])
                    i += 2
                else:
                    out.append(parts[i])
                    i += 1
            parts = out
        self._cache[word] = parts
        return parts

    @staticmethod
    def _clean(text):
        try:                                   # the reference passes text through ftfy first; identity for clean input
            import ftfy
            text = ftfy.fix_text(text)
        except ImportError:
            pass
        text = html.unescape(html.unescape(text)).strip()
        return regex.sub(r"\s+", " ", text).strip().lower()

    def encode(self, text):
        sym = _byte_symbols()
        out = []
        for piece in _SPLIT.findall(self._clean(text)):
            if piece in ("<start_of_text>", "<end_of_text>"):
                out.append(self.ids[piece])
                continue
            word = "".join(sym[b] for b in piece.encode("utf-8"))
            out.extend(self.ids[p] for p in self._merge_word(word))
        return out

    def __call__(self, texts, context_length=CONTEXT_LENGTH):
        if isinstance(texts, str):
            texts = [texts]
        res = torch.zeros(len(texts), context_length, dtype=torch.long)
        for i, t in enumerate(texts):
            ids = [self.sot] + self.encode(t) + [self.eot]
            if len(ids) > context_length:
                ids = ids[:context_length]
                ids[-1] = self.eot
            res[i, :len(ids)] = torch.tensor(ids)
        return res


_DEFAULT = None


def tokenize(texts, context_length=CONTEXT_LENGTH):
    """Drop-in for open_clip.tokenize."""
    global _DEFAULT
    if _DEFAULT is None:
        _DEFAULT = ClipTokenizer()
    return _DEFAULT(texts, context_length)
