# -*- coding: utf-8 -*-
"""Host-side text preparation (mirror of east/utils.py:31-133).

These stay in Python on the host (north_star): upper-casing, tokenising and grouping words
into the strings collection a generalized AST is built from.
"""
import importlib
import itertools
import os
import pkgutil
import random
import re

_TOKEN_RE = re.compile(r"[\w']+", re.U)


def prepare_text(text):
    """utf-8 decode (undecodable bytes replaced) and UPPER-case -- east/utils.py:31-34."""
    if isinstance(text, bytes):
        text = text.decode("utf-8", errors="replace")
    return text.upper()


def tokenize(text):
    """Maximal runs of word characters and apostrophes -- east/utils.py:37-38."""
    return _TOKEN_RE.findall(text)


def synonym_variants(query, synonyms):
    """Every substitution of the words of `query` by their synonyms, as the reference scores them with a synonimizer
    (east/asts/easa.py:27-33).  synonyms: the synonimizer's get_synonyms() mapping -- a word it lacks raises KeyError
    unless it is a defaultdict.  Variants are not space-stripped (a synonym with a space keeps it); a query without
    tokens has the single variant ""."""
    options = [synonyms[w] + [w] for w in tokenize(query)]
    return ["".join(words) for words in itertools.product(*options)]


def tokenize_and_filter(text, min_word_length=3, stopwords=None):
    """east/utils.py:41-46 (stop-word list must be supplied; nltk is not a dependency here)."""
    stopwords = stopwords or set()
    return [t for t in tokenize(text) if len(t) >= min_word_length and t not in stopwords]


def text_to_strings_collection(text, words=3):
    """Split a text into strings of `words` consecutive tokens joined without a separator.

    east/utils.py:49-79: tokens of length <= 2 and all-digit tokens are dropped first; a text
    with no usable token yields [" "] so that an AST can still be built.
    """
    tokens = [t for t in tokenize(prepare_text(text)) if len(t) > 2 and not t.isdigit()]
    groups = ["".join(tokens[i:i + words]) for i in range(0, len(tokens), words)]
    return groups or [" "]


def text_collection_to_string_collection(text_collection, words=3):
    return flatten([text_to_strings_collection(text, words) for text in text_collection])


def random_string(length):
    """east/utils.py:86-88 -- NB: yields length-2 characters, as the reference does."""
    return "".join(chr(ord("A") + random.randint(0, 25)) for _ in range(length - 2))


def flatten(lst):
    return list(itertools.chain.from_iterable(lst))


def output_is_redirected():
    try:
        return os.fstat(0) != os.fstat(1)
    except OSError:
        return True


def itersubclasses(cls, _seen=None):
    """All subclasses of cls, depth first (east/utils.py:100-116)."""
    if not isinstance(cls, type):
        raise TypeError("itersubclasses must be called with new-style classes, not %.100r" % cls)
    _seen = set() if _seen is None else _seen
    for sub in cls.__subclasses__():
        if sub not in _seen:
            _seen.add(sub)
            yield sub
            for subsub in itersubclasses(sub, _seen):
                yield subsub


def import_modules_from_package(package):
    """Import every module of `package` so engine classes register (east/utils.py:119-133)."""
    pkg = importlib.import_module(package)
    for info in pkgutil.walk_packages(pkg.__path__, prefix=package + "."):
        if not info.name.rsplit(".", 1)[-1].startswith("__"):
            importlib.import_module(info.name)
