"""Seeded text with exact control of pretoken byte lengths, for the tests of the pretoken tables (hashtab.cuh).

Both pretoken tables -- the count table of training and the encoder's cache -- keep a key in one of three tiers by its byte
length: short (1-7 bytes), medium (8-15) and long (>= 16, the bytes compared through 8-byte loads with a masked tail).  The text
built here holds tens of thousands of distinct pretokens in every tier, so that every table grows while it holds entries, plus the
lengths and near-twins where a key compare, a key load or a per-pretoken BPE kernel switches form.

Every word is a whole GPT-2 pretoken by construction:
  * letter, digit and punctuation runs carry a leading space (` ?\\p{L}+`, ` ?\\p{N}+`, ` ?[^\\s\\p{L}\\p{N}]+`), so the space of the
    next word ends them;
  * a whitespace run is always followed by a word that starts with a space and a non-space, so `\\s+(?!\\S)` takes exactly the run;
    two whitespace runs are never adjacent.
The punctuation alphabet has no apostrophe (no contraction can start inside a run) and includes NUL bytes.  The text is valid UTF-8
without a carriage return.  The oracle's count (oracle.count_pretokens) is the truth the tests compare with; the generator's own
bookkeeping is only what tests/test_pretoken_tables_cpu.py pins about the composition.
"""
from __future__ import annotations

import random

LETTERS = {
    1: "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ",
    2: "éüßçñøåжщыдлπλΩ",                      # Latin-1 / Cyrillic / Greek letters
    3: "中文字日本語アイウ한국",                  # CJK, kana, Hangul (Lo)
    4: "\U0001D400\U0001D401\U0001D41A\U00020000\U00020001",   # mathematical bold letters (Lu / Ll), CJK extension B (Lo)
}
DIGITS = {1: "0123456789", 2: "٠١٢٣٤٥٦٧٨٩"}   # ASCII and Arabic-Indic digits (Nd)
PUNCT = {
    1: "!#$%&()*+,-./:;<=>?@[]^_`{|}~\"\x00",
    2: "§©®°±×÷",
    3: "…€™←→∑≠",
    4: "\U0001F600\U0001F680\U0001F44D",     # emoji (So)
}
WHITESPACE = " \n\t"
# lengths every tier boundary and every switch of the per-pretoken BPE kernels (<= 32 bytes: one thread, more: one warp) sits at
EDGE_LENGTHS = (7, 8, 15, 16, 17, 23, 24, 31, 32, 33, 64, 65, 511, 512, 513, 4095, 4096, 4097, 4103, 6007)
TWIN_POSITIONS = ("last", 8, 15)
LONG_TWIN_PREFIX = 4096                       # long near-twins share this many bytes


def _run(rnd: random.Random, classes: dict, n: int) -> str:
    """Characters from `classes` (bytes per character -> alphabet) that are exactly n UTF-8 bytes long."""
    out, left = [], n
    sizes = sorted(classes)
    while left > 0:
        s = rnd.choice([s for s in sizes if s <= left])   # (every alphabet has 1-byte characters: any remainder can be filled)
        out.append(rnd.choice(classes[s]))
        left -= s
    return "".join(out)


def word(rnd: random.Random, n: int, kind: str | None = None) -> bytes:
    """One pretoken of exactly n bytes (n >= 1).  Kinds: letters / digits / punct (a space and a run of n - 1 bytes), space (a
    whitespace run; the caller follows it with a word that starts with a space)."""
    if kind is None:
        kind = rnd.choices(("letters", "digits", "punct", "space"), (70, 10, 12, 8))[0]
    if n == 1:
        return rnd.choice(("\n", "\t")).encode()
    if kind == "space":
        return "".join(rnd.choice(WHITESPACE) for _ in range(n)).encode()
    classes = {"letters": LETTERS, "digits": DIGITS, "punct": PUNCT}[kind]
    w = (" " + _run(rnd, classes, n - 1)).encode("utf-8")
    assert len(w) == n, (kind, n, w)
    return w


def ascii_word(rnd: random.Random, n: int) -> bytes:
    return (" " + "".join(rnd.choice(LETTERS[1]) for _ in range(n - 1))).encode()


def _is_space_word(w: bytes) -> bool:
    return w.strip(b" \n\t") == b""


def near_twins(rnd: random.Random) -> list[tuple[bytes, bytes]]:
    """Pairs of distinct pretokens that differ in one byte: the last one, byte 8 or byte 15, at every tier's lengths; long words that
    share their first LONG_TWIN_PREFIX bytes and differ in the masked tail of the byte compare (or in its last full 8-byte block)."""
    pairs = []
    for n in (8, 9, 15, 16, 17, 23, 24, 31, 32, 33, 40, 64, 65, 100):
        for pos in TWIN_POSITIONS:
            i = n - 1 if pos == "last" else pos
            if i >= n:
                continue
            a = bytearray(ascii_word(rnd, n))
            b = bytearray(a)
            b[i] = ord("x") if a[i] != ord("x") else ord("y")
            pairs.append((bytes(a), bytes(b)))
    for tail in range(1, 16):
        n = LONG_TWIN_PREFIX + tail
        a = bytearray(ascii_word(rnd, n))
        for i in sorted({n - 1, LONG_TWIN_PREFIX, n - 1 - (n % 8 if n % 8 else 8) + 1}):
            b = bytearray(a)
            b[i] = ord("x") if a[i] != ord("x") else ord("y")
            pairs.append((bytes(a), bytes(b)))
    return pairs


def prefix_chain(rnd: random.Random, n: int = 40) -> list[bytes]:
    """A word and all of its prefixes of >= 2 bytes (every tier; each a pretoken of its own)."""
    w = ascii_word(rnd, n)
    return [w[:k] for k in range(2, n + 1)]


def distinct_words(rnd: random.Random, n_short: int, n_medium: int, n_long: int, avoid=frozenset()) -> list[bytes]:
    """n_short + n_medium + n_long distinct pretokens, none in `avoid`, with lengths spread over each tier: 1-7, 8-15, and >= 16
    (mostly 16-64, a tail to a few hundred bytes)."""
    seen = set(avoid)
    out = []

    def take(k, lengths):
        got = 0
        while got < k:
            w = word(rnd, lengths())
            if w not in seen:
                seen.add(w)
                out.append(w)
                got += 1

    take(n_short, lambda: rnd.randint(2, 7))
    take(n_medium, lambda: rnd.randint(8, 15))
    take(n_long, lambda: rnd.randint(16, 64) if rnd.random() < 0.93 else rnd.randint(65, 700))
    return out


def render(rnd: random.Random, words: list[bytes], frequent: list[bytes] = (), n_frequent: int = 0) -> bytes:
    """Every word 1-4 times (mostly once or twice), every frequent word n_frequent times, in a seeded order; a whitespace run is
    never followed by another one (a separator word " ws" is put between)."""
    occ = []
    for w in words:
        occ += [w] * rnd.choices((1, 2, 3, 4), (50, 25, 15, 10))[0]
    for w in frequent:
        occ += [w] * n_frequent
    rnd.shuffle(occ)
    parts, prev_space = [], False
    for w in occ:
        sp = _is_space_word(w)
        if sp and prev_space:
            parts.append(b" ws")
        parts.append(w)
        prev_space = sp
    if prev_space:
        parts.append(b" end")
    return b"".join(parts)


FREQUENT = [b" the", b" of", b" and", b" a", b" to", b" in", b" is", b" ,", b" .", b" was", b" information", b" constitutional"]


def edge_words(rnd: random.Random) -> list[bytes]:
    """Every EDGE_LENGTHS length in every kind, plus 1-byte words."""
    out = [b"\n", b"\t"]
    for n in EDGE_LENGTHS:
        for kind in ("letters", "digits", "punct", "space"):
            out.append(word(rnd, n, kind))
    return out


def tier_corpus(seed: int = 0, n_short: int = 50000, n_medium: int = 30000, n_long: int = 22000, n_frequent: int = 2000):
    """(text, info): the full tier corpus.  info = {"words": every distinct word placed, "twins": [(a, b)], "edges": [...],
    "prefixes": [...]}."""
    rnd = random.Random(seed)
    twins = near_twins(rnd)
    edges = edge_words(rnd)
    prefixes = prefix_chain(rnd)
    special = [w for p in twins for w in p] + edges + prefixes
    words = special + distinct_words(rnd, n_short, n_medium, n_long, avoid=frozenset(special))
    words = list(dict.fromkeys(words))
    text = render(rnd, words, FREQUENT, n_frequent)
    return text, {"words": words, "twins": twins, "edges": edges, "prefixes": prefixes}


def encoder_texts(seed: int = 1, specials: list[bytes] = ()):
    """(t1, t2, train_text): t2 holds t1's words plus at least twice as many new medium and long ones (and new short ones), in another
    order, each special 300 times in both; train_text (its own words, the same alphabets) trains a tokenizer whose merges reach into
    long pretokens."""
    rnd = random.Random(seed)
    twins = near_twins(rnd)
    edges = edge_words(rnd)
    base = list(dict.fromkeys([w for p in twins for w in p] + edges + prefix_chain(rnd)))
    a = base + distinct_words(rnd, 4000, 5000, 7000, avoid=frozenset(base))
    b = distinct_words(rnd, 8000, 11000, 16000, avoid=frozenset(a))
    t1 = render(rnd, a, FREQUENT + list(specials), 300)
    t2 = render(rnd, a + b, FREQUENT + list(specials), 300)
    train = render(rnd, distinct_words(rnd, 3000, 3000, 3000), FREQUENT, 100)
    return t1, t2, train


def encoder_pretokens(data: bytes, specials: list[bytes]) -> set[bytes]:
    """The distinct pretokens the encoder looks up in its cache: the text is cut at the specials first (the longest one wins at a
    position, tokenizer.py:63-66) and every other piece is pretokenized on its own; the specials themselves are not counted."""
    import re
    from oracle import oracle
    if not specials:
        return set(oracle.count_pretokens(data, []))
    pat = re.compile(b"(" + b"|".join(re.escape(s) for s in sorted(specials, key=len, reverse=True)) + b")")
    out = set()
    for i, piece in enumerate(pat.split(data)):
        if i % 2 == 0 and piece:
            out.update(oracle.count_pretokens(piece, []))
    return out
