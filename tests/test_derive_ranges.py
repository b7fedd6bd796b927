"""Term derivation sweeps each term only over the dictionary words whose first two bytes can pass the first-letter rule (the
F / S / ALL groups of the derivation schedule).  These cases aim at the edges of that schedule: edits at bytes 0 and 1, first
bytes no dictionary word starts with, one- and two-byte terms and words, bytes >= 0x80, caps filled across tiles, 32-word groups
that receive matches from two groups, and the order of the terms in a call.  Every result must equal the CPU oracle's, word for
word and in order."""
import numpy as np
import pytest

from corpus.pyindexgen import IndexImage

pytestmark = pytest.mark.gpu

LETTERS = "abcdefghi"
WIDE = ["é", "ñ", "ü"]  # two bytes each in UTF-8, >= 0xC3


@pytest.fixture(scope="module")
def mb():
    import meilisearch_b200 as m

    m.load_library()
    return m


def _vocabulary():
    rng = np.random.default_rng(2024)
    alphabet = list(LETTERS) + WIDE
    words = set(LETTERS) | set(WIDE) | {a + b for a in LETTERS[:4] for b in LETTERS[:4]} | {"é" + "a", "a" + "é", "ñü"}
    while len(words) < 4000:
        n = int(rng.integers(1, 13))
        words.add(LETTERS[int(rng.integers(len(LETTERS)))] + "".join(alphabet[int(i)] for i in rng.integers(len(alphabet), size=n - 1)))
    # first letter 'k': more than 150 one-typo neighbours of "kabcdefg" among enough other 'k' words to span several tiles
    base = "kabcdefg"
    for p in range(1, len(base)):
        for c in "abcdefghijklmnopqrstuvwxyz":
            words.add(base[:p] + c + base[p + 1:])
    while sum(w.startswith("k") for w in words) < 900:
        words.add("k" + "".join(LETTERS[int(i)] for i in rng.integers(len(LETTERS), size=int(rng.integers(2, 10)))))
    # around the 'y' / 'z' boundary, neighbours of "yzabcdefg" from four groups in a row: S('y') and S('z') at the end of the
    # 'x' words, then F('y'), then F('z')
    edge = {"xyzabcdefg", "xzabcdefg"} | {"yzabcdef" + c for c in "hijklmnopqrstuvwxyz"} | {"zabcdefg"} | {"zabcdefg" + c for c in "abcdefghijklmnopqrstuvwxyz"}
    words |= edge
    # filler 'x' words (they sort before the edge words): pad so that the 'y' / 'z' boundary falls in the middle of a 32-word group
    ordered = sorted(words, key=str.encode)
    z0 = next(i for i, w in enumerate(ordered) if w.startswith("z"))
    for i in range((16 - z0) % 32):
        words.add("xa" + LETTERS[i % 9] * (1 + i // 9))
    return sorted(words, key=str.encode)


@pytest.fixture(scope="module")
def image():
    words = _vocabulary()
    img = IndexImage(1)
    rng = np.random.default_rng(7)
    order = rng.permutation(len(words))
    for d in range(0, len(words), 40):
        img.add_text(d // 40, 0, " ".join(words[i] for i in order[d: d + 40]))
    img = img.build()
    got = [img.word(i) for i in range(img.n_words)]
    assert got == words
    return img


@pytest.fixture(scope="module")
def oracle(image):
    from oracle.pyoracle import OracleIndex

    return OracleIndex(image)


def _check(ix, oracle, terms):
    got = ix.derive([t[0] for t in terms], [t[1] for t in terms], [t[2] for t in terms])
    for (w, mt, p), (g1, g2) in zip(terms, got):
        o1, o2 = oracle.derive(w, mt, p)
        assert list(g1) == list(o1), (w, mt, p, "one")
        assert list(g2) == list(o2), (w, mt, p, "two")
    return got


def _edits_at(w, p):
    """substitution, insertion, deletion and transposition at character p"""
    out = [w[:p] + ("z" if w[p] != "z" else "y") + w[p + 1:], w[:p] + "h" + w[p:], w[:p] + w[p + 1:]]
    if p + 1 < len(w):
        out.append(w[:p] + w[p + 1] + w[p] + w[p + 2:])
    return out


def _edge_terms(image):
    long_words = [image.word(i) for i in range(0, image.n_words, 7) if len(image.word(i)) >= 10 and image.word(i).isascii()][:12]
    terms = []
    for w in long_words:
        for p in (0, 1):
            for t in _edits_at(w, p):
                terms += [(t, 2, 0), (t, 2, 1)]
    # first bytes that no dictionary word starts with ('j', 'q', 'w' and 'r' start none), at q0 and at q1
    for t in ("jabcdefgh", "qzabcdefg", "ajbcdefghi", "bwcdefghia", "rqabcdefg", "érabcdefg", "aébcdefghi"):
        terms += [(t, 2, 0), (t, 2, 1), (t, 1, 0), (t, 1, 1)]
    # one- and two-byte terms with two typos: every word is a candidate (the ALL group)
    for t in ("a", "b", "k", "é", "ab", "ba", "ñü", "zq", "ké"):
        terms += [(t, 2, 0), (t, 2, 1)]
    # caps: > 150 one-typo matches under 'k' across tiles; > 50 two-typo ones
    terms += [("kabcdefg", 1, 0), ("kabcdefg", 1, 1), ("kabcdefgh", 2, 0), ("kabcdefgh", 2, 1), ("kabcdefgh", 1, 1)]
    # the 'y' / 'z' boundary
    terms += [("yzabcdefg", 2, 0), ("yzabcdefg", 2, 1), ("yzabcdefg", 1, 1)]
    return terms


def test_tile_straddles_groups(image):
    # the fixture must really put matches of two groups into one 32-word group
    z0 = next(i for i in range(image.n_words) if image.word(i).startswith("z"))
    assert z0 % 32 == 16
    assert image.word(z0 - 1).startswith("yzabcdef") and image.word(z0) == "zabcdefg"


def test_edits_at_first_bytes(mb, image, oracle):
    ix = mb.Index(image)
    terms = [t for t in _edge_terms(image) if len(t[0]) >= 9 and t[1] == 2]
    assert len(terms) > 150
    _check(ix, oracle, terms)


def test_short_terms_and_absent_first_bytes(mb, image, oracle):
    ix = mb.Index(image)
    got = _check(ix, oracle, [t for t in _edge_terms(image) if len(t[0]) < 9 or t[0][0] in "jqré"])
    assert any(len(g1) + len(g2) for g1, g2 in got)


def test_caps_and_group_boundaries(mb, image, oracle):
    ix = mb.Index(image)
    got = _check(ix, oracle, [("kabcdefg", 1, 0), ("kabcdefgh", 2, 1), ("yzabcdefg", 2, 1), ("yzabcdefg", 2, 0)])
    assert len(got[0][0]) == 150 and len(got[1][1]) == 50
    # the prefix term has matches on both sides of the 'y' / 'z' boundary, inside one 32-word group
    z0 = next(i for i in range(image.n_words) if image.word(i).startswith("z"))
    ids = set(got[2][0].tolist()) | set(got[2][1].tolist())
    assert z0 - 1 in ids and z0 in ids


def test_mixed_call_and_permutation(mb, image, oracle):
    ix = mb.Index(image)
    terms = _edge_terms(image)
    # the same word at every budget
    for w in ("kabcdefgh", "yzabcdefg", "ab", "éabcdefgh"):
        terms += [(w, mt, p) for mt in (1, 2) for p in (0, 1)]
    got = _check(ix, oracle, terms)
    perm = np.random.default_rng(3).permutation(len(terms))
    got_p = ix.derive([terms[i][0] for i in perm], [terms[i][1] for i in perm], [terms[i][2] for i in perm])
    for j, i in enumerate(perm):
        assert list(got_p[j][0]) == list(got[i][0]) and list(got_p[j][1]) == list(got[i][1]), terms[i]


def test_fuzz_edited_words(mb, image, oracle):
    rng = np.random.default_rng(99)
    alphabet = list(LETTERS) + WIDE + ["z", "k"]
    terms = []
    while len(terms) < 3000:
        w = image.word(int(rng.integers(image.n_words)))
        for _ in range(int(rng.integers(1, 3))):
            p = int(rng.integers(len(w)))
            k = int(rng.integers(4))
            c = alphabet[int(rng.integers(len(alphabet)))]
            if k == 0:
                w = w[:p] + c + w[p + 1:]
            elif k == 1:
                w = w[:p] + c + w[p:]
            elif k == 2 and len(w) > 1:
                w = w[:p] + w[p + 1:]
            elif p + 1 < len(w):
                w = w[:p] + w[p + 1] + w[p] + w[p + 2:]
        if 3 <= len(w.encode()) <= 64:
            terms.append((w, int(rng.integers(1, 3)), int(rng.integers(2))))
    _check(mb.Index(image), oracle, terms)
