"""CPU-side checks of the name-containment relation of a locus (hgt_locus_set_names / hgt_locus_name_subsets), the part of
the batched pair model that the legacy code computes with `allele in allele_pair` string tests."""
import ctypes

import numpy as np
import pytest

from conftest import GOLDEN_NAMES, load_golden
from helpers import golden_db, product_locus, synthetic_case


def brute(names):
    return [[x for x in range(len(names)) if names[x] in a] for a in names]


def as_lists(off, idx):
    return [idx[off[a]:off[a + 1]].tolist() for a in range(len(off) - 1)]


def set_names(t, names):
    from hisatgenotype_b200.locus import lib
    arr = (ctypes.c_char_p * len(names))(*[n.encode() for n in names])
    rc = lib().hgt_locus_set_names(t.handle, len(names), arr)
    t._names_set = t._names_set or rc == 0  # t.name_subsets() must not hand over t.names again
    return rc


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_subsets_of_golden_names(name):
    g = load_golden(name)
    db = golden_db(g)
    for cap in g["loci"]:
        t = product_locus(g, db, cap["gene"], cap["Gene_names"], host_only=True)
        off, idx = t.name_subsets()
        assert as_lists(off, idx) == brute(t.names)
        t.close()


SYNTH_NAMES = [
    ["A*01", "A*01:01", "A*01:011", "A*01:0110", "A*02", "A*02:01", "B*07", "B*07:02"],  # prefixes
    ["1", "11", "111", "2", "21", "212", "X1X", "X2X", "Y1Y1"],                             # infixes, repeated substrings
    ["AB", "BA", "CD", "DC", "EF", "FE"],                                                    # equal lengths, no relation
    ["K*%03d:%02d" % (i // 7, i % 7) for i in range(200)],                                  # no relation, many names
    ["X*01:1", "X*01:10", "X*01:100", "X*01:1X*01:10", "X*02", "X*02:2", "X*020"],          # both at once
]


@pytest.mark.parametrize("names", SYNTH_NAMES)
def test_subsets_of_synthetic_names(names):
    args, _, _ = synthetic_case(3, len(names), L=1200, n_pairs=10, n_groups=4, core_vars=20, pool_private=60)
    from hisatgenotype_b200.locus import LocusTables
    t = LocusTables(*args, host_only=True)
    t._names_set = False
    assert t.A >= len(names)
    names = sorted(names + ["~%04d" % i for i in range(t.A - len(names))])  # fillers for the locus's other alleles
    assert set_names(t, names) == 0
    off, idx = t.name_subsets()
    assert as_lists(off, idx) == brute(names)
    t.close()


def test_wrong_names_are_refused():
    from hisatgenotype_b200 import _lib
    from hisatgenotype_b200.locus import LocusTables
    args, _, _ = synthetic_case(3, 12, L=1200, n_pairs=10, n_groups=4, core_vars=20, pool_private=60)
    t = LocusTables(*args, host_only=True)
    t._names_set = False
    names = list(t.names)
    assert set_names(t, names[:-1]) == _lib.HGT_ERR_ARG
    assert set_names(t, names + ["Z*99"]) == _lib.HGT_ERR_ARG
    assert set_names(t, names[::-1]) == _lib.HGT_ERR_ARG            # not in sorted order
    assert set_names(t, names[:-1] + ["Z*1-2"]) == _lib.HGT_ERR_ARG  # the pair key's separator
    n = ctypes.c_int64(0)
    from hisatgenotype_b200.locus import lib
    assert lib().hgt_locus_name_subsets(t.handle, None, None, ctypes.byref(n)) == _lib.HGT_ERR_ARG  # nothing set yet
    assert set_names(t, names) == 0
    small = np.zeros(1, np.int32)
    n.value = 1
    assert lib().hgt_locus_name_subsets(t.handle, None, _lib.ptr(small), ctypes.byref(n)) == _lib.HGT_ERR_ARG  # capacity
    assert n.value == t.A
    assert set_names(t, names) == 0
    off, idx = t.name_subsets()
    assert as_lists(off, idx) == brute(names)
    t.close()


def test_names_from_several_threads():
    """Loci are shared by batches on several host threads: concurrent hand-overs and read-backs of the relation must
    neither corrupt it nor see a half-made one."""
    import threading
    from hisatgenotype_b200.locus import LocusTables
    args, _, _ = synthetic_case(3, 60, L=1200, n_pairs=10, n_groups=4, core_vars=20, pool_private=60)
    t = LocusTables(*args, host_only=True)
    t._names_set = False
    own = list(t.names)
    other = sorted(["Q*%02d" % i for i in range(t.A - 3)] + ["Q*0", "Q*1", "Q*100"])
    errors = []

    def hand_over():
        try:
            t.ensure_names()
        except Exception as e:  # pragma: no cover - reported below
            errors.append(e)

    threads = [threading.Thread(target=hand_over) for _ in range(8)]
    for x in threads:
        x.start()
    for x in threads:
        x.join()
    assert not errors
    assert as_lists(*t.name_subsets()) == brute(own)

    want = (brute(own), brute(other))

    def churn(k):
        try:
            for i in range(40):
                assert set_names(t, own if (i + k) % 2 else other) == 0
                assert as_lists(*t.name_subsets()) in want  # never a mix of two relations
        except Exception as e:  # pragma: no cover - reported below
            errors.append(e)

    threads = [threading.Thread(target=churn, args=(k,)) for k in range(6)]
    for x in threads:
        x.start()
    for x in threads:
        x.join()
    assert not errors, errors[:1]
    assert set_names(t, own) == 0
    assert as_lists(*t.name_subsets()) == brute(own)
    t.close()
