"""The host-side dispatch tables, read from the CUDA sources, against the case lists of tests/test_gpu_shape_dispatch.py.

The GPU matrix only proves what it covers: when a bucket, a scheme pair or a batch-size edge is added to the sources,
these tests fail until the GPU cases walk it too.  They also hold the Python precision names to the pairs the library
instantiates.  No GPU needed.
"""
import os
import re

from tests.test_gpu_shape_dispatch import BATCH_EDGE_NS, BUCKET_DS, SCHEME_CASES

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bocf_b200", "csrc")


def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _function(src, name):
    """Body of the first definition of `name` (from its opening brace to the matching closing one)."""
    m = re.search(r"\b%s\s*\([^;{]*\)\s*\{" % re.escape(name), src)
    assert m, "no definition of %s" % name
    depth, i = 1, m.end()
    while depth:
        depth += {"{": 1, "}": -1}.get(src[i], 0)
        i += 1
    return src[m.end():i - 1]


def _constant(src, name):
    m = re.search(r"constexpr\s+\w+\s+%s\s*=\s*(\d+)\s*;" % re.escape(name), src)
    assert m, "no constant %s" % name
    return int(m.group(1))


def _ladder(body, last):
    """Upper ends of an `if (d <= K) return ...; ... return <last>;` ladder."""
    ends = [int(k) for k in re.findall(r"if\s*\(\s*d\s*<=\s*(\d+)\s*\)", body)]
    assert ends == sorted(ends) and len(ends) >= 2, ends
    return ends + [last]


def _kstar_ladder():
    body = _function(_source("posterior.cu"), "launch_kstar_k")
    tail = re.findall(r"return\s+launch_kstar_t<\s*KIND\s*,\s*(\w+)\s*>", body)[-1]
    return _ladder(body, _constant(_source("model.h"), "MAXD") if tail == "MAXD" else int(tail))


def _grad_ladder():
    body = _function(_source("split_gemm.cu"), "launch_grad")
    return _ladder(body, int(re.findall(r"return\s+launch_grad_d<\s*EPI\s*,\s*(\d+)\s*>", body)[-1]))


def _var_labels():
    """(scheme of the first contraction, digit planes of its re-split V) of every launch_var case."""
    labels = [int(c) for c in re.findall(r"case\s+(\d+)\s*:", _function(_source("split_gemm.cu"), "launch_var"))]
    assert labels
    return {(c // 10, c % 10) for c in labels}


def _scheme_for_slices():
    body = _function(_source("split_gemm.cu"), "split_scheme_for_slices")
    table = {int(s): int(c) for s, c in re.findall(r"S\s*==\s*(\d)\s*\?\s*(\d+)", body)}
    assert sorted(table) == [3, 4, 5, 6], table
    return table


def test_kstar_and_gradient_contraction_share_the_d_buckets():
    assert _kstar_ladder() == _grad_ladder() == [4, 6, 8, 10, 12, 16]


def test_gpu_cases_hold_both_ends_of_every_d_bucket():
    ends = _kstar_ladder()
    lows = [1] + [e + 1 for e in ends[:-1]]
    missing = sorted(set(lows + ends) - set(BUCKET_DS))
    assert not missing, "d values of the DP buckets without a GPU case: %s" % missing


def test_every_split_precision_has_a_first_contraction():
    from bocf_b200 import _lib
    labels, sch = _var_labels(), _scheme_for_slices()
    split = {name: slices for name, (mode, slices) in _lib.PRECISIONS.items() if mode == 1}
    assert split
    for name, slices in split.items():
        s1, s2 = (slices // 10, slices % 10) if slices >= 10 else (slices, slices)
        assert (sch[s1], s2) in labels, "%s: no launch_var instantiation for scheme %d with %d planes" % (name, sch[s1], s2)


def test_gpu_cases_cover_every_first_contraction():
    from bocf_b200 import _lib
    covered = set()
    for name, (sch1, sch2) in SCHEME_CASES:
        covered.add((sch1, sch2 // 100))          # launch_var re-splits V into the digit planes (SA) of the second scheme
        mode, slices = _lib.PRECISIONS[name]
        if mode == 1:                             # an explicit split request: the pair the case asserts is the one named
            s1, s2 = (slices // 10, slices % 10) if slices >= 10 else (slices, slices)
            sch = _scheme_for_slices()
            assert (sch[s1], sch[s2]) == (sch1, sch2), name
    assert covered == _var_labels()


def test_precision_names_are_the_accepted_pairs():
    import pytest
    from bocf_b200 import _lib
    split = sorted(n for n, (mode, _) in _lib.PRECISIONS.items() if mode == 1)
    assert split == ["split3", "split33", "split4", "split43", "split44", "split5", "split54", "split55", "split6",
                     "split65", "split66"]
    for name in ("split53", "split63", "split64", "split32", "split7"):
        assert name not in _lib.PRECISIONS
        with pytest.raises(ValueError):
            _lib.parse_precision(name)


def test_gpu_cases_straddle_every_batch_size_edge():
    """The MC pass shape (tiny / small / sweep), the small final gradient sum and the K* K-split switch at fixed
    candidate counts; section d of the GPU tests sits on both sides of each."""
    acq, post = _source("acq.cu"), _source("posterior.cu")
    edges = {int(k) for k in re.findall(r"Nvalid\s*<=\s*(\d+)", _function(acq, "launch_mc_t"))}
    edges |= {int(k) for k in re.findall(r"Nvalid\s*<=\s*(\d+)", _function(post, "launch_fused_grad_chunk"))}
    edges.add(_constant(post, "KSTAR_SPLIT_MAX"))
    assert edges == {128, 1024}, edges
    for e in sorted(edges):
        assert e in BATCH_EDGE_NS and e + 1 in BATCH_EDGE_NS, e
