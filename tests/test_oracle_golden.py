"""Pins oracle/reference_model.py against the reference's own doctest vectors
(tests/golden/doctests.json, transcribed from the doc comments with file:line)."""
import pytest

from conftest import untuple
from oracle import reference_model as R
from oracle.reference_model import usize, Array, Scalar, all_, fn_view, Coated


def exp(golden, name, key="expect"):
    return [untuple(x) for x in golden[name][key]]


def test_collect_all(golden):  # src/view.rs:138-142 and :91-96 (Rc<V> is a View via Deref)
    a = usize.all(5).collect()
    assert a.as_ref() == exp(golden, "collect_all") == exp(golden, "rc_all_collect")


def test_nested_index_mut(golden):  # src/view.rs:162-172
    a = Array.new(usize, 3, [Scalar("apple"), Scalar("body"), Scalar("crane")])
    n = a.nested()
    assert n.I == (usize, ())
    assert n.at((1, ())) == "body"
    a.at(1).value = "BODY"  # (&mut a).nested()[(1, ())] = "BODY"
    assert [s.value for s in a.as_ref()] == exp(golden, "nested_index_mut")


def test_nested_collect_behead(golden):  # src/view.rs:197-221
    class Behead(R.View):
        I = usize
        def __init__(self, v): self.v = v
        def size(self): return self.v.size() - 1
        def at(self, index): return self.v.at(index + 1)

    a = all_((bool, usize), 4).collect()
    assert a.as_ref() == exp(golden, "nested_collect_behead", "expect_a")
    b = a.rows(bool, usize).map(Behead).nested_collect(3)
    assert b.as_ref() == exp(golden, "nested_collect_behead")


def test_each_total(golden):  # src/view.rs:243-249
    a = usize.all(5).collect()
    total = []
    a.each(total.append)
    assert sum(total) == golden["each_total"]["expect"]


def test_enumerate(golden):  # src/view.rs:257-266
    a = Array.new(usize, 3, ["apple", "body", "crane"])
    assert a.enumerate().collect().as_ref() == exp(golden, "enumerate")


def test_diagonal(golden):  # src/view.rs:276-284
    a = usize.all(3).map(lambda x: x + 10).diagonal(0).collect()
    assert a.as_ref() == exp(golden, "diagonal")
    assert a.size() == (3, 3)


def test_map_square(golden):  # src/view.rs:294-298
    assert usize.all(5).map(lambda x: x * x).collect().as_ref() == exp(golden, "map_square")


def test_compose(golden):  # src/view.rs:307-313
    a = Array.new(bool, (), [2, 1])
    b = Array.new(usize, 3, ["apple", "body", "crane"])
    ab = a.compose(b).collect()
    assert ab.I is bool and ab.as_ref() == exp(golden, "compose")


def test_compose_out_of_bounds():  # src/int.rs:17 panic text
    a = Array.new(bool, (), [2, 3])
    b = Array.new(usize, 3, ["apple", "body", "crane"])
    with pytest.raises(R.Panic, match="Index 3 is out of bounds for size 3"):
        a.compose(b).collect()


def test_concat(golden):  # src/view.rs:320-326
    a = Array.new(usize, 2, ["apple", "body"])
    b = Array.new(usize, 2, ["crane", "dump"])
    ab = a.concat(b, (), ()).iso(usize).collect()
    assert ab.as_ref() == exp(golden, "concat")


def test_from_usize(golden):  # src/view.rs:346-351
    g = golden["from_usize"]
    a = Array.new((usize, usize, usize), (3, 2, 1), g["items"])
    b = a.from_usize(usize, bool, usize, lambda _: ()).collect()
    assert b.at(untuple(g["probe_b"])) == a.at(untuple(g["probe_a"]))
    assert b.as_ref() == g["items"]


def test_to_usize(golden):  # src/view.rs:367-372
    g = golden["to_usize"]
    a = Array.new((usize, bool, usize), (3, (), 1), g["items"])
    b = a.to_usize(usize, bool, usize).collect()
    assert b.at(untuple(g["probe_b"])) == a.at(untuple(g["probe_a"]))
    assert b.size() == (3, 2, 1)


def test_insert_remove_one(golden):  # src/view.rs:384-390, :401-407
    a = Array.new((bool, bool), ((), ()), ["A", "a", "B", "b"])
    b = a.insert_one(bool, usize, bool, 1).collect()
    assert b.size() == untuple(golden["insert_one"]["expect_size"])
    assert b.as_ref() == golden["insert_one"]["expect"]
    c = Array.new((bool, usize, bool), ((), 1, ()), ["A", "a", "B", "b"]).remove_one(bool, usize, bool).collect()
    assert c.size() == untuple(golden["remove_one"]["expect_size"])
    assert c.as_ref() == golden["remove_one"]["expect"]


def test_map_axis(golden):  # src/view.rs:423-435
    a = Array.new(usize, 2, [2, 1])
    b = Array.new((bool, usize), 3, ["apple", "body", "crane", "APPLE", "BODY", "CRANE"])
    ab = b.map_axis(a, bool, ()).collect()
    assert ab.as_ref() == exp(golden, "map_axis")


def test_zip(golden):  # src/view.rs:451-487
    a = usize.all(3).collect()
    b = Array.new(usize, 3, ["apple", "body", "crane"])
    assert a.zip(b).collect().as_ref() == exp(golden, "zip_same_shape")
    assert a.zip(Scalar("repeated")).collect().as_ref() == exp(golden, "zip_scalar")
    a2 = usize.all(3).iso((usize, ())).collect()
    b2 = all_(bool, ()).iso(((), bool)).collect()
    ab = a2.zip(b2).collect()
    assert ab.I == (usize, bool)
    assert ab.as_ref() == exp(golden, "zip_broadcast")


def test_zip_unequal_sizes():  # src/broadcast.rs:38
    a = usize.all(3).collect()
    b = usize.all(4).collect()
    with pytest.raises(R.Panic, match="Unequal sizes"):
        a.zip(b).collect()


def test_binary_add(golden):  # src/view.rs:499-506
    a = Array.new(usize, 3, [9, 8, 7])
    b = Array.new(usize, 3, [10, 20, 30])
    assert a.binary(b, R.Add).collect().as_ref() == exp(golden, "binary_add")
    assert (a + b).collect().as_ref() == exp(golden, "binary_add")


def test_coat_group_pairs(golden):  # src/view.rs:523-548
    def group_pairs(view, I):
        view = view.coat((Coated(I), usize))
        view = view.from_usize(Coated(I), (usize, bool), (), lambda n: (n // 2, ()))
        view = view.iso((Coated(I), usize, bool))
        return view.coat((I, usize, bool))

    g = golden["coat_group_pairs"]
    a = Array.new((usize, usize), (2, 6), ["a", "b", "c", "d", "e", "f", "A", "B", "C", "D", "E", "F"])
    b = group_pairs(a, usize).collect()
    assert b.size() == untuple(g["expect_size"])
    assert b.as_ref() == g["expect"]


def test_transpose(golden):  # src/view.rs:572-585
    a = all_((usize, usize), (3, 2)).collect()
    assert a.as_ref() == exp(golden, "transpose", "expect_a")
    b = a.transpose((), usize, usize, ()).collect()
    assert b.as_ref() == exp(golden, "transpose")


def test_row_column(golden):  # src/view.rs:596-608, :626-638
    a = all_((usize, usize), (3, 2)).collect()
    assert a.row(usize, usize, 1).collect().as_ref() == exp(golden, "row")
    assert a.column(usize, usize, 1).collect().as_ref() == exp(golden, "column")


def test_fn_view_and_from_fn(golden):  # src/view.rs:1431-1435, src/array.rs:38-42
    assert fn_view(usize, 10, lambda x: x % 3 == 0).collect().as_ref() == golden["fn_view"]["expect"]
    assert Array.from_fn(usize, 10, lambda x: x % 3 == 0).as_ref() == golden["array_from_fn"]["expect"]


def test_array_new_indexing(golden):  # src/array.rs:18-27
    g = golden["array_new_indexing"]
    a = Array.new((usize, bool), 3, g["items"])
    for idx, want in g["probes"]:
        assert a[untuple(idx)] == want
    with pytest.raises(R.Panic):  # src/array.rs:12
        Array.new((usize, bool), 3, g["items"][:-1])


def test_tuple_isomorphism(golden):  # src/tuple.rs:195-248
    forms = [untuple(f) for f in golden["tuple_isomorphic"]["forms"]]
    for t in forms:
        for u in forms:
            assert R.flatten_value(t) == R.flatten_value(u)
            # rebuild u's structure from t's leaves
            def shape(x): return tuple(shape(y) for y in x) if isinstance(x, tuple) else None
            assert R.unflatten(shape(u), R.flatten_value(t)) == u
    for value, flat in golden["tuple_push_pop"]["flat_of"]:
        assert R.flatten_value(untuple(value)) == list(flat)


def test_index_roundtrip_and_order():
    """Index::each visits in to_usize order and from_usize inverts it (contract src/view.rs:28-29,
    src/index.rs:60-66) for every index type the model implements."""
    cases = [
        (usize, 5), (bool, ()), ((), ()), ((usize,), (3,)), ((usize, bool), (3, ())),
        ((usize, (usize, usize), ()), (2, (3, 4), ())), (R.Reversed, 4), (R.Fixed(3), ()),
        (R.Option(usize), 3), ((R.Option(bool), usize), ((), 2)), (Coated((usize, bool)), R.CoatedV((2, ()))),
    ]
    for I, size in cases:
        seen = []
        R.each(I, size, seen.append)
        assert len(seen) == R.length(I, size)
        for k, i in enumerate(seen):
            assert R.to_usize(I, i, size) == k
            assert R.from_usize(I, size, k) == (0, i)
        assert R.from_usize(I, size, len(seen) + 0)[0] == 1


def test_fold_rows_sequential_order():
    """rows().map(fold) is a left-to-right fold in index order (src/view.rs:250-252, :1341)."""
    a = Array.new((usize, usize), (2, 3), [1, 2, 3, 4, 5, 6])
    trace = R.fold_rows(a, usize, usize, lambda s, x: s * 10 + x, 0).collect()
    assert trace.as_ref() == [123, 456]


def test_product_library_is_fresh():
    """The in-tree .so must be newer than every source it is built from (stale builds hide fixes)."""
    import glob, os
    from multidimension_b200 import LIB_PATH
    assert os.path.exists(LIB_PATH), "run __graft_entry__.build()"
    src = glob.glob(os.path.join(os.path.dirname(LIB_PATH), "csrc", "*.*")) + [os.path.join(os.path.dirname(LIB_PATH), "..", "include", "mdim.h")]
    newest = max(os.path.getmtime(p) for p in src if not p.endswith(".log"))
    assert os.path.getmtime(LIB_PATH) >= newest, "libmdim_b200.so is older than its sources: run __graft_entry__.build()"


def test_golden_vectors_are_extracted_from_the_reference_sources():
    """tests/golden/doctests.json must be exactly what make_doctest_vectors.py parses out of the assert_eq! lines of the
    reference's src/*.rs.  Those sources are not part of this repository: the test runs where MDIM_REFERENCE names a
    checkout of apt1002/multidimension 0.3.3 and skips elsewhere."""
    import os, subprocess, sys
    ref = os.environ.get("MDIM_REFERENCE")
    if not ref or not os.path.isdir(os.path.join(ref, "src")):
        pytest.skip("MDIM_REFERENCE does not name a checkout of the reference sources")
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_doctest_vectors.py")
    r = subprocess.run([sys.executable, script, "--check"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
