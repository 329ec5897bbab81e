"""The order-pinning kit (tools/diff_sym.py + pob_write_components): the tool itself is exercised on .sym files fabricated from
our own component lists (circom is absent here); with circom on PATH the same test pins the ORDER against the real compiler."""
import io, os, shutil, sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def _fake_sym(comps, path):
    """what `circom --sym` would write for a layout with exactly these components: `s,w,c,name`"""
    with open(path, "w") as f:
        for c, (first, n, tmpl) in enumerate(comps):
            comp = "main" if c == 0 else "main.c%d_%s" % (c, tmpl.split("/")[0])
            for j in range(n):
                f.write("%d,%d,%d,%s.x[%d]\n" % (first + j, first + j, c, comp, j))


def test_component_list_covers_every_signal_once():
    import pob_b200, diff_sym
    for expr in ("Spend(31)", "LeafDetector(544)", "RlpMerklePatriciaTrieLeaf(32, 31)", "KeccakBytes(2)"):
        for hc in (False, True):
            comps = diff_sym.our_components(expr, hc)
            nxt = 1
            for first, n, _t in comps:
                assert first == nxt and n > 0
                nxt = first + n
            assert nxt == pob_b200.layout_info(expr, hcreate=hc)["n_signals"]


def test_diff_tool_verdicts(tmp_path):
    import diff_sym
    expr = "Num2BitsSafe(256)"                     # contains Num2Bits_strict: the two numbering policies differ here
    default, created = diff_sym.our_components(expr, False), diff_sym.our_components(expr, True)
    assert default != created
    sym = str(tmp_path / "a.sym")
    out = io.StringIO()
    _fake_sym(default, sym)
    assert diff_sym.compare(sym, expr, out) == 0 and "IDENTICAL" in out.getvalue()
    _fake_sym(created, sym)
    out = io.StringIO()
    assert diff_sym.compare(sym, expr, out) == 1 and "hcreate=1" in out.getvalue()
    broken = list(default)
    k = len(broken) // 2
    broken[k] = (broken[k][0], broken[k][1] + 1, broken[k][2])          # a component with one more own signal
    broken[k + 1:] = [(a + 1, b, t) for a, b, t in broken[k + 1:]]
    _fake_sym(broken, sym)
    out = io.StringIO()
    assert diff_sym.compare(sym, expr, out) == 2 and (">> #%-8d" % k) in out.getvalue()


def test_order_against_real_circom_when_available():
    """pins the witness ORDER whenever circom is on PATH and POB_REFERENCE names a proof-of-burn checkout; otherwise states
    that it is unpinned"""
    import diff_sym
    ref = os.environ.get("POB_REFERENCE")
    if not shutil.which("circom") or not ref or not os.path.isdir(os.path.join(ref, "circuits")):
        pytest.skip("needs circom on PATH and POB_REFERENCE set to a proof-of-burn checkout: the whole-witness ORDER remains "
                    "unpinned (values, outputs, accept/reject are pinned)")
    assert diff_sym.auto(ref, ["main_spend"]) == 0
