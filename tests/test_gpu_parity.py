"""GPU parity tests proper: the CUDA path, called through the C-ABI (ctypes), against the CPU oracle on the
same inputs.  Bit-exact (integer field work).  Run with `pytest -m gpu` on a B200."""
import numpy as np
import pytest

from helpers import gold, suite, pob_fixture, repad_pob

pytestmark = pytest.mark.gpu

FULL_COMPARE_LIMIT = 6_000_000     # entries; larger witnesses are compared by digest + sampled windows


def _check_suite(s, full_limit=FULL_COMPARE_LIMIT):
    import pob_b200
    from oracle import oracle
    c = pob_b200.Circuit(s["main"], max_slots=max(2, len(s["cases"])))
    try:
        res = c.run([k["input"] for k in s["cases"]], expand=True, digest=True)
        assert c.desc["n_slots"] >= len(s["cases"])
        for i, case in enumerate(s["cases"]):
            w = oracle.run(s["main"], case["input"])
            try:
                assert c.n_signals == w.n_signals
                assert int(res.status[i]) == w.status, "%s case %d: status %d vs oracle %d" % (s["suite"], i, res.status[i], w.status)
                if case["expected"] is None:
                    assert res.status[i] != 0
                    continue
                assert res.status[i] == 0
                assert res.outputs[i] == [int(e) for e in case["expected"]], "%s case %d outputs" % (s["suite"], i)
                assert int(res.digests[i]) == w.digest(), "%s case %d digest" % (s["suite"], i)
                if w.n_signals <= full_limit:
                    gw = c.witness(i)
                    neq = np.nonzero((gw != w.limbs).any(axis=1))[0]
                    assert len(neq) == 0, "%s case %d: %d entries differ, first at %d" % (s["suite"], i, len(neq), neq[0])
            finally:
                w.free()
    finally:
        c.close()


SMALL = [s for s in gold() if s["suite"] != "test_proof_of_burn"]


@pytest.mark.parametrize("s", SMALL, ids=[s["suite"] for s in SMALL])
def test_gadget_suite(s):
    """all 55 gadget suites of the reference (tests/test.py:146-201) incl. Spend(31), KeccakBytes, Poseidon, RLP/MPT"""
    _check_suite(s)


def test_smoke_entry():
    import __graft_entry__
    __graft_entry__.smoke()


def test_proof_of_burn_test_shape():
    """ProofOfBurn(4,4,5,...) on tests/test_pob_input.json and its four corruptions
    (tests/testcases/proof_of_burn.py:52-76): status, commitment, digest of all 64.4 M entries, and the full
    witness of case 0 entry by entry."""
    import pob_b200
    from oracle import oracle
    s = suite("test_proof_of_burn")
    c = pob_b200.Circuit(s["main"], max_slots=5)
    try:
        res = c.run([k["input"] for k in s["cases"]], expand=True, digest=True)
        for i, case in enumerate(s["cases"]):
            w = oracle.run(s["main"], case["input"])
            try:
                assert int(res.status[i]) == w.status
                if case["expected"] is None:
                    assert res.status[i] != 0
                    continue
                assert res.outputs[i] == [int(e) for e in case["expected"]]
                assert int(res.digests[i]) == w.digest()
                if i == 0:
                    step = 1 << 22
                    for first in range(0, w.n_signals, step):
                        cnt = min(step, w.n_signals - first)
                        assert np.array_equal(c.witness(0, first, cnt), w.limbs[first:first + cnt]), "window at %d" % first
            finally:
                w.free()
    finally:
        c.close()


def test_main_proof_of_burn_shape(tmp_path):
    """BASELINE.json configs[1]: main_proof_of_burn = ProofOfBurn(16,4,16,50,31,2,10^19,10^20), reference fixture
    re-padded to the main shape; 215,907,954 entries (6.9 GB).  Commitment (padding-independent, so equal to the
    pinned (4,4,5) value), whole-witness digest and sampled windows vs the oracle; plus a rejected instance."""
    import pob_b200
    from oracle import oracle
    inp = repad_pob(pob_fixture(), 16, 4, 16)
    bad = repad_pob(pob_fixture(), 16, 4, 16)
    bad["layers"][1][0] = str(int(bad["layers"][1][0]) + 1)
    expected = [int(e) for e in suite("test_proof_of_burn")["cases"][0]["expected"]]
    c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN, max_slots=2)
    try:
        assert c.n_signals == 215907954
        res = c.run([inp, bad], expand=True, digest=True)
        w = oracle.run(pob_b200.MAIN_PROOF_OF_BURN, inp)
        try:
            assert w.ok and w.n_signals == c.n_signals and w.outputs() == expected
            assert res.status[0] == 0 and res.outputs[0] == expected
            assert int(res.digests[0]) == w.digest()
            rng = np.random.default_rng(7503)
            for first in [0, c.n_signals - 4096] + [int(v) for v in rng.integers(0, c.n_signals - 65536, 24)]:
                cnt = min(65536, c.n_signals - first)
                assert np.array_equal(c.witness(0, first, cnt), w.limbs[first:first + cnt]), "window at %d" % first
        finally:
            w.free()
        wb = oracle.run(pob_b200.MAIN_PROOF_OF_BURN, bad)
        try:
            assert not wb.ok and int(res.status[1]) == wb.status
        finally:
            wb.free()
        # a rejected main-shape instance has no witness: all three accessors refuse it, and nothing was expanded for it
        assert int(res.digests[1]) == 0
        for call in (lambda: c.witness(1, 0, 8), lambda: c.witness_device_ptr(1), lambda: c.write_wtns(1, str(tmp_path / "rejected_main.wtns"))):
            with pytest.raises(pob_b200.PobError) as e:
                call()
            assert e.value.code == pob_b200.E_REJECTED
    finally:
        c.close()


def test_wtns_file_roundtrip(tmp_path):
    """The exported .wtns is byte-identical to the oracle's (SURVEY.md Appendix B layout)."""
    import pob_b200
    from oracle import oracle
    s = suite("test_spend")
    c = pob_b200.Circuit("Spend(31)", max_slots=1)
    try:
        res = c.run([s["cases"][0]["input"]])
        assert res.status[0] == 0
        a, b = str(tmp_path / "gpu.wtns"), str(tmp_path / "oracle.wtns")
        c.write_wtns(0, a)
        w = oracle.run("Spend(31)", s["cases"][0]["input"])
        w.write_wtns(b)
        w.free()
        da, db = open(a, "rb").read(), open(b, "rb").read()
        assert len(da) == 83307596 and da == db
        assert da[:4] == b"wtns" and int.from_bytes(da[4:8], "little") == 2
    finally:
        c.close()


@pytest.mark.parametrize("layers", [4, 12])
def test_config5_shapes_match_oracle(layers):
    """BASELINE.json configs[4] shapes ProofOfBurn(L,4,16,...), L = 4 and 12 (8 and 16 are covered elsewhere): synthetic
    valid instances with numLayers up to L; commitment, 64-bit digest of all S(L) entries and sampled windows against
    the oracle; a corrupted copy must be rejected with the oracle's status code."""
    import pob_b200
    from pob_b200 import synth
    from oracle import oracle
    shape = (layers, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
    expr = "ProofOfBurn(%d, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)" % layers
    insts = synth.make_batch(3, shape, seed=1000 + layers)
    packed = synth.pack_instances(insts, shape)
    packed[2, 6 + 544 + 3, 0] ^= 1                           # one byte of layer 1 of instance 2: breaks the keccak chain
    c = pob_b200.Circuit(expr, max_slots=3)
    try:
        assert c.n_signals == 51277058 + 10289431 * layers
        res = c.run_packed(packed, digest=True)
        assert res.status[0] == 0 and res.status[1] == 0 and res.status[2] != 0
        for i in (0, 1):
            w = oracle.run_flat(*oracle.parse_main(expr), packed[i])
            try:
                assert w.ok and w.n_signals == c.n_signals and res.outputs[i] == w.outputs() and int(res.digests[i]) == w.digest()
                if i == 0:
                    rng = np.random.default_rng(layers)
                    for first in [0, c.n_signals - 70000] + [int(v) for v in rng.integers(0, c.n_signals - 65536, 6)]:
                        cnt = min(65536, c.n_signals - first)
                        assert np.array_equal(c.witness(0, first, cnt), w.limbs[first:first + cnt]), "window at %d" % first
            finally:
                w.free()
        wb = oracle.run_flat(*oracle.parse_main(expr), packed[2])
        try:
            assert not wb.ok and int(res.status[2]) == wb.status
        finally:
            wb.free()
        with pytest.raises(pob_b200.PobError) as e:
            c.witness(2, 0, 16)
        assert e.value.code == pob_b200.E_REJECTED
    finally:
        c.close()


def _dir_with_space(tmp_path, need):
    import shutil
    for d in (str(tmp_path), "/dev/shm", "/tmp"):
        try:
            if shutil.disk_usage(d).free > need:
                return d
        except OSError:
            pass
    raise RuntimeError("no directory with %.1f GB free for the main-shape .wtns" % (need / 1e9))


def test_cli_main_proof_of_burn_wtns_is_the_oracles(tmp_path):
    """BASELINE.json configs[1] through the reference argv: `python -m pob_b200 main_proof_of_burn input.json witness.wtns`
    (reference Makefile:5).  The 6,909,054,604-byte file is compared byte for byte with the oracle's witness: the 76-byte
    iden3 header (SURVEY.md Appendix B) built here from the format, then all 215,907,954 entries streamed in 64 MiB
    blocks against the oracle's limbs.  A corrupted input exits non-zero, prints to stderr and writes no file."""
    import json, os, subprocess, sys
    import pob_b200
    from oracle import oracle
    d = _dir_with_space(tmp_path, 8 << 30)
    inp_json = repad_pob(pob_fixture(), 16, 4, 16)
    inp, out = os.path.join(d, "pob_input.json"), os.path.join(d, "pob_witness.wtns")
    json.dump(inp_json, open(inp, "w"))
    env = dict(os.environ, PYTHONPATH=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "proof-of-burn_b200"))
    try:
        r = subprocess.run([sys.executable, "-m", "pob_b200", "main_proof_of_burn", inp, out], env=env, capture_output=True, text=True)
        assert r.returncode == 0 and not r.stderr.strip(), r.stderr
        w = oracle.run(pob_b200.MAIN_PROOF_OF_BURN, inp_json)
        try:
            n = w.n_signals
            assert w.ok and n == 215907954 and os.path.getsize(out) == 76 + 32 * n == 6909054604
            P = pob_b200.P
            hdr = (b"wtns" + (2).to_bytes(4, "little") + (2).to_bytes(4, "little") + (1).to_bytes(4, "little") + (40).to_bytes(8, "little")
                   + (32).to_bytes(4, "little") + P.to_bytes(32, "little") + n.to_bytes(4, "little") + (2).to_bytes(4, "little") + (32 * n).to_bytes(8, "little"))
            ref = w.limbs.reshape(-1).view(np.uint8)
            with open(out, "rb") as f:
                assert f.read(76) == hdr
                off, step = 0, 64 << 20
                while off < ref.size:
                    blk = np.frombuffer(f.read(step), dtype=np.uint8)
                    assert blk.size == min(step, ref.size - off) and np.array_equal(blk, ref[off:off + blk.size]), "byte offset %d" % (76 + off)
                    off += blk.size
                assert f.read(1) == b""
        finally:
            w.free()
        os.remove(out)
        bad = dict(inp_json); bad["layers"] = [list(l) for l in inp_json["layers"]]
        bad["layers"][1][0] = str(int(bad["layers"][1][0]) + 1)
        json.dump(bad, open(inp, "w"))
        r = subprocess.run([sys.executable, "-m", "pob_b200", "main_proof_of_burn", inp, out], env=env, capture_output=True, text=True)
        assert r.returncode != 0 and r.stderr.strip() and not os.path.exists(out)
    finally:
        for f in (inp, out):
            if os.path.exists(f):
                os.remove(f)
