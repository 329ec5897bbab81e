"""More GPU parity: fuzzed gadget inputs, ordering policy, slot ring / residency, staged inputs, synthetic batches at
the full main shape, a second circuit shape, and the proof-of-work grinder.  All through the C-ABI."""
import numpy as np
import pytest

from helpers import suite, pob_fixture, repad_pob, cuda_poke

pytestmark = pytest.mark.gpu


def test_fuzz_gadgets_match_oracle():
    import pob_b200
    from oracle import oracle
    from fuzz_cases import cases
    by_main = {}
    for main, inp in cases():
        by_main.setdefault(main, []).append(inp)
    rejected = 0
    for main, inps in by_main.items():
        c = pob_b200.Circuit(main, max_slots=len(inps))
        try:
            res = c.run(inps, expand=True, digest=True)
            for i, inp in enumerate(inps):
                w = oracle.run(main, inp)
                try:
                    assert int(res.status[i]) == w.status, "%s %s: status %d vs oracle %d" % (main, inp, res.status[i], w.status)
                    if w.ok:
                        assert int(res.digests[i]) == w.digest()
                        assert np.array_equal(c.witness(i), w.limbs), "%s %s" % (main, inp)
                    else:
                        rejected += 1
                finally:
                    w.free()
        finally:
            c.close()
    assert rejected > 10


def test_creation_order_policy_on_gpu():
    import pob_b200
    from oracle import oracle
    s = suite("test_spend")
    c = pob_b200.Circuit("Spend(31)", hcreate=True, max_slots=1)
    try:
        res = c.run([s["cases"][0]["input"]])
        w = oracle.run("Spend(31)", s["cases"][0]["input"], hcreate=True)
        w0 = oracle.run("Spend(31)", s["cases"][0]["input"], hcreate=False)
        assert res.status[0] == 0 and np.array_equal(c.witness(0), w.limbs)
        assert not np.array_equal(w.limbs, w0.limbs)
        w.free(); w0.free()
    finally:
        c.close()


def test_slot_ring_wraps_and_residency_is_enforced():
    import pob_b200
    from oracle import oracle
    base = suite("test_spend")["cases"][0]["input"]
    inps = [dict(base, extraCommitment=str(1000 + i)) for i in range(8)]
    c = pob_b200.Circuit("Spend(31)", max_slots=3)
    try:
        assert c.desc["n_slots"] == 3
        with pytest.raises(pob_b200.PobError) as e:           # 8 witnesses into 3 slots: the library refuses to drop 5 unread
            c.run(inps)
        assert e.value.code == pob_b200.E_RANGE
        res = c.run(inps, discard=True)                       # ... unless told to (generation-only run)
        assert (res.status == 0).all() and len({o[0] for o in res.outputs}) == 8
        for i in (5, 6, 7):                                   # the last three are resident
            w = oracle.run("Spend(31)", inps[i])
            assert np.array_equal(c.witness(i), w.limbs) and res.outputs[i] == w.outputs()
            w.free()
        for i in (0, 4):                                      # overwritten by later instances
            with pytest.raises(pob_b200.PobError) as e:
                c.witness(i)
            assert e.value.code == pob_b200.E_RANGE
        with pytest.raises(pob_b200.PobError):
            c.witness(8)
        res2 = c.run(inps[:2], expand=False)                  # status/outputs only: nothing resident afterwards
        assert res2.outputs == res.outputs[:2]
        with pytest.raises(pob_b200.PobError):
            c.witness(0)
    finally:
        c.close()


def test_retain_list_materialises_only_the_named_instances():
    """SURVEY.md 8(b) "which indices to retain": all instances are evaluated, only the listed ones get a witness"""
    import pob_b200
    from oracle import oracle
    base = suite("test_spend")["cases"][0]["input"]
    inps = [dict(base, extraCommitment=str(50 + i)) for i in range(40)]          # 40 instances, 3 slots
    c = pob_b200.Circuit("Spend(31)", max_slots=3)
    try:
        res = c.run(inps, retain=[2, 17, 39], digest=True)
        assert (res.status == 0).all() and len({o[0] for o in res.outputs}) == 40
        assert res.timing["expand_launches"] >= 1
        for i in (2, 17, 39):
            w = oracle.run("Spend(31)", inps[i])
            assert np.array_equal(c.witness(i), w.limbs) and int(res.digests[i]) == w.digest()
            w.free()
        assert int(res.digests[3]) == 0
        for i in (0, 3, 38):
            with pytest.raises(pob_b200.PobError) as e:
                c.witness(i)
            assert e.value.code == pob_b200.E_RANGE
        with pytest.raises(pob_b200.PobError):
            c.run(inps, retain=[1, 2, 3, 4])                 # more than the 3 slots
        with pytest.raises(pob_b200.PobError):
            c.run(inps, retain=[5, 5])                       # not strictly ascending
        res0 = c.run(inps, retain=[])
        assert res0.outputs == res.outputs and res0.timing["expand_launches"] == 0
    finally:
        c.close()


def test_rejected_instance_has_no_witness(tmp_path):
    """SURVEY.md 8(b): a failed instance contributes no witness (the reference calculator aborts, tests/test.py:65-68):
    every accessor answers POB_E_REJECTED, its digest stays 0, and the neighbours are unaffected."""
    import pob_b200
    from oracle import oracle
    s = suite("test_spend")
    good, bad = s["cases"][0]["input"], s["cases"][1]["input"]
    assert s["cases"][1]["expected"] is None
    never = str(tmp_path / "never.wtns")
    c = pob_b200.Circuit("Spend(31)", max_slots=3)
    try:
        res = c.run([good, bad, good], digest=True)
        assert res.status[0] == 0 and res.status[1] != 0 and res.status[2] == 0
        assert int(res.digests[1]) == 0 and res.digests[0] == res.digests[2] != 0
        for call in (lambda: c.witness(1), lambda: c.witness_device_ptr(1), lambda: c.write_wtns(1, never), lambda: c.selfcheck_keccak(1)):
            with pytest.raises(pob_b200.PobError) as e:
                call()
            assert e.value.code == pob_b200.E_REJECTED
        import os
        assert not os.path.exists(never)
        w = oracle.run("Spend(31)", good)
        assert np.array_equal(c.witness(2), w.limbs)
        w.free()
    finally:
        c.close()


def test_consumer_paced_handoff_drops_nothing():
    """pob_submit / pob_acquire / pob_release / pob_finish: 11 instances through 3 slots; the consumer (here: a D2H copy)
    sees EVERY accepted witness, bit-exact, in order; the rejected one is reported and skipped; holding all slots gives
    POB_E_BUSY instead of an overwrite."""
    import pob_b200
    from oracle import oracle
    s = suite("test_spend")
    base, bad = s["cases"][0]["input"], s["cases"][1]["input"]
    inps = [dict(base, extraCommitment=str(300 + i)) for i in range(11)]
    inps[4] = bad
    c = pob_b200.Circuit("Spend(31)", max_slots=3)
    try:
        packed = c.pack(inps)
        c.submit(packed, digest=True)
        seen = []
        while True:
            r = c.acquire()
            if r is None:
                break
            idx, dptr = r
            if dptr is None:
                assert idx == 4
                seen.append((idx, None))
                continue
            assert dptr == c.witness_device_ptr(idx)         # held witnesses are accessible while the batch is in flight
            w = oracle.run("Spend(31)", inps[idx])
            assert np.array_equal(c.witness(idx), w.limbs), "instance %d" % idx
            w.free()
            seen.append((idx, dptr))
            c.release(idx)
            with pytest.raises(pob_b200.PobError):
                c.release(idx)                               # double release
        assert [i for i, _ in seen] == list(range(11))
        res = c.finish()
        assert [int(v != 0) for v in res.status] == [0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0] and int(res.digests[4]) == 0
        # hold everything: generation must stall, not overwrite
        c.submit(packed)
        held = []
        with pytest.raises(pob_b200.PobError) as e:
            while True:
                r = c.acquire()
                if r[1] is not None:
                    held.append(r[0])
        assert e.value.code == pob_b200.E_BUSY and len(held) == 3
        first = {i: c.witness(i, 0, 64).copy() for i in held}
        c.release(held[0])
        r = c.acquire()
        assert r is not None and r[0] == 3
        for i in held[1:]:
            assert np.array_equal(c.witness(i, 0, 64), first[i])        # still intact while held
        res = c.finish()
        assert res.n_ok == 10
    finally:
        c.close()


def test_export_batch_writes_every_accepted_witness(tmp_path):
    """pob_export_batch == n runs of `./main_spend input_i.json witness_i.wtns` (reference Makefile:5-6) with only 2 slots
    for 7 instances: every accepted instance's file is byte-identical to the oracle's, the rejected one leaves no file."""
    import os
    import pob_b200
    from oracle import oracle
    s = suite("test_spend")
    base, bad = s["cases"][0]["input"], s["cases"][1]["input"]
    inps = [dict(base, extraCommitment=str(900 + i)) for i in range(7)]
    inps[2] = bad
    c = pob_b200.Circuit("Spend(31)", max_slots=2)
    try:
        paths = [str(tmp_path / ("w%d.wtns" % i)) for i in range(7)]
        res, st = c.export_batch(c.pack(inps), paths)
        assert res.status[2] != 0 and res.n_ok == 6 and st["witnesses"] == 6 and st["bytes"] == 6 * 83307596
        assert not os.path.exists(paths[2])
        for i in (0, 1, 3, 6):
            w = oracle.run("Spend(31)", inps[i]); ref = str(tmp_path / "ref.wtns"); w.write_wtns(ref); w.free()
            assert open(paths[i], "rb").read() == open(ref, "rb").read(), "instance %d" % i
        res2, st2 = c.export_batch(c.pack(inps))              # host-memory sink only (PCIe measurement mode)
        assert st2["witnesses"] == 6 and res2.outputs == res.outputs
    finally:
        c.close()


def test_staged_inputs_equal_host_inputs():
    import pob_b200
    base = suite("test_spend")["cases"][0]["input"]
    inps = [dict(base, extraCommitment=str(7 + i)) for i in range(40)]     # > one eval chunk
    c = pob_b200.Circuit("Spend(31)", max_slots=4)
    try:
        packed = c.pack(inps)
        a = c.run_packed(packed, digest=True)
        c.stage(packed)
        b = c.run_packed(None, n=len(inps), staged=True, digest=True)
        assert np.array_equal(a.status, b.status) and np.array_equal(a.outputs_limbs, b.outputs_limbs) and np.array_equal(a.digests, b.digests)
        assert a.timing["h2d_bytes"] == 40 * 4 * 32 and b.timing["h2d_bytes"] == 0
    finally:
        c.close()


def test_synthetic_batch_main_shape():
    """BASELINE.json configs[2] in miniature: 40 synthetic valid main-shape inputs (more than the 21 resident slots, more
    than one eval chunk): all accepted; three instances checked against the oracle by commitment + whole-witness digest."""
    import pob_b200
    from pob_b200 import synth
    from oracle import oracle
    shape = (16, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
    insts = synth.make_batch(40, shape, seed=99)
    c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN)
    try:
        res = c.run_packed(synth.pack_instances(insts, shape), digest=True)
        assert (res.status == 0).all()
        for i in (0, 21, 39):
            w = oracle.run(pob_b200.MAIN_PROOF_OF_BURN, synth.to_json(insts[i], shape))
            try:
                assert w.ok and res.outputs[i] == w.outputs() and int(res.digests[i]) == w.digest()
            finally:
                w.free()
        first = 215907954 - 70000
        w = oracle.run(pob_b200.MAIN_PROOF_OF_BURN, synth.to_json(insts[39], shape))
        assert np.array_equal(c.witness(39, first, 70000), w.limbs[first:])
        w.free()
    finally:
        c.close()


def test_second_shape_eight_layers():
    """config 5 point: ProofOfBurn(8,4,16,...) -- S(8) = 133,592,506 entries"""
    import pob_b200
    from pob_b200 import synth
    from oracle import oracle
    shape = (8, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
    expr = "ProofOfBurn(8, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)"
    insts = synth.make_batch(2, shape, seed=5)
    c = pob_b200.Circuit(expr, max_slots=2)
    try:
        assert c.n_signals == 51277058 + 10289431 * 8
        res = c.run_packed(synth.pack_instances(insts, shape), digest=True)
        w = oracle.run(expr, synth.to_json(insts[1], shape))
        assert res.status[1] == 0 and w.ok and res.outputs[1] == w.outputs() and int(res.digests[1]) == w.digest()
        w.free()
    finally:
        c.close()


def test_pow_grinder_finds_the_first_key():
    """reference tests/testcases/proof_of_work.py: (burnKey, 234, 345): 812 -> 1 zero byte, 47109 -> 2, neighbours 0"""
    import pob_b200
    from pob_b200 import synth
    assert pob_b200.pow_grind(812, 234, 345, zero_bytes=1) == (812, 1)
    assert pob_b200.pow_grind(47109, 234, 345, zero_bytes=2) == (47109, 1)

    def cpu_first(start, zb):
        k = start
        post = (234).to_bytes(32, "big") + (345).to_bytes(32, "big") + b"EIP-7503"
        while any(synth.keccak256(k.to_bytes(32, "big") + post)[:zb]):
            k += 1
        return k
    k1, t1 = pob_b200.pow_grind(813, 234, 345, zero_bytes=1)
    assert k1 == cpu_first(813, 1) and t1 == k1 - 813 + 1
    k2, _ = pob_b200.pow_grind(40000, 234, 345, zero_bytes=2)
    assert k2 == cpu_first(40000, 2)
    big = (1 << 200) + 12345                                   # carries across limbs, random large key
    k3, _ = pob_b200.pow_grind(big, 7, 9, zero_bytes=2)
    assert k3 >= big and synth.keccak256(k3.to_bytes(32, "big") + (7).to_bytes(32, "big") + (9).to_bytes(32, "big") + b"EIP-7503")[:2] == b"\x00\x00"
    with pytest.raises(pob_b200.PobError):
        pob_b200.pow_grind(0, 1, 2, zero_bytes=8, max_tries=1 << 16)


def test_cli_matches_reference_argv(tmp_path):
    """`python -m pob_b200 main_spend input.json witness.wtns` == the reference `./main_spend input.json witness.wtns`
    (Makefile:6): same file the oracle writes; a failing input exits non-zero and writes nothing."""
    import json, subprocess, sys, os
    from oracle import oracle
    s = suite("test_spend")
    inp, out = str(tmp_path / "input.json"), str(tmp_path / "witness.wtns")
    json.dump(s["cases"][0]["input"], open(inp, "w"))
    env = dict(os.environ, PYTHONPATH=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "proof-of-burn_b200"))
    r = subprocess.run([sys.executable, "-m", "pob_b200", "main_spend", inp, out], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    w = oracle.run("Spend(31)", s["cases"][0]["input"]); ref = str(tmp_path / "ref.wtns"); w.write_wtns(ref); w.free()
    assert open(out, "rb").read() == open(ref, "rb").read()
    bad, out2 = str(tmp_path / "bad.json"), str(tmp_path / "bad.wtns")
    json.dump(s["cases"][1]["input"], open(bad, "w"))
    r = subprocess.run([sys.executable, "-m", "pob_b200", "main_spend", bad, out2], env=env, capture_output=True, text=True)
    assert r.returncode != 0 and r.stderr and not os.path.exists(out2)


def test_non_canonical_input_limbs_are_reduced():
    """limbs >= p handed straight to the C-ABI are reduced mod p (circom's loader semantics): p + x behaves as x"""
    import pob_b200
    s = suite("test_spend")
    c = pob_b200.Circuit("Spend(31)", max_slots=2)
    try:
        packed = c.pack([s["cases"][0]["input"], s["cases"][0]["input"]])
        v = pob_b200.from_limbs(packed[1, 3]) + pob_b200.P          # extraCommitment + p, still < 2^256
        packed[1, 3] = [(v >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)]
        res = c.run_packed(packed, digest=True)
        assert (res.status == 0).all() and res.outputs[0] == res.outputs[1] and res.digests[0] == res.digests[1]
    finally:
        c.close()


def test_cli_batch_mode(tmp_path):
    import json, subprocess, sys, os
    from oracle import oracle
    s = suite("test_spend")
    files = []
    for i in (0, 3, 1):                       # two accepted inputs and one that must be rejected
        f = str(tmp_path / ("case%d.json" % i)); json.dump(s["cases"][i]["input"], open(f, "w")); files.append(f)
    out = str(tmp_path / "out")
    env = dict(os.environ, PYTHONPATH=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "proof-of-burn_b200"))
    r = subprocess.run([sys.executable, "-m", "pob_b200", "main_spend", "--batch"] + files + ["--out", out], env=env, capture_output=True, text=True)
    assert r.returncode == 1 and "case1.json" in r.stderr
    assert sorted(os.listdir(out)) == ["case0.wtns", "case3.wtns"]
    w = oracle.run("Spend(31)", s["cases"][3]["input"]); ref = str(tmp_path / "ref.wtns"); w.write_wtns(ref); w.free()
    assert open(os.path.join(out, "case3.wtns"), "rb").read() == open(ref, "rb").read()


def test_commitments_of_a_batch_match_the_formula_independently_of_the_oracle():
    """Size-independent property at the full main shape: for every instance of a 48-instance synthetic batch the output
    signal equals keccak(blockRoot | nullifier | remainingCoin | revealAmount | burnExtraCommitment |
    _proofExtraCommitment) >> 8 (reference tests/testcases/proof_of_burn.py:18-36), computed with the pure-Python
    keccak / Poseidon of pob_b200.synth -- no oracle involved.  Also witness[0] = 1 and the input section of a resident
    witness equals the packed inputs (circuits/proof_of_burn.circom:43-72 order)."""
    import pob_b200
    from pob_b200 import synth
    shape = (16, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
    insts = synth.make_batch(48, shape, seed=4242)
    packed = synth.pack_instances(insts, shape)
    c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN)
    try:
        res = c.run_packed(packed, retain=[47])                # 48 evaluated, one witness materialised
        assert (res.status == 0).all()
        for i, it in enumerate(insts):
            block_root = synth.keccak256(it["blockHeader"])
            nullifier = synth.poseidon([synth.POSEIDON_PREFIX + 1, it["burnKey"]])
            coin = synth.poseidon([synth.POSEIDON_PREFIX + 2, it["burnKey"], it["intendedBalance"] - it["revealAmount"]])
            msg = block_root + b"".join(int(v).to_bytes(32, "big") for v in
                                        (nullifier, coin, it["revealAmount"], it["burnExtraCommitment"], it["_proofExtraCommitment"]))
            assert res.outputs[i] == [int.from_bytes(synth.keccak256(msg)[:31], "big")], "instance %d" % i
        head = c.witness(47, 0, 2 + c.n_inputs)
        assert pob_b200.from_limbs(head[0]) == 1 and res.outputs[47] == [pob_b200.from_limbs(head[1])]
        assert np.array_equal(head[2:], packed[47])
    finally:
        c.close()


def test_on_gpu_keccak_selfcheck_detects_corruption():
    """pob_selfcheck_keccak: every KeccakfRound block of a materialised witness satisfies out == KeccakRound(in); a single
    flipped bit inside the in/out signals of one block is detected, and only that block fails."""
    import pob_b200
    s = suite("test_keccak_2")
    c = pob_b200.Circuit("KeccakBytes(2)", max_slots=2)
    try:
        res = c.run([s["cases"][3]["input"]])
        assert res.status[0] == 0
        assert c.selfcheck_keccak(0) == (48, 0)
        w = c.witness(0)
        dptr = c.witness_device_ptr(0)
        detected = 0
        for idx in range(c.n_signals - 1, 0, -4001):        # ~1280 probes; 3 % of the entries are in/out of a round block
            if w[idx, 1:].any() or w[idx, 0] > 1:
                continue
            cuda_poke(dptr, idx, int(w[idx, 0]) ^ 1)
            nb, bad = c.selfcheck_keccak(0)
            cuda_poke(dptr, idx, int(w[idx, 0]))
            assert nb == 48 and bad in (0, 1)
            detected += bad
        assert detected >= 1, "no injected fault was detected"
        assert c.selfcheck_keccak(0) == (48, 0)
        assert np.array_equal(c.witness(0), w)
    finally:
        c.close()


def test_selfcheck_main_shape_all_blocks_pass():
    import pob_b200
    from pob_b200 import synth
    shape = (16, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
    insts = synth.make_batch(2, shape, seed=77)
    c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN, max_slots=2)
    try:
        res = c.run_packed(synth.pack_instances(insts, shape))
        assert (res.status == 0).all()
        assert c.selfcheck_keccak(0) == (2016, 0) and c.selfcheck_keccak(1) == (2016, 0)
    finally:
        c.close()
