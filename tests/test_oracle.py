"""CPU: the oracle against the reference's own known-answer vectors and property tests
(SURVEY.md section 8c), the C restatement against the Python one, and the committed golden file."""
import os

import numpy as np
import pytest

from conftest import hx, mont, unmont

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_reference_kats(oracle):
    """src/hades.rs:128-162: 6 absolute digests (tag 0, padding one)."""
    ins = oracle.kat_inputs()
    for n, want in oracle.KAT_EXPECTED.items():
        assert oracle.debug_hex(oracle.kat_poseidon_hash(ins[:n])) == want


def test_constants_match_reference_assets(oracle):
    """Constants regenerated from assets/HOWTO.md equal the reference's .bin files byte for byte
    (tests/golden/arc.bin and mds.bin are unmodified copies of dusk-poseidon's assets/arc.bin and assets/mds.bin)."""
    with open(os.path.join(GOLDEN, "arc.bin"), "rb") as f:
        assert oracle.arc_bin_bytes() == f.read()
    with open(os.path.join(GOLDEN, "mds.bin"), "rb") as f:
        assert oracle.mds_bin_bytes() == f.read()


def test_round_constants_nonzero_and_roundtrip(oracle):
    """src/hades/round_constants.rs:61-70"""
    assert len(oracle._ARC_FLAT) == 340
    for c in oracle._ARC_FLAT:
        assert c != 0 and c < oracle.P
        assert int.from_bytes(c.to_bytes(32, "little"), "little") == c


def test_hades_det(oracle):
    """src/hades/permutation/scalar.rs:86-98"""
    x, y, z = oracle.perm([17] * 5), oracle.perm([17] * 5), oracle.perm([19] * 5)
    assert x == y and x != z


def test_readme_doctest_properties(oracle):
    """README.md:37-50: chunked update == one-shot digest; Merkle4 != Other on the same 4 inputs."""
    import random
    rnd = random.Random(0xBEEF)
    x = [rnd.randrange(oracle.P) for _ in range(42)]
    one = oracle.Hash.digest(oracle.Domain.Other, x)
    h = oracle.Hash(oracle.Domain.Other)
    h.update(x[:3])
    h.update(x[3:])
    assert h.finalize() == one
    assert oracle.Hash.digest(oracle.Domain.Merkle4, x[:4]) != oracle.Hash.digest(oracle.Domain.Other, x[:4])


def test_merkle_arity_violation(oracle):
    """src/hash.rs:71-76"""
    for dom, n in ((oracle.Domain.Merkle4, 3), (oracle.Domain.Merkle4, 5), (oracle.Domain.Merkle2, 3)):
        with pytest.raises(oracle.IOPatternViolation):
            oracle.Hash.digest(dom, [1] * n)


def test_output_len_rule(oracle):
    """src/hash.rs:111-115: output_len only for Domain::Other and > 0"""
    h = oracle.Hash(oracle.Domain.Merkle4)
    h.output_len(3)
    h.update([1, 2, 3, 4])
    assert len(h.finalize()) == 1
    h = oracle.Hash(oracle.Domain.Other)
    h.output_len(0)
    h.update([1, 2, 3])
    assert len(h.finalize()) == 1
    h.output_len(7)
    assert len(h.finalize()) == 7


def test_encryption_properties(oracle):
    """tests/encryption.rs:31-115 and src/encryption.rs:29-42"""
    import random
    rnd = random.Random(0x42424242)
    for L in (3, 21, 42):
        msg = [rnd.randrange(oracle.P) for _ in range(L)]
        sec = [rnd.randrange(oracle.P), rnd.randrange(oracle.P)]
        nonce = rnd.randrange(oracle.P)
        cipher = oracle.encrypt(msg, sec, nonce)
        assert len(cipher) == L + 1                       # src/encryption.rs:61
        assert oracle.decrypt(cipher, sec, nonce) == msg
        with pytest.raises(oracle.DecryptionFailed):
            oracle.decrypt(cipher, [sec[0], (sec[1] + 1) % oracle.P], nonce)
        with pytest.raises(oracle.DecryptionFailed):
            oracle.decrypt(cipher, sec, (nonce + 1) % oracle.P)
        for idx in (L, 0):
            bad = list(cipher)
            bad[idx] = (bad[idx] + 42) % oracle.P
            with pytest.raises(oracle.DecryptionFailed):
                oracle.decrypt(bad, sec, nonce)
    assert oracle.decrypt(oracle.encrypt([10, 20, 30], [5, 6], 7), [5, 6], 7) == [10, 20, 30]


def test_golden_file_matches_oracle(oracle, golden):
    for e in golden["perm"]:
        assert [oracle.debug_hex(v) for v in oracle.perm([hx(s) for s in e["in"]])] == e["out"]
    # the vectors listed in SURVEY.md 8(c)
    assert golden["perm"][0]["out"][0] == "0x4b9d72d92f0ba052ad683a030a4a0de861e8b84c5929397e195b516a7927971a"
    assert golden["perm"][1]["out"][4] == "0x63d231187fc467edd22ce38374db305267e9fb211723b766f0c608914f70f032"
    assert golden["perm"][4]["out"][0] == "0x4fd86cf4af6a218f186d995890a4b8bbfb90388cff65577243b7a25a329ed1ba"
    for e in golden["digest"]:
        h = oracle.Hash(e["domain"])
        h.output_len(e["out_len"])
        h.update([hx(s) for s in e["in"]])
        assert [oracle.debug_hex(v) for v in h.finalize()] == e["out"]
    for e in golden["encrypt"]:
        c = oracle.encrypt([hx(s) for s in e["msg"]], [hx(s) for s in e["secret"]], hx(e["nonce"]))
        assert [oracle.debug_hex(v) for v in c] == e["cipher"]


def test_c_oracle_matches_python(oracle, coracle, golden):
    rng = np.random.default_rng(5)
    # permutation
    ins = [[hx(s) for s in e["in"]] for e in golden["perm"]]
    out = coracle.permute(mont(ins))
    for row, e in zip(out, golden["perm"]):
        assert [oracle.debug_hex(v) for v in unmont(row)] == e["out"]
    # KATs through the C sponge
    kin = oracle.kat_inputs()
    for n, want in oracle.KAT_EXPECTED.items():
        d = coracle.digest_padded(mont(0), mont(kin[:n]).reshape(1, n, 4), n, mont(1))
        assert oracle.debug_hex(unmont(d)[0]) == want
    # digests with real tags
    for e in golden["digest"]:
        pat = [oracle.Absorb(len(e["in"])), oracle.Squeeze(e["out_len"])]
        tag = oracle.hash_to_scalar(oracle.tag_input(pat, e["domain"]))
        d = coracle.digest(mont(tag), mont([hx(s) for s in e["in"]]).reshape(1, -1, 4), len(e["in"]), e["out_len"])
        assert [oracle.debug_hex(v) for v in unmont(d[0])] == e["out"]
    # encryption
    for e in golden["encrypt"]:
        L = e["L"]
        tag = mont(hx(golden["tags"]["encrypt2"])) if L == 2 else mont(oracle.hash_to_scalar(oracle.tag_input(
            [oracle.Absorb(2), oracle.Absorb(1), oracle.Squeeze(L), oracle.Absorb(L), oracle.Squeeze(1)],
            oracle.Domain.Encryption)))
        msg = mont([hx(s) for s in e["msg"]]).reshape(1, L, 4)
        sec = mont([hx(s) for s in e["secret"]]).reshape(1, 2, 4)
        non = mont(hx(e["nonce"])).reshape(1, 4)
        c = coracle.encrypt(tag, msg, L, sec, non)
        assert [oracle.debug_hex(v) for v in unmont(c[0])] == e["cipher"]
        m, ok = coracle.decrypt(tag, c, L, sec, non)
        assert ok[0] == 1 and np.array_equal(m, msg)
        c[0, 0, 0] ^= np.uint64(1)
        m, ok = coracle.decrypt(tag, c, L, sec, non)
        assert ok[0] == 0
    # multi-thread wrapper == single thread
    s = mont([[int(v) for v in rng.integers(0, 1 << 62, 5)] for _ in range(64)])
    assert np.array_equal(coracle.permute(s), coracle.permute(s, threads=4))


def test_merkle_golden_vs_c_oracle(golden, coracle, oracle):
    """CPU: the committed tree / opening vectors (Python oracle) agree with the C port level by level."""
    from conftest import hx, mont, unmont
    for t in golden["merkle"]:
        arity = t["arity"]
        dom = oracle.Domain.Merkle4 if arity == 4 else oracle.Domain.Merkle2
        tag = mont(oracle.hash_to_scalar(oracle.tag_input([oracle.Absorb(arity), oracle.Squeeze(1)], dom)))
        cur, nodes = mont([hx(v) for v in t["leaves"]]), []
        while cur.shape[0] > 1:
            cur = coracle.digest(tag, cur.reshape(-1, arity, 4), arity, 1).reshape(-1, 4)
            nodes += ["0x%064x" % v for v in unmont(cur)]
        assert nodes == t["nodes"]
        assert t["opening"][0][t["opening_leaf"] % arity] == t["leaves"][t["opening_leaf"]]
