"""Product-side artefact readers (distributed_groth16_b200/formats.py), CPU only."""
import hashlib
import lzma
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
G = os.path.join(HERE, "golden")


def test_zkey_and_wtns_roundtrip_through_test_writer():
    import artefact_writer as aw
    from distributed_groth16_b200 import formats
    d = np.load(os.path.join(G, "complex_circuit.zkey.pk.npz"))
    zk = formats.read_zkey(aw.write_zkey(d))
    n_vars, n_public, m, nc = (int(x) for x in d["dims"])
    assert (zk.n_vars, zk.n_public, zk.domain_size, zk.num_constraints) == (n_vars, n_public, m, nc)
    for k in ("a_query", "b_g1_query", "b_g2_query", "l_query", "h_query", "ic"):
        assert (getattr(zk, k) == d[k]).all(), k
    assert (zk.vk_points() == np.concatenate([d["vk_g1"].reshape(-1), d["vk_g2"][:2].reshape(-1)])).all()
    z = aw.f1_witness(n_vars)
    w = formats.read_wtns(aw.write_wtns(z))
    assert w.shape == (n_vars, 4) and int.from_bytes(w[5].tobytes(), "little") == z[5]
    ptr, col, val = formats.coo_to_csr(zk.coef_row[zk.coef_matrix == 0], zk.coef_col[zk.coef_matrix == 0],
                                       zk.coef_val_r2[zk.coef_matrix == 0], nc)
    assert ptr[-1] == nc and (col[:3] == d["a_cols"][:3]).all()
    with pytest.raises(formats.FormatError):
        formats.read_zkey(b"nope" + bytes(64))


def _reference_fixture(name):
    """The reference's fixture files (ark-circom/test-vectors/complex-circuit/complex-circuit-10000-10000.{zkey,r1cs},
    fixtures/sha256/sha256.r1cs, fixtures/million/witness.wtns), rebuilt from tests/golden and checked byte for byte
    against the SHA-256 of the original (tests/golden/make_golden.py)."""
    import artefact_writer as aw
    f = np.load(os.path.join(G, "reference_fixtures.npz"))
    if name == "complex_zkey":
        buf = aw.write_zkey(np.load(os.path.join(G, "complex_circuit.zkey.pk.npz")), f["complex_zkey_section_order"],
                            {10: f["complex_zkey_section10"].tobytes()}, coefs_by_constraint=True)
    elif name == "complex_r1cs":
        buf = lzma.decompress(f["complex_r1cs_xz"].tobytes())
    elif name == "sha256_r1cs":
        s = np.load(os.path.join(G, "sha256_circuit.npz"))
        buf = aw.write_r1cs(f["sha256_r1cs_header"].tobytes(), [(s[k + "_rows"], s[k + "_cols"], s[k + "_vals"]) for k in "abc"],
                            np.cumsum(f["sha256_r1cs_label_steps"], dtype=np.uint64), f["sha256_r1cs_section_order"])
    else:                       # million_wtns: in = 1, intermediate[i] = i + 2, out = 999992
        buf = aw.write_wtns([1, 999992] + list(range(1, 999992)))
    assert hashlib.sha256(buf).hexdigest() == str(f[name + "_sha256"]), name
    return buf


def test_readers_on_the_reference_fixtures():
    from distributed_groth16_b200 import formats
    from oracle import bn254 as o
    d = np.load(os.path.join(G, "complex_circuit.zkey.pk.npz"))
    zk = formats.read_zkey(_reference_fixture("complex_zkey"))
    for k in ("a_query", "b_g1_query", "b_g2_query", "l_query", "h_query", "ic"):
        assert (getattr(zk, k) == d[k]).all(), k
    assert zk.num_constraints == int(d["dims"][3])
    w = formats.read_wtns(_reference_fixture("million_wtns"))
    assert w.shape[0] == 999993 and int(w[0, 0]) == 1 and int(w[1, 0]) == 999992
    r1 = formats.read_r1cs(_reference_fixture("sha256_r1cs"))
    assert (r1.n_wires, r1.n_constraints, r1.n_pub_out) == (29823, 30134, 1)
    ref = o.read_r1cs(_reference_fixture("complex_r1cs"))
    mine = formats.read_r1cs(_reference_fixture("complex_r1cs"))
    assert mine.n_constraints == ref["n_constraints"] and int(mine.cols[0][0]) == ref["constraints"][0][0][0][1]


def test_readers_reject_out_of_range_indices():
    """A malformed zkey / r1cs must fail on the host (FormatError), not index device memory out of bounds: the reference panics
    on the same inputs (index out of bounds in ark-circom/src/zkey.rs / circom/r1cs_reader.rs)."""
    import struct
    import artefact_writer as aw
    from distributed_groth16_b200 import formats
    d = np.load(os.path.join(G, "complex_circuit.zkey.pk.npz"))
    good = bytearray(aw.write_zkey(d))
    zk = formats.read_zkey(bytes(good))
    secs = formats._sections(bytes(good), b"zkey")
    o4, _ = secs[4][0]
    bad = bytearray(good)
    struct.pack_into("<I", bad, o4 + 4 + 8, zk.n_vars + 5)             # signal index of the first coefficient record
    with pytest.raises(formats.FormatError):
        formats.read_zkey(bytes(bad))
    bad = bytearray(good)
    struct.pack_into("<I", bad, o4 + 4, 7)                             # matrix index > 1
    with pytest.raises(formats.FormatError):
        formats.read_zkey(bytes(bad))
    bad = bytearray(good)
    struct.pack_into("<I", bad, o4, 0x7FFFFFFF)                        # record count far beyond the section
    with pytest.raises(formats.FormatError):
        formats.read_zkey(bytes(bad))
