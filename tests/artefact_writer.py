"""Test-side writers for snarkjs / circom artefacts (zkey / wtns / r1cs), so that the product readers are exercised from
data stored under tests/golden.  The zkey byte layout follows ark-circom/src/zkey.rs:53-387 (sections 1-9)."""
import struct

import numpy as np

Q = 21888242871839275222246405745257275088696311157297823662689037894645226208583
R = 21888242871839275222246405745257275088548364400416034343698204186575808495617


def _sec(sid, payload):
    return struct.pack("<IQ", sid, len(payload)) + payload


def write_zkey(d, section_order=range(1, 10), extra_sections=None, coefs_by_constraint=False) -> bytes:
    """d: the npz produced by tests/golden/make_golden.py (limb arrays; coefficient values in Montgomery form).
    section_order, extra_sections ({id: payload}, e.g. snarkjs' section 10 of contributions) and coefs_by_constraint
    (records ordered by constraint, then matrix, as snarkjs writes them) reproduce a snarkjs-made file byte for byte."""
    from oracle import bn254 as o, layout
    n_vars, n_public, m, nc = (int(x) for x in d["dims"])
    hdr = struct.pack("<I", 32) + Q.to_bytes(32, "little") + struct.pack("<I", 32) + R.to_bytes(32, "little")
    hdr += struct.pack("<III", n_vars, n_public, m)
    vk1, vk2 = d["vk_g1"], d["vk_g2"]           # vk_g1 = alpha, beta1, delta1 ; vk_g2 = beta2, delta2, gamma2
    hdr += vk1[0].tobytes() + vk1[1].tobytes() + vk2[0].tobytes() + vk2[2].tobytes() + vk1[2].tobytes() + vk2[1].tobytes()
    # coefficients: file stores value * R^2; the npz holds Montgomery form (value * R) -> multiply by R once more
    coefs = []
    for mi, key in ((0, "a"), (1, "b")):
        vals = layout.arr_to_fr(d[key + "_vals"])
        for r_, c_, v in zip(d[key + "_rows"], d[key + "_cols"], vals):
            coefs.append(struct.pack("<III", mi, int(r_), int(c_)) + (v * o.MONT_R * o.MONT_R % o.R).to_bytes(32, "little"))
    # snarkjs appends the public-input rows (constraint index nc + j): they fix max_constraint_index (zkey.rs:171)
    for j in range(n_public + 1):
        coefs.append(struct.pack("<III", 0, nc + j, j) + (o.MONT_R * o.MONT_R % o.R).to_bytes(32, "little"))
    if coefs_by_constraint:
        coefs.sort(key=lambda rec: struct.unpack_from("<II", rec)[::-1])       # stable: (constraint, matrix)
    sec4 = struct.pack("<I", len(coefs)) + b"".join(coefs)
    secs = {1: struct.pack("<I", 1), 2: hdr, 3: d["ic"].tobytes(), 4: sec4, 5: d["a_query"].tobytes(),
            6: d["b_g1_query"].tobytes(), 7: d["b_g2_query"].tobytes(), 8: d["l_query"].tobytes(), 9: d["h_query"].tobytes()}
    secs.update(extra_sections or {})
    body = [_sec(sid, secs[sid]) for sid in section_order]
    return b"zkey" + struct.pack("<II", 1, len(body)) + b"".join(body)


def write_r1cs(header: bytes, matrices, labels, section_order=(1, 2, 3)) -> bytes:
    """header: the 64-byte section 1 (field size, prime, wire / input counts, label count, constraint count);
    matrices: (rows, cols, canonical value limbs) of A, B and C, rows ascending; labels: wire -> label map (section 3)."""
    n_cons = struct.unpack_from("<I", header, 60)[0]
    term = np.dtype([("w", "<u4"), ("v", "<u8", (4,))])
    per_matrix = []
    for rows, cols, vals in matrices:
        t = np.zeros(len(rows), dtype=term)
        t["w"], t["v"] = cols, vals
        per_matrix.append((np.searchsorted(rows, np.arange(n_cons + 1)), t.tobytes()))
    cons = []
    for i in range(n_cons):
        for bounds, raw in per_matrix:
            lo, hi = int(bounds[i]), int(bounds[i + 1])
            cons.append(struct.pack("<I", hi - lo) + raw[lo * term.itemsize:hi * term.itemsize])
    secs = {1: header, 2: b"".join(cons), 3: np.asarray(labels, dtype="<u8").tobytes()}
    return b"r1cs" + struct.pack("<II", 1, len(secs)) + b"".join(_sec(sid, secs[sid]) for sid in section_order)


def write_wtns(values) -> bytes:
    s1 = struct.pack("<I", 32) + R.to_bytes(32, "little") + struct.pack("<I", len(values))
    s2 = b"".join(int(v).to_bytes(32, "little") for v in values)
    return b"wtns" + struct.pack("<II", 2, 2) + _sec(1, s1) + _sec(2, s2)


def f1_witness(n_vars):
    z = [0] * n_vars
    z[0], z[2] = 1, 3
    for i in range(3, n_vars):
        z[i] = z[i - 1] * z[i - 1] % R
    z[1] = z[n_vars - 1] ** 2 % R
    return z
