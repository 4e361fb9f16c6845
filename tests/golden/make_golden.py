"""Regenerates tests/golden/* from the reference's own fixtures: `python tests/golden/make_golden.py <checkout of
zkHubHQ/distributed-groth16>`.  The tests read only what this writes, never the checkout.  Everything copied here is
test DATA (goldens the reference's tests hold), never source:

  sha256_proof.bin            zk-cli/test-circuits/sha256/proof.bin  (128 B, the only full-prover golden)
  reference_goldens.json      - decimal coordinates of that proof as printed in zk-cli/README.md:82
                              - Montgomery byte goldens ark-circom/src/zkey.rs:417-455 (Fq one, G1 gen, G2 gen)
                              - snarkjs proof / vk / public of fixtures/million (pairing KAT)
                              - r1cs / zkey header primes (BN254 check, r1cs_reader.rs:180-188)
  complex_circuit.zkey.pk.npz the proving key of ark-circom/test-vectors/complex-circuit/*.zkey as limb arrays
                              (+ QAP matrices in COO form) -- fixture F1 of SURVEY 8c
  sha256_circuit.npz          fixture F2: fixtures/sha256/sha256.r1cs as COO matrices + the witness for {a: 1, b: 2}
                              computed by running fixtures/sha256/sha256_js/sha256.wasm under oracle/wasm_witness.py
                              (public output == the KAT of groth16/examples/sha256.rs:231-233; all 30 134 constraints hold)
  complex_circuit_proof.json  the oracle's proof for witness a = 3 on that key (r = s = 0 and r, s != 0),
                              both verified against the zkey's own vk with the oracle pairing
  reference_fixtures.npz      what tests/test_formats.py needs beside the files above to rebuild four fixture files
                              byte for byte (SHA-256 of each original): the complex-circuit zkey (section order and
                              section 10), its r1cs (xz-compressed), fixtures/sha256/sha256.r1cs (header, section
                              order, wire label steps) and fixtures/million/witness.wtns (1, 999992, 1, 2, ..., 999991)
"""
import hashlib
import json
import lzma
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import bn254 as o, layout  # noqa: E402

REF = None         # the reference checkout, from the command line


def make_sha256_fixture(g):
    from oracle import wasm_witness
    from distributed_groth16_b200 import formats
    r1 = formats.read_r1cs(open(REF + "/fixtures/sha256/sha256.r1cs", "rb").read())
    w, prime = wasm_witness.calculate_witness(open(REF + "/fixtures/sha256/sha256_js/sha256.wasm", "rb").read(),
                                              {"a": 1, "b": 2})          # zk-cli/test-circuits/sha256/input.json
    assert prime == o.R and len(w) == r1.n_wires == 29823
    assert w[1] == int(g["sha256_public_input"])                        # groth16/examples/sha256.rs:231-233
    wl = np.array([[(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)] for v in w], dtype=np.uint64)
    np.savez_compressed(os.path.join(HERE, "sha256_circuit.npz"), witness=wl,
                        dims=np.array([r1.n_wires, r1.n_pub_out + r1.n_pub_in, r1.n_constraints], dtype=np.uint64),
                        a_rows=r1.rows[0], a_cols=r1.cols[0], a_vals=r1.vals[0], b_rows=r1.rows[1], b_cols=r1.cols[1],
                        b_vals=r1.vals[1], c_rows=r1.rows[2], c_cols=r1.cols[2], c_vals=r1.vals[2])


def main():
    g = {}
    pb = open(REF + "/zk-cli/test-circuits/sha256/proof.bin", "rb").read()
    open(os.path.join(HERE, "sha256_proof.bin"), "wb").write(pb)
    readme = open(REF + "/zk-cli/README.md").read().splitlines()[81]          # line 82: verify transcript
    nums = [int(x) for x in re.findall(r"\d{60,}", readme)]
    assert len(nums) >= 9, len(nums)
    g["sha256_public_input"] = str(nums[0])
    g["sha256_proof_coords"] = dict(a=[str(nums[1]), str(nums[2])],
                                    b=[[str(nums[3]), str(nums[4])], [str(nums[5]), str(nums[6])]],
                                    c=[str(nums[7]), str(nums[8])])
    src = open(REF + "/ark-circom/src/zkey.rs").read()

    def vec_after(name):
        body = src[src.index("fn %s()" % name):]
        body = body[body.index("vec!["):body.index("]")]
        return [int(x) for x in re.findall(r"\d+", body)]

    g["fq_one_mont_bytes"] = vec_after("fq_buf")
    g["g1_gen_mont_bytes"] = vec_after("g1_buf")
    g["g2_gen_mont_bytes"] = vec_after("g2_buf")
    d = REF + "/fixtures/million/"
    g["snarkjs_million"] = dict(vk=json.load(open(d + "verification_key.json")), proof=json.load(open(d + "proof.json")),
                                public=json.load(open(d + "public.json")))
    # (ark-circom/test-vectors/{proof,public,verification_key}.json is a stale triple: it does not satisfy the
    #  verification equation -- checked with the oracle pairing -- so it is not used as a fixture)
    r1 = open(REF + "/fixtures/sha256/sha256.r1cs", "rb").read()
    secs = o._sections(r1, b"r1cs")
    off, _ = secs[1][0]
    g["sha256_r1cs_header"] = dict(prime=str(int.from_bytes(r1[off + 4:off + 36], "little")),
                                   n_wires=int.from_bytes(r1[off + 36:off + 40], "little"))
    json.dump(g, open(os.path.join(HERE, "reference_goldens.json"), "w"), indent=1)

    zk = open(REF + "/ark-circom/test-vectors/complex-circuit/complex-circuit-10000-10000.zkey", "rb").read()
    pk, ma, mb, nc = o.read_zkey(zk)

    def coo(m):
        rows, cols, vals = [], [], []
        for i, lc in enumerate(m):
            for v, w in lc:
                rows.append(i); cols.append(w); vals.append(v)
        return np.array(rows, dtype=np.uint32), np.array(cols, dtype=np.uint32), layout.fr_to_arr(vals)

    ar, ac, av = coo(ma)
    br, bc, bv = coo(mb)
    np.savez_compressed(
        os.path.join(HERE, "complex_circuit.zkey.pk.npz"),
        a_query=layout.g1_to_arr(pk.a_query), b_g1_query=layout.g1_to_arr(pk.b_g1_query),
        b_g2_query=layout.g2_to_arr(pk.b_g2_query), l_query=layout.g1_to_arr(pk.l_query),
        h_query=layout.g1_to_arr(pk.h_query), ic=layout.g1_to_arr(pk.ic),
        vk_g1=layout.g1_to_arr([pk.alpha_g1, pk.beta_g1, pk.delta_g1]),
        vk_g2=layout.g2_to_arr([pk.beta_g2, pk.delta_g2, pk.gamma_g2]),
        dims=np.array([pk.n_vars, pk.n_public, pk.domain_size, nc], dtype=np.uint64),
        a_rows=ar, a_cols=ac, a_vals=av, b_rows=br, b_cols=bc, b_vals=bv)
    z = [0] * pk.n_vars
    z[0], z[2] = 1, 3
    for i in range(3, pk.n_vars):
        z[i] = z[i - 1] * z[i - 1] % o.R
    z[1] = z[pk.n_vars - 1] ** 2 % o.R
    qa, qb, qc = o.qap(ma, mb, pk.n_public + 1, nc, z)
    h = o.h_circom(qa, qb, qc)
    out = {}
    for name, (r, s) in dict(r0s0=(0, 0), r_s=(12345, 67890)).items():
        A, B, C = o.groth16_prove(pk, z, h, r, s)
        assert o.groth16_verify(pk.alpha_g1, pk.beta_g2, pk.gamma_g2, pk.delta_g2, pk.ic, [z[1]], A, B, C)
        out[name] = dict(r=r, s=s, proof_hex=o.proof_compress(A, B, C).hex())
    out["public_input"] = str(z[1])
    json.dump(out, open(os.path.join(HERE, "complex_circuit_proof.json"), "w"), indent=1)
    make_sha256_fixture(g)
    make_fixture_rebuild_data()
    print("golden files written")


def make_fixture_rebuild_data():
    sha = lambda b: np.array(hashlib.sha256(b).hexdigest())
    order = lambda secs: np.array(sorted(secs, key=lambda sid: secs[sid][0][0]), dtype=np.uint32)
    zk = open(REF + "/ark-circom/test-vectors/complex-circuit/complex-circuit-10000-10000.zkey", "rb").read()
    zs = o._sections(zk, b"zkey")
    (o10, l10), = zs[10]
    cr = open(REF + "/ark-circom/test-vectors/complex-circuit/complex-circuit-10000-10000.r1cs", "rb").read()
    sr = open(REF + "/fixtures/sha256/sha256.r1cs", "rb").read()
    ss = o._sections(sr, b"r1cs")
    (o1, l1), = ss[1]
    (o3, l3), = ss[3]
    labels = np.frombuffer(sr, dtype="<u8", count=l3 // 8, offset=o3)
    wtns = open(REF + "/fixtures/million/witness.wtns", "rb").read()
    np.savez_compressed(
        os.path.join(HERE, "reference_fixtures.npz"),
        complex_zkey_sha256=sha(zk), complex_zkey_section_order=order(zs),
        complex_zkey_section10=np.frombuffer(zk, dtype=np.uint8, count=l10, offset=o10),
        complex_r1cs_sha256=sha(cr), complex_r1cs_xz=np.frombuffer(lzma.compress(cr, preset=9 | lzma.PRESET_EXTREME), dtype=np.uint8),
        sha256_r1cs_sha256=sha(sr), sha256_r1cs_section_order=order(ss),
        sha256_r1cs_header=np.frombuffer(sr, dtype=np.uint8, count=l1, offset=o1),
        sha256_r1cs_label_steps=np.diff(labels, prepend=0).astype(np.uint32),
        million_wtns_sha256=sha(wtns))


if __name__ == "__main__":
    REF = os.path.abspath(sys.argv[1])
    main()
