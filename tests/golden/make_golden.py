#!/usr/bin/env python
"""Regenerates the committed golden vectors under tests/golden/.

Run from the repo root:  python tests/golden/make_golden.py

Sources
* kats.json            -- hand-transcribed known answers of the reference's own unit and
                          integration tests (file:line beside each), NOT produced by our code.
* fixtures/            -- byte copies of the reference's tests/examples/<dir>/{in,out}.fasta for
                          the canonicalize/uniq path (test DATA, not source), plus test.fasta and the
                          676-record real-monomer corpus (nim_cated.../out.fasta) used as extra input.
* xxh3_vectors.json    -- XXH3-64 (seed 0) of deterministic inputs at every length class and of seeded
                          random bytes, produced by python-xxhash 3.7.0 (libxxhash 0.8.2): an independent
                          implementation of the algorithm xxhash-rust 0.8.6 implements (src/uniq.rs:45).
* oracle_cli/*.out     -- the ORACLE's byte-exact CLI output for each fixture input (the reference's
                          out.fasta files lack the final newline the program writes, src/canonicalize.rs:37,
                          so byte-exact expectations have to come from the source-following oracle).
"""
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def kats():
    return {
        "lmsr_index": [  # lib/src/canonicalize.rs:70-82
            {"in": "AAA", "out": 0, "ref": "lib/src/canonicalize.rs:70-72"},
            {"in": "banana", "out": 5, "ref": "lib/src/canonicalize.rs:75-77"},
            {"in": "TAA", "out": 1, "ref": "lib/src/canonicalize.rs:80-82"},
        ],
        "lmsr": [  # lib/src/canonicalize.rs:89-99
            {"in": "AAA", "out": "AAA", "ref": "lib/src/canonicalize.rs:89-91"},
            {"in": "banana", "out": "abanan", "ref": "lib/src/canonicalize.rs:93-95"},
            {"in": "TAA", "out": "AAT", "ref": "lib/src/canonicalize.rs:97-99"},
        ],
        "lmsr_idempotent": ["ATGCAGATACAGA"],  # lib/src/canonicalize.rs:102-106
        "canonicalize": [  # lib/src/canonicalize.rs:113-119, tests/canon_uniq.rs:24-29
            {"in": "AAA", "out": "AAA", "ref": "lib/src/canonicalize.rs:113-115"},
            {"in": "ATT", "out": "AAT", "ref": "lib/src/canonicalize.rs:117-119"},
            {"in": "ATGCA", "out": "AATGC", "ref": "tests/canon_uniq.rs:24-29"},
        ],
        "same_circle": [  # lib/src/canonicalize.rs:122-132: two rotations of one monomer
            ["AATCAATTTCCTCCATCACCTAGTTTATGTAGAAACGCTGCTA",
             "TCCTCCATCACCTAGTTTATGTAGAAACGCTGCTAAATCAATT"],
        ],
        "cli_fixtures": {  # tests/canon_uniq.rs:35-47 (uniq always with --canonicalize, :69-71)
            "canonicalize": ["simple", "multiple_sequences", "multiple_sequences_split_lines", "rna_input",
                             "compressed_output", "compressed_input"],
            "uniq": ["simple", "multiple_sequences", "multiple_sequences_split_lines", "rna_input", "repeated",
                     "compressed_output", "compressed_input"],
        },
    }


def xxh3_vectors():
    import xxhash
    lens = [0, 1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 96, 97, 127, 128, 129, 143, 144, 160,
            191, 192, 239, 240, 241, 255, 256, 257, 300, 325, 400, 511, 512, 513, 1023, 1024, 1025, 1088, 1089,
            2047, 2048, 2049, 3000, 4096, 5000, 10000, 65536, 200000]
    vec = []
    for L in lens:
        # deterministic DNA-like and binary-like inputs
        dna = bytes(b"ACGT"[(i * 7 + (i >> 3) * 3 + L) & 3] for i in range(L))
        raw = bytes((i * 131 + 17 + L) & 0xFF for i in range(L))
        vec.append({"len": L, "kind": "dna", "xxh3_64": "%016x" % xxhash.xxh3_64_intdigest(dna)})
        vec.append({"len": L, "kind": "raw", "xxh3_64": "%016x" % xxhash.xxh3_64_intdigest(raw)})
    # random bytes: one random.Random(11) stream, consumed length after length in this order
    rng = random.Random(11)
    rnd = []
    for L in list(range(0, 300)) + [1023, 1024, 1025, 2048, 4097, 70000]:
        data = bytes(rng.getrandbits(8) for _ in range(L))
        rnd.append({"len": L, "xxh3_64": "%016x" % xxhash.xxh3_64_intdigest(data)})
    return {"generator": "python-xxhash %s / libxxhash %s" % (xxhash.VERSION, xxhash.XXHASH_VERSION),
            "dna": "bytes(b'ACGT'[(i*7 + (i>>3)*3 + L) & 3] for i in range(L))",
            "raw": "bytes((i*131 + 17 + L) & 0xFF for i in range(L))",
            "random": "rng = random.Random(11), then for each length in order: bytes(rng.getrandbits(8) for _ in range(L))",
            "known": {"": "2d06800538d394c2", "AAT": "a6ab697c798b7cdd"},
            "vectors": vec, "random_vectors": rnd}


def oracle_cli():
    from oracle import cli
    fx = os.path.join(HERE, "fixtures")
    outdir = os.path.join(HERE, "oracle_cli")
    os.makedirs(outdir, exist_ok=True)
    for d in sorted(os.listdir(fx)):
        p = os.path.join(fx, d, "in.fasta")
        if not os.path.isfile(p):
            continue
        data = open(p, "rb").read()
        open(os.path.join(outdir, d + ".canonicalize.out"), "wb").write(cli.cli_canonicalize(data))
        for canon in (False, True):
            out, table = cli.cli_uniq(data, canonicalize=canon, table_ext="csv")
            tag = "uniq_c" if canon else "uniq"
            open(os.path.join(outdir, d + "." + tag + ".out"), "wb").write(out)
            if canon:
                open(os.path.join(outdir, d + ".uniq.table.csv"), "wb").write(table)


if __name__ == "__main__":
    json.dump(kats(), open(os.path.join(HERE, "kats.json"), "w"), indent=1)
    json.dump(xxh3_vectors(), open(os.path.join(HERE, "xxh3_vectors.json"), "w"), indent=0)
    oracle_cli()
    print("golden vectors written to", HERE)
