"""Goldens of the read ingestion: the UNMODIFIED reference reader (DataLayer/FastaReader.cpp through oracle/_ref/ref_arith
reads dump, built by `make -C oracle ref`) on the seeded files of tests/test_host_reader.py, with every reader option set
those tests use.  Writes reader_cases.json (sha256 and line count of each output).

    python tests/golden/make_golden_reader.py
"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_host_reader as t  # noqa: E402

REF_ARITH = os.path.join(ROOT, "oracle", "_ref", "ref_arith")


def dump(paths, opts=None):
    r = subprocess.run([REF_ARITH, "reads", "dump", *paths], capture_output=True, text=True, check=True,
                       env=dict(os.environ, **{"REF_" + k: v for k, v in (opts or {}).items()}))
    return r.stdout


def main():
    out = {}
    with tempfile.TemporaryDirectory() as d:
        text = dump(t.reference_reader_inputs(d))
        assert d not in text
        out["fastq_fasta_gz"] = t.golden_digest(text)
    out["formats"] = {}
    for opts in t.READER_OPTS:
        with tempfile.TemporaryDirectory() as d:
            text = dump(t.format_inputs(d), opts)
            assert d not in text
            out["formats"][t.opts_key(opts)] = t.golden_digest(text)
    with open(os.path.join(HERE, "reader_cases.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
