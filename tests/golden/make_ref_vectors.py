"""Write tests/golden/ref_vectors.json: the answers tests/test_oracle_vs_ref.py holds the oracle port
(and, where it is built, the reference) to, computed by one implementation on that module's inputs.

    python tests/golden/make_ref_vectors.py [--impl reference|port]

`reference` (the default) needs oracle/_ref/libref.so (`make -C oracle ref REF=<reference checkout>`).
`port` records the oracle port's answers instead; the file names its source.
"""
import argparse
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, ".."))
from oracle import oracle as O  # noqa: E402
from test_oracle_vs_ref import VECTORS_PATH, all_answers  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--impl", choices=["reference", "port"], default="reference")
    args = ap.parse_args()
    O.build(ref=args.impl == "reference")
    if args.impl == "reference" and not O.ref_available():
        raise SystemExit("oracle/_ref/libref.so is not built: make -C oracle ref REF=<reference checkout>")
    source = {"reference": "the unmodified reference (oracle/_ref/libref.so)",
              "port": "the oracle port (oracle/rspt_oracle.c)"}[args.impl]
    vectors = {"source": source, **all_answers(O, args.impl)}
    with open(VECTORS_PATH, "w") as f:
        json.dump(vectors, f, indent=0)
        f.write("\n")
    print("wrote", VECTORS_PATH, os.path.getsize(VECTORS_PATH), "bytes from", source)


if __name__ == "__main__":
    main()
