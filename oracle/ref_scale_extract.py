"""Write oracle/_ref/gen/sw_methods_scaled.inc: the verbatim blocks of sw_methods.inc (oracle/ref_extract.py) without the
cut getScale block, which the useScale build of the reference supplies from a spec (oracle/ref_scale/sw_methods.inc).
Whole blocks are dropped, each kept block keeps its "verbatim file:lines" header, so the result is verbatim too.

    python oracle/ref_scale_extract.py [--gen oracle/_ref/gen]
"""
import argparse
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))


def main(gen):
    with open(os.path.join(gen, "sw_methods.inc"), encoding="utf-8", errors="surrogateescape") as fh:
        text = fh.read()
    starts = [m.start() for m in re.finditer(r"^// ---- verbatim ", text, re.M)]
    head, blocks = text[:starts[0]], [text[a:b] for a, b in zip(starts, starts[1:] + [len(text)])]
    keep = [b for b in blocks if not re.search(r"inline Eigen::Matrix3d getScale\(const double t\)", b)]
    assert len(keep) == len(blocks) - 1, "expected exactly one getScale block"
    with open(os.path.join(gen, "sw_methods_scaled.inc"), "w", encoding="utf-8", errors="surrogateescape") as fh:
        fh.write(head + "".join(keep))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gen", default=os.path.join(HERE, "_ref", "gen"))
    main(ap.parse_args().gen)
