"""TEST / BASELINE INFRASTRUCTURE ONLY -- never imported by the product path (adt_b200/).

Stages the UNMODIFIED reference sources of the hot path from the reference checkout (REF below) into oracle/_ref/,
so that a copy of this tree carries them to a machine without that checkout: oracle/_ref/ is git-ignored (the reference's
sources never enter this repository's history).

    python -m oracle.build_ref            # copies, byte for byte, and writes oracle/_ref/MANIFEST.json (sha256 per file)

`__graft_entry__.build()` calls this.  What is staged:
  sasrec/model.py, sasrec/modules.py                         the SASRecADT model (forward / predict)
  sasrec/supersasrec.py, super_modules.py, base_super_modules.py   the supernet of evolution.py
The loss / clip / Adam lines of sasrec/main.py:146-173 are NOT importable (they sit inside main()); oracle/ref_runner.py
restates those ~25 lines around the staged model, which is what `bench.py --impl reference` and the `cpu_baseline`
leg time (kind: "reference").
"""
import hashlib
import json
import os
import shutil
import sys

# the reference checkout (its sources are not part of this repository): $ADT_REFERENCE_DIR, by default /root/reference
REF = os.environ.get("ADT_REFERENCE_DIR") or "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
FILES = ["sasrec/model.py", "sasrec/modules.py", "sasrec/supersasrec.py", "sasrec/super_modules.py", "sasrec/base_super_modules.py"]


def build(verbose=True):
    if not os.path.isdir(REF):
        if verbose:
            print(f"oracle.build_ref: no reference checkout at {REF} -- keeping the staged copy as it is")
        return os.path.exists(os.path.join(OUT, "MANIFEST.json"))
    manifest = {}
    for rel in FILES:
        src, dst = os.path.join(REF, rel), os.path.join(OUT, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(src, dst)
        with open(dst, "rb") as f:
            manifest[rel] = hashlib.sha256(f.read()).hexdigest()
    with open(os.path.join(OUT, "MANIFEST.json"), "w") as f:
        json.dump({"source": REF, "files": manifest}, f, indent=1)
    if verbose:
        print(f"oracle.build_ref: staged {len(FILES)} unmodified reference files into {OUT}")
    return True


if __name__ == "__main__":
    sys.exit(0 if build() else 1)
