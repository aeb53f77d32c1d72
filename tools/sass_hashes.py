#!/usr/bin/env python
"""Per-kernel SASS fingerprints of serf_b200/libserfsim.so.

  python tools/sass_hashes.py --write profiles/<name>.json     record the fingerprints of the current build
  python tools/sass_hashes.py --check profiles/<name>.json     list the kernels whose machine code differs from that record

Used to state precisely which kernels changed since the build a GPU parity run last passed on (source refactors that
leave the machine code untouched — launch macros, host-only #ifdefs — show up as "no kernel changed")."""
import argparse
import hashlib
import json
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ANON = re.compile(r"_GLOBAL__N__[0-9a-f]{8}_\d+_\w+?_cu_[0-9a-f]{8}")


def fingerprints(so):
    txt = subprocess.check_output(["cuobjdump", "-sass", so], text=True)
    txt = "\n".join(l for l in txt.splitlines() if not re.match(r"^\s*//(## |--)", l))
    out = {}
    for part in re.split(r"\n\s*Function : ", txt)[1:]:
        name, body = part.split("\n", 1)
        body = ANON.sub("ANON", body.split("Fatbin elf code")[0].rstrip())
        body = re.sub(r"[ \t]+", " ", body)              # cuobjdump pads the comment column to the longest line of the WHOLE listing
        out[ANON.sub("ANON", name.strip())] = hashlib.sha256(body.encode()).hexdigest()[:16]
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--so", default=os.path.join(ROOT, "serf_b200", "libserfsim.so"))
    ap.add_argument("--write")
    ap.add_argument("--check")
    a = ap.parse_args()
    fp = fingerprints(a.so)
    if a.write:
        json.dump(fp, open(a.write, "w"), indent=0, sort_keys=True)
        print(f"{len(fp)} kernels → {a.write}")
    if a.check:
        ref = json.load(open(a.check))
        changed = sorted(k for k in ref if k in fp and fp[k] != ref[k])
        removed = sorted(k for k in ref if k not in fp)
        new = sorted(k for k in fp if k not in ref)
        print(f"{len(ref) - len(changed) - len(removed)} of {len(ref)} recorded kernels unchanged")
        for k in changed:
            print("  changed:", k)
        for k in removed:
            print("  removed:", k)
        for k in new:
            print("  new:    ", k)
