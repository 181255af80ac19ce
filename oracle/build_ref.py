"""Recipe for `oracle/_ref`: a byte-for-byte copy of the reference's python package so that the UNMODIFIED reference
can run on the GPU box, where /root/reference does not exist.

TEST / MEASUREMENT INFRASTRUCTURE.  `oracle/_ref/` is git-ignored (no reference source enters the history) but not
gpurun-ignored, so it travels with the snapshot like the built `.so`.  It is used by
  * `bench.py --impl reference`  (cpu_baseline.kind = "reference": the reference's own `alg.local_update` on the host
    cores) and the `gpu_eager_baseline` leg (the same code with `use_gpu=True`, the "existing Blackwell path").
No test needs it, and nothing under `gops_b200/` imports it.

Run:  python oracle/build_ref.py          (also called by __graft_entry__.build() when /root/reference exists)
Copies  <reference>/gops/**/*.py  (+ the shipped FHADP idpendulum checkpoint and its config used as a known answer)
into oracle/_ref/, and writes oracle/_ref/MANIFEST.json (file count, sha256 of the concatenated sources, reference
commit if a .git is present) so that a stale copy is detectable.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
SRC = os.environ.get("GOPS_REFERENCE_SRC", "/root/reference")
EXTRA = [os.path.join("results", "FHADP", "idpendulum", "apprfunc", "apprfunc_100000.pkl"),
         os.path.join("results", "FHADP", "idpendulum", "config.json")]


def _sources():
    root = os.path.join(SRC, "gops")
    for d, _, files in sorted(os.walk(root)):
        for f in sorted(files):
            if f.endswith(".py"):
                yield os.path.relpath(os.path.join(d, f), SRC)


def digest(base):
    h = hashlib.sha256()
    n = 0
    root = os.path.join(base, "gops")
    for d, _, files in sorted(os.walk(root)):
        for f in sorted(files):
            if f.endswith(".py"):
                h.update(open(os.path.join(d, f), "rb").read())
                n += 1
    return n, h.hexdigest()


def build(force=False):
    if not os.path.isdir(os.path.join(SRC, "gops")):
        return False            # GPU box: use the copy that travelled with the snapshot
    man = os.path.join(DST, "MANIFEST.json")
    n_src, h_src = digest(SRC)
    if not force and os.path.exists(man):
        try:
            m = json.load(open(man))
            if m.get("sha256") == h_src and m.get("files") == n_src:
                return True
        except Exception:
            pass
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    for rel in list(_sources()) + [e for e in EXTRA if os.path.exists(os.path.join(SRC, e))]:
        dst = os.path.join(DST, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(os.path.join(SRC, rel), dst)
    n, h = digest(DST)
    assert (n, h) == (n_src, h_src), "copy differs from the reference"
    json.dump({"files": n, "sha256": h, "source": SRC}, open(man, "w"), indent=1)
    return True


if __name__ == "__main__":
    ok = build(force="--force" in sys.argv)
    print("oracle/_ref:", "built" if ok else "reference tree not present (nothing to do)")
