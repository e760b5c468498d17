"""Install the UNMODIFIED reference into ``baseline/_ref`` (git-ignored).

The prescribed ``pip install --no-index --no-build-isolation --find-links /opt/wheelhouse
--target baseline/_ref /root/reference`` fails because the reference has neither ``setup.py`` nor
``pyproject.toml`` ("Directory ... is not installable", recorded in DESIGN.md) -- it is four flat
scripts.  So the install is a byte-for-byte copy of those scripts, verified against the SHA-256 list
committed in ``baseline/REF_SHA256.json`` (hashes of /root/reference at survey time)."""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
FILES = ["train_dist.py", "gloo.py", "allreduce.py", "ptp.py", "tuto.md", "LICENSE", "README.md"]
SHA_FILE = os.path.join(HERE, "REF_SHA256.json")


def sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def verify(dst=DST):
    if not os.path.isfile(SHA_FILE):
        return False, "REF_SHA256.json missing"
    want = json.load(open(SHA_FILE))
    for name, h in want.items():
        p = os.path.join(dst, name)
        if not os.path.isfile(p):
            return False, f"{name} missing"
        if sha(p) != h:
            return False, f"{name} differs from the reference (sha256 mismatch)"
    return True, "ok"


def install(src, dst=DST, record=False):
    if not os.path.isdir(src):
        return verify(dst)
    os.makedirs(dst, exist_ok=True)
    for name in FILES:
        s = os.path.join(src, name)
        if os.path.isfile(s):
            shutil.copyfile(s, os.path.join(dst, name))
    if record or not os.path.isfile(SHA_FILE):
        json.dump({n: sha(os.path.join(src, n)) for n in FILES if os.path.isfile(os.path.join(src, n))},
                  open(SHA_FILE, "w"), indent=1, sort_keys=True)
    return verify(dst)


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if a != "--record"]
    if len(args) != 1:
        sys.exit("usage: python baseline/install_ref.py <directory of the original tutorial> [--record]")
    ok, why = install(args[0], record="--record" in sys.argv)
    print("reference install:", "OK" if ok else "FAILED", why)
    sys.exit(0 if ok else 1)
