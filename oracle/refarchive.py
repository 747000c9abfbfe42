"""TEST / BENCH INFRASTRUCTURE -- never imported by the product (selfrec_b200/).

The unmodified reference is pure Python without a setup.py and its sources are not part of this repository.  Where a
checkout of it is at hand, __graft_entry__.build() packs it once into the git-ignored archive oracle/_ref/reference.zip:
the reference's .py / .yaml files plus the three datasets BASELINE.json's configs name (douban-book, yelp2018,
amazon-kindle).  Where the archive exists it is unpacked into a scratch directory by
  * tests/test_gpu_reference_files.py  (the reference's own model files running on the drop-in modules),
  * bench.py --impl reference / the cpu_baseline leg (the reference's own CPU path, kind "reference"),
all of which fall back (port / skip) when the archive is absent."""
import os
import zipfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARCHIVE = os.path.join(ROOT, "oracle", "_ref", "reference.zip")
DATASETS = ("douban-book", "yelp2018", "amazon-kindle")


def make_archive(ref="/root/reference", out=ARCHIVE):
    """Zip the reference tree (sources + the named datasets).  No-op when `ref` is absent or the archive exists."""
    if not os.path.isdir(ref):
        return None
    if os.path.exists(out):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    tmp = out + f".tmp{os.getpid()}"
    with zipfile.ZipFile(tmp, "w", zipfile.ZIP_DEFLATED, compresslevel=6) as z:
        for base, dirs, files in os.walk(ref):
            rel = os.path.relpath(base, ref)
            parts = [] if rel == "." else rel.split(os.sep)
            if parts and parts[0] == "dataset" and (len(parts) < 2 or parts[1] not in DATASETS):
                dirs[:] = [d for d in dirs if not parts[1:] and d in DATASETS]
                continue
            dirs[:] = [d for d in dirs if d not in (".git", "__pycache__")]
            for f in files:
                if f.endswith((".py", ".yaml", ".txt", ".md")):
                    z.write(os.path.join(base, f), os.path.join(rel, f) if rel != "." else f)
    os.replace(tmp, out)
    return out


def unpack(dst):
    """Extract the archive into `dst`; returns the reference root or None when there is no archive."""
    if not os.path.exists(ARCHIVE):
        return None
    with zipfile.ZipFile(ARCHIVE) as z:
        z.extractall(dst)
    return dst


def available():
    return os.path.exists(ARCHIVE)
