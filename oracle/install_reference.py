"""Copy the parts of the original SepReformer project that run its model (pure Python) into ``oracle/_ref/``
(git-ignored): the runnable reference for the drop-in test and the reference legs of bench.py.

    python oracle/install_reference.py

The original is read from ``SEPREFORMER_REFERENCE`` when set, else from ``/root/reference``.
``__graft_entry__.build()`` runs this whenever that checkout is present.

What is copied - unmodified - and why:
  models/<name>/{model.py, configs.yaml, modules/*.py}   the reference Model / Separator (bench.py --impl reference,
                                                         the reference-on-B200 leg, the install() drop-in tests)
  utils/decorators.py                                    imported by every reference module (needs loguru: in the image)
  utils/implements/criterions.py                         PIT_SISNRi, to pin the device-side metric
  sample_wav/sample_WSJ.wav                              BASELINE.json configs[0] input (147 KB)
Nothing here is product code and nothing under sepreformer_b200/ imports it.
"""
import os
import shutil
import sys

SRC = os.environ.get("SEPREFORMER_REFERENCE") or "/root/reference"
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def available():
    """True when SRC is a readable checkout of the original project."""
    return os.path.isdir(os.path.join(SRC, "models"))


def main():
    if not available():
        sys.exit(f"{SRC!r} is not a checkout of the original project (set SEPREFORMER_REFERENCE)")
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    n = 0
    for model in sorted(os.listdir(os.path.join(SRC, "models"))):
        mdir = os.path.join(SRC, "models", model)
        if not os.path.isdir(mdir):
            continue
        for rel in ("model.py", "configs.yaml", "modules/module.py", "modules/network.py"):
            src = os.path.join(mdir, rel)
            if os.path.exists(src):
                dst = os.path.join(DST, "models", model, rel)
                os.makedirs(os.path.dirname(dst), exist_ok=True)
                shutil.copy2(src, dst)
                n += 1
    for rel in ("utils/decorators.py", "utils/implements/criterions.py", "sample_wav/sample_WSJ.wav", "LICENSE"):
        dst = os.path.join(DST, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copy2(os.path.join(SRC, rel), dst)
        n += 1
    print(f"copied {n} files into {DST}")


if __name__ == "__main__":
    main()
