"""Vendor the UNMODIFIED reference (pix2pix3D) into baseline/_ref/ so that it travels to the GPU box with `gpurun`.

The reference is a script tree without setup.py / pyproject.toml, so `pip install --target baseline/_ref /root/reference`
has nothing to install (DESIGN.md section 2); the equivalent for a script tree is a verbatim copy of its importable
modules. `baseline/_ref/` is git-ignored (never part of this repository's history) but not gpurun-ignored. The copy is
byte-identical: `bench.py --impl reference` / `--impl reference-cuda` and oracle/make_golden_vs_reference.py import it from
there under its own module names (`training`, `torch_utils`, `dnnlib`), never mixed into the product path.

    python baseline/vendor_reference.py            # no-op when /root/reference is absent (GPU box: uses the shipped copy)
"""
import filecmp
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get('P3D_REFERENCE_ROOT', '/root/reference')
DST = os.path.join(HERE, '_ref')
# importable code + the three CUDA plugins' sources (JIT-built on the box by the reference's own custom_ops.get_plugin)
TREES = ('training', 'torch_utils', 'dnnlib', 'metrics')
FILES = ('camera_utils.py', 'legacy.py', 'train.py', 'LICENSE', 'applications/generate_samples.py',
         'applications/generate_video.py', 'applications/extract_mesh.py')
SUFFIXES = ('.py', '.cu', '.cpp', '.h', '.txt')


def vendor(verbose=False):
    if not os.path.isdir(os.path.join(SRC, 'training')):
        return os.path.isdir(os.path.join(DST, 'training'))
    n = 0
    for tree in TREES:
        for root, dirs, files in os.walk(os.path.join(SRC, tree)):
            dirs[:] = [d for d in dirs if d != '__pycache__']
            for f in files:
                if f.endswith(SUFFIXES):
                    rel = os.path.relpath(os.path.join(root, f), SRC)
                    n += _copy(rel)
    for rel in FILES:
        if os.path.exists(os.path.join(SRC, rel)):
            n += _copy(rel)
    if verbose:
        print(f'vendored reference -> {DST} ({n} files updated)')
    return True


def _copy(rel):
    s, d = os.path.join(SRC, rel), os.path.join(DST, rel)
    if os.path.exists(d) and filecmp.cmp(s, d, shallow=False):
        return 0
    os.makedirs(os.path.dirname(d), exist_ok=True)
    shutil.copyfile(s, d)
    return 1


def available():
    return os.path.isdir(os.path.join(DST, 'training'))


if __name__ == '__main__':
    ok = vendor(verbose=True)
    sys.exit(0 if ok else 1)
