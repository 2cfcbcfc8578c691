"""Stage the original project's hot-path sources -- TEST / BASELINE INFRASTRUCTURE.

The files oracle/reference_lift.py imports (`render` out of run.py by AST, the original
Generator, its synthesis network, nerf_utils, ops, pose_utils) are copied UNMODIFIED from a
checkout of the original project into `oracle/_ref/`, which git ignores: they are never part of
this repository's history, but a copy of the working tree taken after `build()` carries them to a
machine that has no such checkout.  The original project has no setup.py / pyproject.toml, so a
file-level copy of its Apache-2.0 sources is what installing it means here.

Used by `__graft_entry__.build()`, from `source()`: `NFI_REFERENCE_ROOT` when set, else
DEFAULT_SOURCE, where the build machine keeps the original checkout; read by
`oracle/reference_lift.py`.
"""
import hashlib
import json
import os
import shutil
import sys

FILES = ('run.py', 'LICENSE', 'lib/nerf_utils.py', 'lib/ops.py', 'lib/pose_utils.py',
         'models/generator.py', 'models/stylegan.py')

DEST = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')
DEFAULT_SOURCE = '/root/reference'


def source():
    """The original checkout to stage from, or None when there is none."""
    src = os.environ.get('NFI_REFERENCE_ROOT') or DEFAULT_SOURCE
    return src if os.path.isfile(os.path.join(src, 'run.py')) else None


def stage(src, dest=DEST, quiet=False):
    """Copies FILES from ``src`` to ``dest``; returns the manifest (path -> sha256)."""
    if not os.path.isfile(os.path.join(src, 'run.py')):
        raise FileNotFoundError('no checkout of the original project at %s' % src)
    manifest = {}
    for rel in FILES:
        s, d = os.path.join(src, rel), os.path.join(dest, rel)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
        with open(d, 'rb') as f:
            manifest[rel] = hashlib.sha256(f.read()).hexdigest()
    with open(os.path.join(dest, 'MANIFEST.json'), 'w') as f:
        json.dump({'files': manifest}, f, indent=1, sort_keys=True)
    if not quiet:
        print('staged %d files of the original project into %s' % (len(manifest), dest))
    return manifest


if __name__ == '__main__':
    stage(sys.argv[1] if len(sys.argv) > 1 else source() or DEFAULT_SOURCE)
