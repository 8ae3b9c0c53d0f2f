"""Install the UNMODIFIED reference into oracle/_ref/ (git-ignored; built next to the package so that it ships with the built tree).

    python oracle/install_reference.py [--force]

The reference is a directory of scripts, not a package (it has neither setup.py nor pyproject.toml), and nothing in it needs compiling.
"Installing" it therefore means copying its Python sources and its params/*.json byte for byte (no edits; corpora, notebooks and images
are skipped).  bench.py --impl reference, the extra baselines of bench.py and tests/test_gpu_reference_train.py import it from
oracle/_ref/; nothing under oracle/_ref/ is ever committed.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = '/root/reference'
DST = os.path.join(HERE, '_ref')
KEEP_DIRS = ('modules', 'params', 'utils', 'dataset')
KEEP_FILES = ('train.py', 'synthesize.py', 'gta.py', 'LICENSE.md', 'requirements.txt')


def installed():
    return os.path.exists(os.path.join(DST, 'modules', 'tacotron2.py'))


def install(force=False):
    if not os.path.isdir(SRC):
        return installed()
    if installed() and not force:
        return True
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    os.makedirs(DST)
    manifest = {}
    for d in KEEP_DIRS:
        for root, _, files in os.walk(os.path.join(SRC, d)):
            for f in files:
                if f.endswith(('.py', '.json')):
                    src = os.path.join(root, f)
                    rel = os.path.relpath(src, SRC)
                    os.makedirs(os.path.dirname(os.path.join(DST, rel)), exist_ok=True)
                    shutil.copyfile(src, os.path.join(DST, rel))
                    manifest[rel] = hashlib.sha256(open(src, 'rb').read()).hexdigest()
    for f in KEEP_FILES:
        if os.path.exists(os.path.join(SRC, f)):
            shutil.copyfile(os.path.join(SRC, f), os.path.join(DST, f))
            manifest[f] = hashlib.sha256(open(os.path.join(SRC, f), 'rb').read()).hexdigest()
    with open(os.path.join(DST, 'MANIFEST.json'), 'w') as fh:
        json.dump({'source': SRC, 'files': manifest}, fh, indent=1, sort_keys=True)
    return True


if __name__ == '__main__':
    ok = install(force='--force' in sys.argv)
    print('oracle/_ref installed' if ok else 'reference sources not available here and oracle/_ref is absent')
