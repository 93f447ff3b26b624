"""Installs the UNMODIFIED reference modules into git-ignored baseline/_ref/ for `bench.py --impl reference` (the
reference's own Fingerprint.quantize under multiprocessing.Pool; without the copy an oracle port stands in):

    python scripts/install_reference.py <reference checkout>      (or DCTD_REFERENCE=<reference checkout>)

The reference has no installable package (its pyproject.toml lists build requirements only), so the "install" is a
verbatim copy of <checkout>/src/*.py plus a manifest of their sha256 digests.  Nothing under dctdomain_b200/ or tests/
imports it."""
import hashlib
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, 'baseline', '_ref')


def main():
    ref = sys.argv[1] if len(sys.argv) > 1 else os.environ.get('DCTD_REFERENCE')
    if not ref:
        print(__doc__)
        return 2
    src = os.path.join(ref, 'src')
    if not os.path.isdir(src):
        print(f'{src} not present: baseline/_ref left as it is')
        return 1
    os.makedirs(DST, exist_ok=True)
    manifest = {}
    for name in sorted(os.listdir(src)):
        if not name.endswith('.py'):
            continue
        shutil.copyfile(os.path.join(src, name), os.path.join(DST, name))
        manifest[name] = hashlib.sha256(open(os.path.join(DST, name), 'rb').read()).hexdigest()
    json.dump({'source': src, 'files': manifest}, open(os.path.join(DST, 'MANIFEST.json'), 'w'), indent=1)
    print(f'installed {len(manifest)} reference modules into {DST}')
    return 0


if __name__ == '__main__':
    sys.exit(main())
