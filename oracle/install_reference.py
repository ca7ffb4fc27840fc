"""Install the reference's training-step modules into oracle/_ref for the comparison legs of bench.py.

The reference (Onr/Council-GAN, MIT licence) is a script tree without setup.py / pyproject.toml, so ``pip install --target
oracle/_ref <tree>`` has nothing to install; this does what that command would have done for the four modules the training
step imports.  The tree is taken from ``$COUNCIL_REF_DIR`` (a checkout of Onr/Council-GAN), else from DEFAULT_SRC, where the
build environment keeps that checkout; where neither exists nothing is installed and bench.py's comparison legs run the
oracle port instead.  Only the build reads the checkout; bench.py reads the install.  ``oracle/_ref/`` is listed in
.gitignore: the reference's sources never enter this repository's history, but the install stays in the tree, so a copy of
the built tree carries it to a machine that has no reference checkout.  ``__graft_entry__.build()`` calls it.
"""
from __future__ import annotations

import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
FILES = ('trainer_council.py', 'networks.py', 'utils.py', 'data.py', 'LICENSE')
DEFAULT_SRC = '/root/reference'


def install(src=None, dst=None, quiet=False):
    src = src or os.environ.get('COUNCIL_REF_DIR') or DEFAULT_SRC
    dst = dst or os.path.join(HERE, '_ref')
    if not os.path.exists(os.path.join(src, 'trainer_council.py')):
        if not quiet:
            print('no reference tree at %s: nothing installed (bench.py will use the oracle port)' % src)
        return None
    os.makedirs(dst, exist_ok=True)
    for f in FILES:
        shutil.copyfile(os.path.join(src, f), os.path.join(dst, f))
    with open(os.path.join(dst, 'INSTALLED_FROM'), 'w') as fh:
        fh.write('%s (unmodified copies of %s; install only, git-ignored)\n' % (src, ', '.join(FILES)))
    if not quiet:
        print('installed the reference training-step modules into', dst)
    return dst


if __name__ == '__main__':
    install(*(sys.argv[1:3]))
