"""The one offline install of the reference (bench contract): `pip install --no-index --target baseline/_ref <reference>`.

    CFPP_REFERENCE_SRC=<upstream contextflow checkout> python tools/install_reference.py

Outcome recorded in DESIGN.md: the wheel builds, but the reference's setup.py declares `packages=['contextflow']` only, so the
installed tree holds config.py / model.py / experiment_*.py WITHOUT the layers/, utils/ and datasets/ sub-packages model.py imports
-- it cannot run.  This script therefore completes the install by copying those sub-packages (python sources only, no images /
binaries) next to the installed files.  baseline/_ref/ is git-ignored (never part of this repo's history); where it exists, bench.py
times the unmodified reference on CUDA (`torch_cuda_baseline`) and tests/test_gpu_boundary.py runs its unmodified experiment loops
over this repo's layers."""
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get('CFPP_REFERENCE_SRC')
DST = os.path.join(ROOT, 'baseline', '_ref')


def main():
    if not SRC or not os.path.isdir(SRC):
        print('set CFPP_REFERENCE_SRC to an upstream contextflow checkout: nothing to install'); return 0
    with tempfile.TemporaryDirectory() as tmp:
        tmp = os.path.join(tmp, 'src')
        shutil.copytree(SRC, tmp, ignore=shutil.ignore_patterns('.git', 'images'))      # the build writes into the source tree, which may be read-only
        shutil.rmtree(DST, ignore_errors=True)
        r = subprocess.run([sys.executable, '-m', 'pip', 'install', '--no-index', '--no-build-isolation', '--no-deps', '--target', DST, tmp],
                           capture_output=True, text=True)
    print(r.stdout[-600:], r.stderr[-600:])
    pkg = os.path.join(DST, 'contextflow')
    os.makedirs(pkg, exist_ok=True)
    for top in ('config.py', 'model.py', 'experiment_ad.py', 'experiment_cl.py', '__init__.py'):
        if not os.path.exists(os.path.join(pkg, top)):
            shutil.copy2(os.path.join(SRC, 'contextflow', top), os.path.join(pkg, top))
    for sub in ('layers', 'utils', 'datasets'):
        shutil.copytree(os.path.join(SRC, 'contextflow', sub), os.path.join(pkg, sub), dirs_exist_ok=True,
                        ignore=lambda d, names: [n for n in names if os.path.isfile(os.path.join(d, n)) and not n.endswith('.py')])
    print('installed:', sorted(os.listdir(pkg)))
    return 0


if __name__ == '__main__':
    sys.exit(main())
