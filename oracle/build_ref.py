"""Build oracle/_ref/ from a checkout of the reference.  TEST INFRASTRUCTURE ONLY.

    KGC_REFERENCE_DIR=<checkout of weilonghu/KGC-GCN> python oracle/build_ref.py      (also called by __graft_entry__.build())

The reference (weilonghu/KGC-GCN) is pure Python and is not part of this repository; its four modules are byte-compiled
from $KGC_REFERENCE_DIR into ``oracle/_ref/{model,data_loader,main,utils}.refbc`` (CPython bytecode: a BUILT artefact like
a .so - git-ignored; no reference source is copied into the repository).  With ``oracle/shims`` on the path (stand-ins
for the reference's absent third-party imports) they import unmodified, which is what ``bench.py --impl reference`` times
(cpu_baseline.kind = "reference") and what the tests that name the reference cross-check the port against.  Without
KGC_REFERENCE_DIR nothing is built: bench.py falls back to the pinned port (oracle/mgcn_oracle.py), those tests skip, and
the committed fixtures in tests/golden (written by oracle/make_golden.py from the reference) still pin the port.
"""
import os
import py_compile
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, '_ref')
MODULES = ('utils', 'model', 'data_loader', 'main')      # import order: main imports the other three
EXT = '.refbc'                 # not '.pyc': snapshot tools commonly drop *.pyc


def build_ref(ref_dir=None):
    """-> list of written files ([] when no reference checkout is given or it lacks a module)."""
    ref_dir = ref_dir or os.environ.get('KGC_REFERENCE_DIR')
    if not ref_dir or not all(os.path.exists(os.path.join(ref_dir, m + '.py')) for m in MODULES):
        return []
    os.makedirs(OUT, exist_ok=True)
    written = []
    for m in MODULES:
        dst = os.path.join(OUT, m + EXT)
        py_compile.compile(os.path.join(ref_dir, m + '.py'), cfile=dst, dfile='reference/' + m + '.py', doraise=True)
        written.append(dst)
    return written


def load_reference():
    """(model, data_loader, main) modules of the UNMODIFIED reference from oracle/_ref, or None when it was not built
    (or was built by another interpreter version).  Puts oracle/shims on sys.path and registers the four modules under
    the names the reference imports them by (utils, model, data_loader, main)."""
    import importlib.machinery
    import importlib.util
    paths = {m: os.path.join(OUT, m + EXT) for m in MODULES}
    if not all(os.path.exists(p) for p in paths.values()):
        return None
    shims = os.path.join(HERE, 'shims')
    if shims not in sys.path:
        sys.path.insert(0, shims)
    loaded = {}
    try:
        for m in MODULES:
            cur = sys.modules.get(m)
            if cur is not None and getattr(cur, '__file__', None) == paths[m]:
                loaded[m] = cur
                continue
            if cur is not None:
                return None                     # some other 'model' / 'main' / 'utils' module is already imported
            loader = importlib.machinery.SourcelessFileLoader(m, paths[m])
            spec = importlib.util.spec_from_loader(m, loader, origin=paths[m])
            mod = importlib.util.module_from_spec(spec)
            mod.__file__ = paths[m]
            sys.modules[m] = mod
            loader.exec_module(mod)
            loaded[m] = mod
    except Exception:                           # stale bytecode (other interpreter), missing third-party module, ...
        for m in MODULES:
            if m in sys.modules and getattr(sys.modules[m], '__file__', None) == paths[m]:
                del sys.modules[m]
        return None
    return loaded['model'], loaded['data_loader'], loaded['main']


if __name__ == '__main__':
    print(build_ref() or 'KGC_REFERENCE_DIR is not a reference checkout: nothing built')
