"""Import the UNMODIFIED reference (TEST / BASELINE INFRASTRUCTURE, never on the product path).

Two places hold it:
  * a read-only checkout of AntoinePassemiers/Oriana at CHECKOUT below ($ORIANA_REFERENCE_CHECKOUT overrides its
    default); `oracle/make_golden.py` records the fixtures under `tests/golden/` from it;
  * `oracle/_ref/` -- the reference INSTALLED from that checkout by `install()` below
    (`pip install --no-index --no-build-isolation --no-deps --target oracle/_ref <copy of the checkout>`; run by
    `__graft_entry__.build()` whenever the checkout is visible).  The directory is git-ignored (not product source); a
    copy of the tree that carries it lets `bench.py --impl reference` and `bench.py`'s `cpu_baseline` leg run the
    reference's own `ZIGaP.step()` on a machine without the checkout.  The test suite does not need either: it compares
    against the fixtures.

The reference pins numpy 1.13 and uses `np.float` / `np.int` (`oriana/parameters.py:11`), removed in numpy >= 1.24; the
two-line alias below is the only change needed (SURVEY.md section 8c) -- the installed files are byte-identical to the
checkout's.
"""
import os, shutil, subprocess, sys, tempfile
import numpy as np

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECKOUT = os.environ.get('ORIANA_REFERENCE_CHECKOUT', '/root/reference')
INSTALLED = os.path.join(_REPO, 'oracle', '_ref')


def _checkout_present():
    return bool(CHECKOUT) and os.path.isdir(os.path.join(CHECKOUT, 'oriana', 'models'))


def _root():
    env = os.environ.get('ORIANA_REFERENCE_ROOT')
    if env:
        return env
    if os.path.isdir(os.path.join(INSTALLED, 'oriana', 'models')):
        return INSTALLED                      # the install (byte-identical files) wins: same path here and on the GPU box
    if _checkout_present():
        return CHECKOUT
    return INSTALLED


REFERENCE_ROOT = _root()


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, 'oriana'))


def install(force=False):
    """Install the reference from the read-only checkout into oracle/_ref (no-op when the checkout is absent or when the
    install is already there).  pip builds a wheel in the source tree, hence the temporary copy."""
    if not _checkout_present():
        return os.path.isdir(os.path.join(INSTALLED, 'oriana'))
    if os.path.isdir(os.path.join(INSTALLED, 'oriana', 'models')) and not force:
        return True
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, 'reference')
        shutil.copytree(CHECKOUT, src)
        for d, _, files in os.walk(src):
            os.chmod(d, 0o755)
            for f in files:
                os.chmod(os.path.join(d, f), 0o644)
        shutil.rmtree(INSTALLED, ignore_errors=True)
        os.makedirs(os.path.dirname(INSTALLED), exist_ok=True)
        r = subprocess.run([sys.executable, '-m', 'pip', 'install', '--no-index', '--no-build-isolation', '--no-deps',
                            '--target', INSTALLED, src], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('pip install of the reference failed:\n' + r.stdout + r.stderr)
    return True


def import_reference():
    if not available():
        raise ImportError('reference not present at %s (neither the checkout nor oracle/_ref)' % REFERENCE_ROOT)
    np.float = float  # noqa: alias shim
    np.int = int
    sys.dont_write_bytecode = True  # the reference tree is read-only
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    # our own repo ships an `oriana` alias package: make sure the reference's wins here
    for k in [k for k in sys.modules if k == 'oriana' or k.startswith('oriana.')]:
        del sys.modules[k]
    import oriana  # noqa
    assert os.path.realpath(oriana.__file__).startswith(os.path.realpath(REFERENCE_ROOT)), oriana.__file__
    return oriana


def release_reference():
    """Undo import_reference(): drop the reference modules and its sys.path entry, so that the repo's own
    `oriana` alias package is importable again in the same process."""
    for k in [k for k in sys.modules if k == 'oriana' or k.startswith('oriana.')]:
        del sys.modules[k]
    while REFERENCE_ROOT in sys.path:
        sys.path.remove(REFERENCE_ROOT)


STATE_KEYS_ZIGAP = ('a1', 'a2', 'b1', 'b2', 'p_d', 'pi_d', 'alpha1', 'alpha2', 'beta1', 'beta2')
STATE_KEYS_GAP = ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2')
STATE_KEYS_SPARSE = STATE_KEYS_ZIGAP + ('p_s', 'pi_s')


def snapshot(model):
    """Copy the state vector (SURVEY.md 8c) out of a constructed reference model."""
    keys = STATE_KEYS_SPARSE if hasattr(model, 'p_s') else (STATE_KEYS_ZIGAP if hasattr(model, 'p_d') else STATE_KEYS_GAP)
    s = {k: np.array(getattr(model, k)[:], dtype=np.float64, copy=True) for k in keys}
    s['X'] = np.array(model.X[:], copy=True)
    return s
