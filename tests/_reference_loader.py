"""Import the UNMODIFIED reference module from a copy of the reference's
figure_generation directory: $LSTED_REFERENCE_DIR, else the git-ignored
baseline/_ref/.  Used by the golden-vector generators in tests/golden/; the
test suite itself reads only the stored vectors.  The reference imports (but
never uses) matplotlib, which need not be installed, so a stub is injected."""
import importlib.util
import os
import sys
import types
import warnings

REFERENCE_DIR = os.environ.get('LSTED_REFERENCE_DIR') or os.path.join(
    os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'baseline', '_ref')


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_DIR, 'line_sted_tools.py'))


def load_reference():
    if 'matplotlib' not in sys.modules:
        mpl = types.ModuleType('matplotlib')
        mpl.pyplot = types.ModuleType('matplotlib.pyplot')
        sys.modules['matplotlib'] = mpl
        sys.modules['matplotlib.pyplot'] = mpl.pyplot
    if 'np_tif' not in sys.modules:
        spec = importlib.util.spec_from_file_location(
            'np_tif', os.path.join(REFERENCE_DIR, 'np_tif.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        sys.modules['np_tif'] = mod
    spec = importlib.util.spec_from_file_location(
        '_reference_line_sted_tools',
        os.path.join(REFERENCE_DIR, 'line_sted_tools.py'))
    mod = importlib.util.module_from_spec(spec)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        spec.loader.exec_module(mod)
    return mod
