import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "c-ray_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")
GOLDEN_SCENES = ["g_nodes", "g_legacy", "g_single", "g_meshmat"]
# + the fixture whose node graphs no JSON can express (SURVEY 8 f4: built by the reference's C constructors in oracle/ref_harness.c):
# only its flat export exists, so the loader tests skip it
GOLDEN_FLAT = GOLDEN_SCENES + ["g_f4"]
SUMMARY_LINES = []   # headline parity figures (tests/test_zz_full_config.py): repeated in the terminal summary so the run's tail shows them


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_terminal_summary(terminalreporter):
    for line in SUMMARY_LINES:
        terminalreporter.write_line(line)


@pytest.fixture(scope="session", autouse=True)
def _built():
    """Make sure the shared libraries exist (cheap no-op when they are already built)."""
    import __graft_entry__ as g
    g.build(quiet=True)


@pytest.fixture(scope="session")
def bundled_scene(tmp_path_factory):
    """bundled_scene(name) -> path of the flat scene of the reference's bundled input/<name>.json (copied to oracle/_ref/input by
    build()), made by this repository's loader (tests/test_loader.py holds it to the reference's own export), or None when
    oracle/_ref/input is missing."""
    import ctypes as C
    import crgpu
    import crscene
    made = {}
    refdir = os.path.join(ROOT, "oracle", "_ref")

    def get(name):
        if name not in made:
            made[name] = None
            if os.path.exists(os.path.join(refdir, "input", name + ".json")):
                cwd = os.getcwd()
                os.chdir(refdir)              # node-graph texture paths are relative to the reference's working directory
                try:
                    flat = crscene.load_json(os.path.join("input", name + ".json"))
                finally:
                    os.chdir(cwd)
                path = str(tmp_path_factory.mktemp("bundled") / (name + ".crscene"))
                L = crgpu.lib()
                L.crscene_save.argtypes = [C.POINTER(crgpu.FlatScene), C.c_char_p]
                assert L.crscene_save(C.byref(flat), path.encode()) == 0
                crscene.free(flat)
                made[name] = path
        return made[name]
    return get


NO_BUNDLED = "oracle/_ref/input (the reference's bundled scenes, copied by build()) is missing"
