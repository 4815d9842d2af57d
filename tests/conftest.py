import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "team02-objectdetection_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_sessionstart(session):
    """Tests never run against a stale or missing library: build (no-op when up to date) before collection, because the
    test modules import b200seg, which loads the library."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("b200seg_build", os.path.join(ROOT, "team02-objectdetection_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
