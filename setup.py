"""Build glue: `pip install -e .` / `python setup.py build_ext --inplace` compile the sm_100a
library in-tree with nvcc (same command as `python structuredetector_b200/build.py`)."""
from setuptools import setup
from setuptools.command.build_py import build_py


class BuildWithCuda(build_py):
    def run(self):
        import importlib.util
        from pathlib import Path

        spec = importlib.util.spec_from_file_location("sdnet_build", Path(__file__).parent / "structuredetector_b200" / "build.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build(force=False)
        # the public C header travels with the package data, so an installed copy can rebuild its libraries
        root = Path(__file__).parent
        (root / "structuredetector_b200" / "csrc" / "sdnet_decode.h").write_bytes((root / "include" / "sdnet_decode.h").read_bytes())
        super().run()


setup(cmdclass={"build_py": BuildWithCuda})
