"""The FETAL_B200_* environment switches the library and the Python package read are exactly the ones README.md
documents: a switch cannot be added without being announced, and the README names none that is gone."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "fetal-mri-segmentation_b200")
SOURCES = (".cu", ".cuh", ".h", ".cpp", ".py")


def switches_read():
    # a switch is read through its name as a string literal: getenv in the CUDA host code, os.environ in Python
    names = set()
    for sub in ("csrc", "fetal_net"):
        for dirpath, _, files in os.walk(os.path.join(PKG, sub)):
            for f in files:
                if f.endswith(SOURCES):
                    with open(os.path.join(dirpath, f), encoding="utf-8") as fh:
                        names.update(re.findall(r"""["'](FETAL_B200_[A-Z0-9_]+)["']""", fh.read()))
    return names


def test_environment_switches_match_readme():
    with open(os.path.join(ROOT, "README.md"), encoding="utf-8") as fh:
        documented = set(re.findall(r"FETAL_B200_[A-Z0-9_]+", fh.read()))
    read = switches_read()
    assert "FETAL_B200_DETERMINISTIC" in read, "the source scan found nothing"
    assert read == documented, "read but not in README.md: %s; in README.md but read nowhere: %s" % (
        sorted(read - documented), sorted(documented - read))
