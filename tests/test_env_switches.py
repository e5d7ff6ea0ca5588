"""CPU: the engine is configured through irmv_engine_config alone.  The only environment variables the native code
reads are two diagnostics that do not change what it computes: IRMV_ARMOR_PROF (per-phase cycle counts of
irmv_extract_armors) and IRMV_SYNC_EACH (synchronise after every op and name the one that faulted)."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_native_code_reads_only_the_diagnostic_variables():
    names = set()
    for path in glob.glob(os.path.join(ROOT, "irmv_detection_b200", "csrc", "**", "*"), recursive=True):
        if os.path.isfile(path):
            with open(path, encoding="utf-8") as f:
                names.update(re.findall(r'getenv\(\s*"([^"]*)"', f.read()))
    assert names == {"IRMV_ARMOR_PROF", "IRMV_SYNC_EACH"}
