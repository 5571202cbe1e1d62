"""The library reads only the environment variables it documents or its tests drive: every other code path is chosen
from the shapes and dtypes of a call, so no variable can switch a user onto an untested kernel."""
import glob
import os
import re

ROOT = os.path.join(os.path.dirname(__file__), "..", "image-super-resolution_b200")

KEPT = {
    "FFSR_TC_GELU_ERF",       # erf GELU in the tcgen05 epilogues (INTEGRATION.md)
    "FFSR_TC_EPI_OWN_FORCE",  # tests: tile-owning epilogue on small images
    "FFSR_TC_DEBUG",          # tests: conv_tc launch geometry on stderr
    "FFSR_WATTN_TC0",         # tests: CUDA-core reference window attention
    "FFSR_DRCT_QKV_PLAIN",    # tests: DRCT qkv without head padding
}
LAUNCHER = {"RANK", "WORLD_SIZE", "LOCAL_RANK"}   # set by torchrun, read by dist.py

READ = re.compile(r"(getenv\s*\(|os\.environ\b)")
NAMED = re.compile(r"""(?:getenv\s*\(\s*|os\.environ(?:\.get\(\s*|\[\s*))["'](\w+)["']""")


def test_library_reads_only_the_kept_environment_variables():
    found = set()
    sources = (glob.glob(os.path.join(ROOT, "csrc", "*.cu")) + glob.glob(os.path.join(ROOT, "csrc", "*.cuh"))
               + glob.glob(os.path.join(ROOT, "*.py")))
    assert sources
    for path in sources:
        comment = r"//[^\n]*" if path.endswith((".cu", ".cuh")) else r"#[^\n]*"
        code = re.sub(comment, "", open(path).read())
        names = NAMED.findall(code)
        assert len(names) == len(READ.findall(code)), f"{os.path.basename(path)}: environment read without a literal name"
        found.update(names)
    assert found - LAUNCHER == KEPT
