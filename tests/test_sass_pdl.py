"""CPU: the kernels of the pruned Chamfer chain (sort -> pruned scan -> fall-back scan -> epilogue) are built for programmatic
dependent launch -- every kernel launched as a dependent waits for its predecessor (griddepcontrol.wait: ACQBULK) and every kernel
with a dependent behind it lets it be dispatched early (griddepcontrol.launch_dependents: PREEXIT).  Reads `cuobjdump -sass` of
genpc_b200/libgenpc_b200.so -- no GPU needed."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "genpc_b200", "libgenpc_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


@pytest.fixture(scope="module")
def sass():
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not available")
    if not os.path.exists(LIB):
        from genpc_b200.csrc import build

        build.build()
    out = subprocess.run([CUOBJDUMP, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None:
            funcs[name].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


def _all(sass, fragment):
    hits = {k: v for k, v in sass.items() if fragment in k}
    assert hits, f"no kernel matching {fragment}"
    return hits


@pytest.mark.parametrize("fragment", ["nn_prune_kernelILi", "nn_sym_balanced_kernelILi", "nn_sym_kernelILi",
                                      "nn_sym_epilogue_kernelILb"])
def test_dependent_kernels_wait_for_their_predecessor(sass, fragment):
    for name, body in _all(sass, fragment).items():
        assert re.search(r"\bACQBULK\b", body), f"{name}: no griddepcontrol.wait"


@pytest.mark.parametrize("fragment", ["nn_bin_sort_kernelILi", "nn_prune_kernelILi", "nn_sym_balanced_kernelILi",
                                      "nn_sym_kernelILi", "nn_sym_gated_kernelILi"])
def test_predecessors_release_their_dependents_early(sass, fragment):
    for name, body in _all(sass, fragment).items():
        assert re.search(r"\bPREEXIT\b", body), f"{name}: no griddepcontrol.launch_dependents"
