"""Static evidence, from the SASS of the in-tree ``libbezk.so`` (cuobjdump, no GPU needed), that the hot kernels are what
DESIGN.md says: sm_100a code, TMA bulk copies (``UBLKCP``) + mbarrier waits (``SYNCS``) in the tile / learner / rollout kernels,
64-byte-granule gathers (``LDG...LTC64B``) and programmatic-dependent-launch markers in the task kernel, and no division /
square-root slow-path CALL on the main path beyond the documented fallbacks.  Skips when cuobjdump or the library is missing."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "bez_isaacgym_b200", "libbezk.so")


@pytest.fixture(scope="module")
def sass():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(LIB) or not (shutil.which("cuobjdump") or os.path.exists(exe)):
        pytest.skip("needs cuobjdump and a built libbezk.so")
    text = subprocess.check_output([exe, "-sass", LIB], text=True)
    assert "sm_100a" in text or "sm_100" in text
    funcs = {}
    name = None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None:
            funcs[name].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


def _find(sass, fragment):
    hits = [k for k in sass if fragment in k]
    assert hits, f"no kernel matching {fragment}"
    return hits


def test_library_targets_sm_100a_only():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(LIB) or not os.path.exists(exe):
        pytest.skip("needs cuobjdump and a built libbezk.so")
    out = subprocess.check_output([exe, "-lelf", LIB], text=True)
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_tile_kernels_use_tma_bulk_copies_and_64B_gathers(sass):
    for task in ("Li0E", "Li1E", "Li2E"):                      # kick, walk, orient: the fused step
        for name in _find(sass, f"task_tile_kernelILi7ELb0ELi128E{task}"):
            body = sass[name]
            assert body.count("UBLKCP.S.G") >= 2, "two bulk loads (dof_state, root_states) per warp"
            assert "UBLKCP.G.S" in body, "bulk store of the observation rows"
            assert "SYNCS" in body and "LTC64B" in body, "mbarrier wait and 64-byte-granule gathers"
            assert "ACQBULK" in body or "PREEXIT" in body, "programmatic dependent launch markers"
            assert "BAR.SYNC" not in body, "the kernel has no CTA-wide barrier"


def test_learner_and_rollout_kernels_use_tma(sass):
    for frag in ("rms_partials_tma_kernelILb0", "rms_partials_tma_kernelILb1", "ppo_loss_kernel", "policy_head_kernel"):
        for name in _find(sass, frag):
            assert "UBLKCP.S.G" in sass[name] and "SYNCS" in sass[name], name
    for name in _find(sass, "ppo_loss_kernel") + _find(sass, "policy_head_kernel"):
        assert "UBLKCP.G.S" in sass[name], "gradient / action tiles leave by bulk store"


def test_no_local_memory_in_the_streaming_kernels(sass):
    """No spills / local arrays in the streaming kernels (``dr_noise_kernel`` included since round 2: its ragged tail is fully
    unrolled, predicated scalar code).  Known exception, not listed: K0's scalar fallback indexes the constant block dynamically."""
    for frag in ("gae_kernelIhLi8", "gae_kernelIfLi8", "rms_normalize_kernelILb0", "rms_partials_tma_kernelILb0", "swap_flatten_kernelIm",
                 "adv_normalize_kernel", "flat_partials_kernel", "dr_noise_kernel"):
        for name in _find(sass, frag):
            assert "STL" not in sass[name] and "LDL" not in sass[name], name


def test_fused_kernel_divides_without_a_branch_per_operation(sass):
    """``Mth<true>``: the main path keeps NVIDIA's fast sequences but not their per-operation FCHK + slow-path branch; what
    remains are the three ``atan2f`` calls' internal divides and the once-per-env precise fallbacks."""
    body = sass[_find(sass, "task_tile_kernelILi7ELb0ELi128ELi0E")[0]]
    assert body.count("MUFU.RCP") >= 10 and body.count("MUFU.RSQ") >= 6
    assert body.count("FCHK") <= 24            # 3 inside atan2f + the fallback copies; the first version had 16 on the MAIN path


def test_fused_kernel_fits_five_ctas_worth_of_registers(sass):
    """Round 2: the dof half of the observation row is written before the long dependent chains, so the fused BezKick step needs
    ~101 registers instead of 126 (cuobjdump -res-usage)."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.check_output([exe, "-res-usage", LIB], text=True)
    m = re.search(r"Function _ZN4bezk16task_tile_kernelILi7ELb0ELi128ELi0EE[^\n]*\n\s*REG:(\d+)", out)
    assert m, "resource usage of the fused kernel not found"
    assert int(m.group(1)) <= 104, m.group(1)


def test_cooperative_statistics_kernel_has_a_grid_barrier(sass):
    body = sass[_find(sass, "fused_stats_kernelILi1E")[0]]
    assert "STL" not in body and "LDL" not in body
