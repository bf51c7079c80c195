"""CPU: the build-time hunks for the relinked meshclust2 (integration/patch_cluster_factory.py, integration/patch_crunner.py)
apply to the reference sources where they lie, add only the offers to the batched entry points, and leave every reference line
in place (the original loops stay as the declined path).  The hunk tests skip where the reference sources are absent;
the check that a patch refuses an unexpected source needs none."""
import difflib
import os
import subprocess
import sys

import pytest

from conftest import ROOT

REF = os.environ.get("MC2_REFERENCE_ROOT", "/root/reference")
needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "src", "cluster")), reason="reference sources not present")


def _patched(script, rel, tmp_path):
    src = os.path.join(REF, "src", "cluster", rel)
    dst = str(tmp_path / rel)
    subprocess.run([sys.executable, os.path.join(ROOT, "integration", script), src, dst], check=True)
    a, b = open(src).read().splitlines(), open(dst).read().splitlines()
    added = [l[2:] for l in difflib.ndiff(a, b) if l.startswith("+ ")]
    removed = [l[2:] for l in difflib.ndiff(a, b) if l.startswith("- ")]
    return added, removed


@needs_reference
def test_cluster_factory_hunks(tmp_path):
    added, removed = _patched("patch_cluster_factory.py", "ClusterFactory.cpp", tmp_path)
    text = "\n".join(added)
    assert '#include "update_batch_b200.h"' in text
    assert text.count("mc2_batched_update(part, trn, delta)") == 1 and text.count("mc2_batched_update(part, trn, 0)") == 1
    assert text.count("mc2_batched_merge(part, trn, delta)") == 1
    # the only reference line that moves is the merge() call, which reappears inside the declined branch
    assert [l.strip() for l in removed] == ["merge(part, trn, delta, bandwidth);"]
    assert any(l.strip() == "merge(part, trn, delta, bandwidth);" for l in added)


@needs_reference
def test_crunner_hunks(tmp_path):
    added, removed = _patched("patch_crunner.py", "CRunner.cpp", tmp_path)
    text = "\n".join(added)
    assert '#include "get_points_b200.h"' in text
    for call in ("mc2_batched_effective_length(all_files.at(i), is_single_file", "mc2_batched_largest_count(f, is_single_file, k",
                 "mc2_batched_read_points<T>(files.at(i), is_single_file, _id, k, points)",
                 "mc2_batched_get_points<T>(*chromList, _id, k, points)"):
        assert text.count(call) == 1, call
    assert removed == []


def test_patch_fails_loudly_on_unexpected_source(tmp_path):
    bogus = tmp_path / "x.cpp"
    bogus.write_text("int main() { return 0; }\n")
    for script in ("patch_cluster_factory.py", "patch_crunner.py"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "integration", script), str(bogus), str(tmp_path / "y.cpp")],
                           capture_output=True, text=True)
        assert r.returncode != 0 and "expected exactly one" in (r.stderr + r.stdout)
