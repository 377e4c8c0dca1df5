"""The product's device arithmetic (opencl_render_b200/csrc/rt_core.h -- the header every CUDA kernel instantiates -- plus the
scene packer), compiled for the host by the test suite, against the oracle.  This is the GPU-less half of the parity gate:
packed triGeo/brick layout, hoisted per-triangle terms and the restated control flow give bit-identical planes and ids."""
import json

import numpy as np
import pytest

from tests import helpers

GOLDEN = __import__("pathlib").Path(__file__).resolve().parent / "golden"


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_hostemu_equals_golden(name, hostemu):
    sc, cam, lists, samples = helpers.make_case(name)
    gold = np.load(GOLDEN / f"{name}.npz")
    img, ids, flags, cnt = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    ok = flags == 0
    res = helpers.compare_rgb(img, (gold["r"], gold["g"], gold["b"]), mask=ok)
    assert res["diff_pixels"] == 0, res                 # bit exact wherever the reference is defined
    if samples != 1:                                    # golden ids come from the S = 1 ID-material render
        ids = helpers.hostemu_render(hostemu, cam, lists, sc, 1)[1]
    assert np.array_equal(ids, gold["ids"])
    if name != "terrain_textured":
        assert flags.sum() == 0
    else:
        assert 0 < flags.sum() < 200
    assert cnt["segments"] >= cam.width * cam.height * samples


@pytest.mark.parametrize("name", ["soup_mirror_glass", "terrain_textured"])
def test_hostemu_equals_port_everywhere(name, hostemu, port):
    # the port resolves the reference's undefined case the same way as the product, so these agree on EVERY pixel
    sc, cam, lists, samples = helpers.make_case(name)
    img, ids, flags, _ = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    r, g, b, pid = port.render(cam, lists, sc, samples, want_ids=True)
    assert np.array_equal(img[0], r) and np.array_equal(img[1], g) and np.array_equal(img[2], b) and np.array_equal(ids, pid)


def test_hostemu_counters_match_reference_accounting(hostemu):
    sc, cam, lists, samples = helpers.make_case("spheres")
    _, _, _, cnt = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    rays = cam.width * cam.height * samples
    assert cnt["cellsNonEmpty"] <= cnt["cells"] and cnt["bricksLoaded"] <= cnt["cells"]
    assert cnt["gridRays"] > 0 and cnt["primCandidates"] > 0 and cnt["shadedHits"] <= cnt["segments"]
    assert cnt["segments"] >= rays


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_two_level_walk_is_exact(name, hostemu, monkeypatch):
    """The brick-granular (two-level) DDA of rt_core.h -- the trace kernel's way through empty 4x4x4 bricks -- visits the same
    bricks and returns bit-identical planes and ids, while touching far fewer cells."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    flat = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "1")
    hier = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(flat[0][c], hier[0][c])
    assert np.array_equal(flat[1], hier[1]) and np.array_equal(flat[2], hier[2])
    assert hier[3]["bricksLoaded"] == flat[3]["bricksLoaded"]          # same brick sequence
    assert hier[3]["gridCandidates"] == flat[3]["gridCandidates"] and hier[3]["cellsNonEmpty"] == flat[3]["cellsNonEmpty"]
    assert hier[3]["cells"] <= flat[3]["cells"]


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_packed_walk_is_exact(name, hostemu, monkeypatch):
    """rt_walk.h -- the walk as the production trace kernel runs it (packed coordinates, incremental brick ids, face masks and
    mailbox skipping) -- against the reference's cell walk: identical planes, ids and flags, same brick sequence, same set of
    non-empty cells; triangle tests can only go down (entries shared with the previous cell / already tested are skipped)."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    flat = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "2")
    packed = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(flat[0][c], packed[0][c])
    assert np.array_equal(flat[1], packed[1]) and np.array_equal(flat[2], packed[2])
    assert packed[3]["bricksLoaded"] <= flat[3]["bricksLoaded"]          # (super-brick steps pass bricks by without reading them)
    assert packed[3]["cellsNonEmpty"] == flat[3]["cellsNonEmpty"]
    assert packed[3]["gridCandidates"] <= flat[3]["gridCandidates"]
    assert packed[3]["cells"] <= flat[3]["cells"]


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_three_level_walk_is_exact(name, hostemu, monkeypatch):
    """The super-brick level of rt_walk.h (an entirely empty block of 4x4x4 bricks is crossed in one step, the brick-level state is
    rebuilt on entering a super-brick that holds triangles or the ray's end cell): identical planes, ids and flags, the same non-empty
    cells and the same triangle tests as the two-level walk (OCLR_SUPER=0: the packer never raises the flag the walk obeys), which
    in turn reads exactly the reference's brick sequence."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "2")
    monkeypatch.setenv("OCLR_SUPER", "0")
    two = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL")
    flat = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "2")
    monkeypatch.setenv("OCLR_SUPER", "1")
    three = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(two[0][c], three[0][c])
    assert np.array_equal(two[1], three[1]) and np.array_equal(two[2], three[2])
    assert two[3]["superSteps"] == 0 and two[3]["bricksLoaded"] == flat[3]["bricksLoaded"]
    for k in ("cells", "cellsNonEmpty", "gridCandidates", "coarseEnters", "gridRays"):
        assert three[3][k] == two[3][k], k
    assert three[3]["superEnters"] >= three[3]["superRefines"]
    if sc.axes_div >= 256:
        assert three[3]["superSteps"] > 0
        assert three[3]["coarseSteps"] < two[3]["coarseSteps"] and three[3]["bricksLoaded"] < two[3]["bricksLoaded"]
    elif sc.axes_div < 32:   # no super-brick level on a 16^3 grid
        assert three[3]["superSteps"] == 0 and three[3]["coarseSteps"] == two[3]["coarseSteps"]


@pytest.mark.parametrize("part_cells", [3, 7, 40])
@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_split_walk_is_exact(name, part_cells, hostemu, monkeypatch):
    """Exact random access into the walk (rt_walk.h pwalk_jump): every walk cut into parts of ~part_cells cells along its dominant
    axis, each part walked on its own from a state computed WITHOUT walking (binary search over the crossing values), first part
    with a hit wins -- planes, ids and flags identical to the uncut reference walk, and the parts together visit exactly the
    non-empty cells the uncut walk visits."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    flat = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", str(part_cells))
    split = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(flat[0][c], split[0][c])
    assert np.array_equal(flat[1], split[1]) and np.array_equal(flat[2], split[2])
    assert split[3]["cellsNonEmpty"] == flat[3]["cellsNonEmpty"]


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_cooperative_walk_is_exact(name, hostemu, monkeypatch):
    """rt_walk.h coop_*: the walk of one ray taken 32 plane crossings at a time, every crossing placed by the merge-order rule
    instead of by stepping (the trace kernel's tail mode) -- identical planes / ids / flags, and exactly the cells (empty and
    non-empty) the reference's cell walk visits."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    flat = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "1000")
    coop = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(flat[0][c], coop[0][c])
    assert np.array_equal(flat[1], coop[1]) and np.array_equal(flat[2], coop[2])
    assert coop[3]["cellsNonEmpty"] == flat[3]["cellsNonEmpty"]
    if name != "coarse_grid":      # rays with a zero direction component fall back to the packed (two-level) walk, which skips empty cells
        assert coop[3]["cells"] <= flat[3]["cells"]


@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_brick_plane_bursts_are_exact(name, hostemu, monkeypatch):
    """rt_walk.h grid_trace_coop_bricks, the host form of rt_tail.cuh's wf_tail_brick_kernel: the walk taken 32 BRICK-plane crossings at
    a time, the cell state rebuilt by pwalk_refine inside every brick that holds triangles or the ray's end cell -- identical planes,
    ids and flags, exactly the non-empty cells and the triangle tests of the two-level walk, and fewer brick records read than the
    reference's walk touches bricks (empty ones are looked at, never walked)."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    flat = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "2")
    packed = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", "1001")
    bricks = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(flat[0][c], bricks[0][c])
    assert np.array_equal(flat[1], bricks[1]) and np.array_equal(flat[2], bricks[2])
    assert bricks[3]["cellsNonEmpty"] == flat[3]["cellsNonEmpty"]
    assert bricks[3]["gridRays"] == packed[3]["gridRays"]
    if name != "coarse_grid":      # (rays with a zero direction component fall back to the packed walk)
        assert bricks[3]["cells"] <= flat[3]["cells"]


@pytest.mark.parametrize("name", ["spheres", "soup_mirror_glass", "terrain_textured", "soup_lights_sun_last", "coarse_grid"])
def test_counters_equal_instrumented_reference(name, hostemu, monkeypatch):
    """SURVEY.md section 8d / Appendix C: the event counts behind `roofline.achieved` (the counting build of the product's own
    arithmetic, here compiled for the host; the CUDA counting kernel is compared with the same numbers in test_gpu_parity.py)
    equal the counts of an INSTRUMENTED COPY OF THE REFERENCE KERNEL (oracle/build_ref.py puts counters at
    raytrace_opencl.c:126, 347, 365, 369, 510, 517, 532, 619), event class by event class.  The reference's counts are stored in
    golden/reference_values.json, its planes in golden/<name>.npz."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)      # the reference's own cell walk
    img, _, flags, cnt = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    gold = np.load(GOLDEN / f"{name}.npz")
    want = json.loads((GOLDEN / "reference_values.json").read_text())["counters"][name]
    ok = flags == 0
    assert helpers.compare_rgb(img, (gold["r"], gold["g"], gold["b"]), mask=ok)["diff_pixels"] == 0
    for k in ("segments", "primCandidates", "gridRays", "cells", "gridCandidates", "shadedHits", "occluderLookups"):
        assert cnt[k] == want[k], (k, cnt[k], want[k])
    assert cnt["cells"] - cnt["cellsNonEmpty"] == want["emptyCells"]


@pytest.mark.parametrize("mode", [2000 + 100 * 0 + 8, 2000 + 100 * 1 + 2, 2000 + 100 * 3 + 8, 2000 + 100 * 6 + 8, 2000 + 100 * 12 + 4, 2000 + 100 * 25 + 5])
@pytest.mark.parametrize("name", helpers.CASE_NAMES)
def test_run_time_split_is_exact(name, mode, hostemu, monkeypatch):
    """The trace kernel's run-time split (rt_walk.h pwalk_split_plan / pwalk_split_part): every walk is interrupted after
    (mode - 2000) // 100 iterations of its loop -- at whichever level it is then, cell by cell or crossing empty bricks -- and what is
    left of it is cut into up to (mode % 100) parts that start from states computed WITHOUT walking; first part with a hit wins.  Planes, ids
    and flags identical to the uncut reference walk; the parts together visit exactly the non-empty cells the uncut walk visits."""
    sc, cam, lists, samples = helpers.make_case(name)
    monkeypatch.delenv("HOSTEMU_HIERARCHICAL", raising=False)
    flat = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    monkeypatch.setenv("HOSTEMU_HIERARCHICAL", str(mode))
    split = helpers.hostemu_render(hostemu, cam, lists, sc, samples)
    for c in range(3):
        assert np.array_equal(flat[0][c], split[0][c])
    assert np.array_equal(flat[1], split[1]) and np.array_equal(flat[2], split[2])
    assert split[3]["cellsNonEmpty"] == flat[3]["cellsNonEmpty"]
