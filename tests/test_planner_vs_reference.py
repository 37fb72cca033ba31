"""The planner objects against the reference's OWN C++ planner (oobleck/csrc/planning/pipeline_template.{h,cpp},
execution_result.h, bound by bind.cpp).

* ``tests/golden/planner.json`` was produced by that module itself (tests/golden/gen_planner_golden.py; oracle/Makefile
  builds it from the sources under /root/reference with single-threaded stand-ins for cppcoro / oneTBB): for 17 seeded
  layer profiles -- 1, 2 and 4 GPUs per node, node ranges up to 8, cheap and expensive in-node all-reduce -- the templates
  ``PipelineTemplateGenerator.create_pipeline_templates`` returns and the rank grid of each.  This repo's template search
  (csrc/planning/template_search.cpp behind ``oob_plan_pipeline_templates``) and ``PipelineTemplate.get_rank_grid`` must
  reproduce them: same stage boundaries, same GPUs per stage, iteration time to 1e-12, rank grids equal.
* ``tests/golden/planner_more.json`` (``gen_planner_golden.py --more``, from the same module) holds further comparisons:
  rank grids of 60 hand-built templates, the templates for 24 more random profiles, stage objects built the reference's
  way, and what the reference's ``get_profile_results`` read back from a profile this package's ``save_profile_results``
  wrote.
* when oracle/_ref holds the built module, the reference's own planner tests (tests/planning/test_pipeline_template.py:
  10-100) run against both modules.
"""
import importlib
import json
import os
import random
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

from gen_planner_golden import results_from_rows  # noqa: E402
from oobleck_b200.planning import pipeline_template as P  # noqa: E402

GOLDEN = json.load(open(os.path.join(ROOT, "tests", "golden", "planner.json")))
MORE = json.load(open(os.path.join(ROOT, "tests", "golden", "planner_more.json")))


def reference_module():
    d = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(d) or not any(f.startswith("pipeline_template") and f.endswith(".so") for f in os.listdir(d)):
        return None
    sys.path.insert(0, d)
    try:
        return importlib.import_module("pipeline_template")
    except ImportError:
        return None
    finally:
        sys.path.remove(d)


@pytest.mark.parametrize("case", GOLDEN, ids=[f"seed{c['seed']}-{c['layers']}L-{c['gpus_per_node']}gpn" for c in GOLDEN])
def test_template_search_reproduces_the_reference_planner(case):
    prof = results_from_rows(P, case["profile"])
    mine = P.PipelineTemplateGenerator().create_pipeline_templates(prof, tuple(case["node_range"]), case["gpus_per_node"])
    assert len(mine) == len(case["templates"])
    for got, want in zip(mine, case["templates"]):
        assert got._num_nodes == want["num_nodes"] and got._num_gpus_per_node == want["num_gpus_per_node"]
        assert [(list(s._layer_indices), s._num_gpus) for s in got.get_stages()] == \
               [(s["layer_indices"], s["num_gpus"]) for s in want["stages"]]
        assert got._iteration_time == pytest.approx(want["iteration_time"], rel=1e-12)
        for s, ws in zip(got.get_stages(), want["stages"]):
            assert s._mem_required == ws["mem_required"]          # 6 x parameter bytes + activation bytes per layer
            assert s._forward == pytest.approx(ws["forward"], rel=1e-13)
            assert s._backward == pytest.approx(ws["backward"], rel=1e-13)
        grid = got.get_rank_grid(want["ranks"])
        assert {str(k): v for k, v in grid.items()} == want["rank_grid"]
        assert list(grid) == sorted(grid)                          # std::map order


def test_rank_grid_of_hand_built_templates_matches_the_reference_module():
    """pipeline_template.h:57-84 directly (before: pinned only through the reference's test tables)."""
    from gen_planner_golden import hand_built_templates
    cases = hand_built_templates()
    assert len(cases) == len(MORE["rank_grids"]) == 60
    for c, want in zip(cases, MORE["rank_grids"]):
        mt = P.PipelineTemplate([P.StageExecutionResult(range(a, b), g) for (a, b), g in zip(c["bounds"], c["gpus"])],
                                1.0, c["layers"], c["nodes"], c["gpus_per_node"])
        assert {str(k): v for k, v in mt.get_rank_grid(c["ranks"]).items()} == want


@pytest.mark.parametrize("seed", range(100, 124))
def test_live_comparison_on_random_profiles(seed):
    from gen_planner_golden import RANDOM_PROFILE_SEEDS, random_profile_case, template_shape
    theirs = MORE["random_profiles"][RANDOM_PROFILE_SEEDS.index(seed)]
    assert theirs["seed"] == seed
    gpn, node_range, rows = random_profile_case(seed)
    mine = P.PipelineTemplateGenerator().create_pipeline_templates(results_from_rows(P, rows), node_range, gpn)
    assert [template_shape(t) for t in mine] == theirs["shapes"]
    for a, b in zip(mine, theirs["iteration_times"]):
        assert a._iteration_time == pytest.approx(b, rel=1e-12)


# ---- the reference's own planner tests (tests/planning/test_pipeline_template.py:10-100), on both modules ---------------
def both():
    mods = [("this repo", P)]
    R = reference_module()
    if R is not None:
        mods.append(("reference", R))
    return mods


MODULES = both()
NUM_LAYERS = 10        # the reference's fixture model has 34 stage layers; its own planner needs minutes there on one thread


@pytest.fixture(params=MODULES, ids=[w for w, _ in MODULES])
def planner(request):
    """(module, profile): tests/conftest.py:119-142 get_dummy_profile -- random times, 1 KiB per layer."""
    mod = request.param[1]
    rnd = random.Random(7)
    profile = mod.LayerExecutionResults([
        mod.LayerExecutionResult(layer_index=i, forward=rnd.random() + 1e-3, backward=rnd.random() * 3 + 1e-3,
                                 allreduce_in_node={g + 1: rnd.random() for g in range(8)},
                                 allreduce_across_nodes={n + 1: rnd.random() * 4 for n in range(64)},
                                 mem_required=(1024, 1024)) for i in range(NUM_LAYERS)])
    return mod, profile


def test_create_pipeline_templates_onegpu(planner):
    mod, profile = planner
    pipeline_templates = mod.PipelineTemplateGenerator().create_pipeline_templates(profile, (1, 1), 1)
    assert len(pipeline_templates) == 1
    assert pipeline_templates[0]._num_nodes == 1
    assert pipeline_templates[0]._num_gpus_per_node == 1
    assert len(pipeline_templates[0].get_stages()) == 1
    assert pipeline_templates[0]._iteration_time > 0


def test_create_pipeline_templates_maxnode(planner):
    mod, profile = planner
    num_nodes = profile.size                     # a property in the binding (bind.cpp:38)
    pipeline_templates = mod.PipelineTemplateGenerator().create_pipeline_templates(profile, (num_nodes, num_nodes), 1)
    assert len(pipeline_templates) == 1
    assert pipeline_templates[0]._num_nodes == num_nodes
    assert pipeline_templates[0]._num_gpus_per_node == 1
    assert len(pipeline_templates[0].get_stages()) == num_nodes
    assert pipeline_templates[0]._iteration_time > 0


def test_create_pipeline_templates_too_many_nodes(planner):
    mod, profile = planner
    num_nodes = profile.size + 1
    assert len(mod.PipelineTemplateGenerator().create_pipeline_templates(profile, (num_nodes, num_nodes), 1)) == 0


def test_create_pipeline_templates_node_range(planner):
    mod, profile = planner
    max_num_nodes = profile.size
    pipeline_templates = mod.PipelineTemplateGenerator().create_pipeline_templates(profile, (2, 8), 1)
    assert 0 < len(pipeline_templates) <= max_num_nodes
    assert 0 < pipeline_templates[0]._num_nodes <= max_num_nodes
    for pipeline_template in pipeline_templates:
        assert pipeline_templates[0]._num_gpus_per_node == 1
        assert 2 <= len(pipeline_template.get_stages()) <= 8
        assert pipeline_template._iteration_time > 0


def test_create_pipeline_templates_multiple_gpus_in_node(planner):
    mod, profile = planner
    pipeline_templates = mod.PipelineTemplateGenerator().create_pipeline_templates(profile, (1, 1), 4)
    assert len(pipeline_templates) >= 1
    assert sum(t._num_gpus_per_node * t._num_nodes for t in pipeline_templates) == 4


def test_create_pipeline_templates_multiple_gpus_in_node_range(planner):
    mod, profile = planner
    pipeline_templates = mod.PipelineTemplateGenerator().create_pipeline_templates(profile, (1, 6), 4)
    assert len(pipeline_templates) >= 1
    for index, template in enumerate(pipeline_templates):
        num_nodes = index + 1
        assert template._num_gpus_per_node == 4
        assert num_nodes == template._num_nodes


def test_stage_objects_built_the_references_way_agree():
    """``StageExecutionResult(layer_results, (begin, end), num_gpus)`` (bind.cpp:40-48): same aggregates on both sides."""
    from gen_planner_golden import STAGE_OBJECT_BOUNDS, profile_rows
    rows = profile_rows(3, 9, 4)
    for (begin, end, gpus), b in zip(STAGE_OBJECT_BOUNDS, MORE["stage_objects"], strict=True):
        a = P.StageExecutionResult(results_from_rows(P, rows), (begin, end), gpus)
        assert a._layer_indices == b["layer_indices"] and a._num_gpus == b["num_gpus"]
        assert a._num_layers == b["num_layers"] == end - begin
        assert a._forward == pytest.approx(b["forward"], rel=1e-15)
        assert a._backward == pytest.approx(b["backward"], rel=1e-15)
        assert a._mem_required == b["mem_required"]
    assert results_from_rows(P, rows).size == MORE["stage_objects_profile_size"] == 9
    assert results_from_rows(P, rows).size() == 9          # the stub file's spelling (pipeline_template.pyi:21)


def test_golden_bookkeeping_vectors_reproduce_with_the_references_own_planner_objects():
    """tests/golden/{reconfigure,dp_groups,sampler,schedule,dtype_ids}.json come from the reference's own Python
    (tests/golden/gen_golden.py).  With oracle/_ref built, the C++ ``PipelineTemplate`` objects inside that run are the
    reference's own too -- and every committed file must come out byte for byte (``--check``)."""
    import subprocess
    if reference_module() is None or not os.path.isdir("/root/reference/oobleck"):
        pytest.skip("needs /root/reference and oracle/_ref (make -C oracle)")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "golden", "gen_golden.py"), "--check"],
                       capture_output=True, text=True, timeout=600)
    assert "the reference's own module" in r.stderr, r.stderr[-2000:]
    assert r.returncode == 0 and "all golden files reproduced" in r.stderr, r.stderr[-2000:]


def test_saved_profile_is_what_the_references_get_profile_results_reads(tmp_path):
    """planning/profiler.py::save_profile_results -> the reference's C++ ``get_profile_results`` (it reads
    /tmp/oobleck/profiles/<model>-<tag>/, pipeline_template.cpp:26-79): the files written must be those the reference
    read back, and what it read back must be this profile."""
    from gen_planner_golden import SAVED_PROFILE, profile_rows
    from oobleck_b200.planning.profiler import get_profile_path, save_profile_results
    seed, layers, gpn, name, tag, mb = SAVED_PROFILE
    mine = results_from_rows(P, profile_rows(seed, layers, gpn))
    assert str(get_profile_path(name, tag)) == f"/tmp/oobleck/profiles/{name}-{tag}"
    directory = save_profile_results(mine, name, tag, mb, cache=str(tmp_path))
    assert directory == tmp_path / f"{name}-{tag}"
    want = MORE["saved_profile"]
    assert {f: json.load(open(directory / f)) for f in sorted(os.listdir(directory))} == want["files"]
    back = want["read_back"]
    assert len(back) == mine.size == 7
    for a, b in zip(mine.get(), back):
        assert b["index"] == a._index
        assert b["forward"] == a._forward and b["backward"] == a._backward            # JSON round-trips doubles exactly
        assert b["allreduce_in_node"] == {str(k): v for k, v in a._allreduce_in_node.items()}
        assert b["allreduce_across_nodes"] == {str(k): v for k, v in a._allreduce_across_nodes.items()}
        assert tuple(b["mem_required"]) == a._mem_required
