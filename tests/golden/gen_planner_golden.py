"""Golden vectors for the planner objects from the reference's OWN C++ planner.

    make -C oracle            # builds oracle/_ref/pipeline_template*.so from /root/reference/oobleck/csrc/planning
    python tests/golden/gen_planner_golden.py
    python tests/golden/gen_planner_golden.py --more

Imports the reference's pybind11 module (see oracle/Makefile for how it is built here) and records, for a set of seeded
random layer profiles, what ``PipelineTemplateGenerator.create_pipeline_templates`` returns (stage splits, GPUs per
stage, iteration time) and ``PipelineTemplate.get_rank_grid`` of every template -> tests/golden/planner.json.
``--more`` records the further comparisons of tests/test_planner_vs_reference.py -> tests/golden/planner_more.json: rank
grids of hand-built templates, templates for 24 more random profiles, stage objects built the reference's way, and what
the reference's ``get_profile_results`` reads back from a profile ``save_profile_results`` wrote.
The .so cannot travel to a machine without the reference's sources; the JSON can."""
import io
import json
import os
import random
import sys
from contextlib import redirect_stdout

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))

CASES = [  # (seed, layers, gpus per node, (min nodes, max nodes), scale of the in-node all-reduce times)
    (0, 6, 1, (1, 4), 1), (1, 8, 1, (1, 6), 1), (2, 10, 1, (2, 5), 1), (3, 5, 2, (1, 3), 1), (4, 8, 2, (1, 4), 1),
    (5, 7, 4, (1, 2), 1), (6, 9, 4, (1, 3), 1), (7, 12, 1, (1, 8), 1), (8, 4, 1, (1, 4), 1), (9, 6, 4, (1, 1), 1),
    (10, 9, 2, (2, 4), 1), (11, 14, 1, (3, 7), 1),
    # expensive in-node all-reduce: sharding a stage over a node's GPUs loses against giving the GPUs to more stages
    (12, 6, 2, (1, 2), 40), (13, 8, 4, (1, 2), 40), (14, 7, 4, (1, 1), 15), (15, 9, 2, (1, 3), 25), (16, 10, 4, (2, 2), 8),
]


def profile_rows(seed, layers, gpn, ar_scale=1):
    """Plain-python description of a random profile (also what the product-side test feeds its own classes)."""
    rnd = random.Random(seed)
    rows = []
    for i in range(layers):
        rows.append({"forward": rnd.uniform(0.2, 3.0), "backward": rnd.uniform(0.4, 6.0),
                     "allreduce_in_node": {str(g): ar_scale * rnd.uniform(0.01, 0.3) for g in range(1, gpn + 1)},
                     "allreduce_across_nodes": {str(n + 1): rnd.uniform(0.05, 0.5) for n in range(8)},
                     "mem_required": [rnd.randrange(1, 1 << 20), rnd.randrange(1, 1 << 20)]})
    return rows


def hand_built_templates(seed=5, count=60):
    """Random templates built stage by stage: every node's GPUs dealt out in power-of-two pieces, random layer cuts."""
    rnd = random.Random(seed)
    cases = []
    for _ in range(count):
        gpn = rnd.choice([1, 2, 4, 8])
        nodes = rnd.randint(1, 4)
        gpus = []
        for _n in range(nodes):
            left = gpn
            while left:
                g = rnd.choice([x for x in (1, 2, 4, 8) if x <= left])
                gpus.append(g)
                left -= g
        layers = len(gpus) + rnd.randint(0, 6)
        cuts = sorted(rnd.sample(range(1, layers), len(gpus) - 1)) if len(gpus) > 1 else []
        bounds = list(zip([0] + cuts, cuts + [layers]))
        ranks = rnd.sample(range(1000), sum(gpus))
        cases.append({"gpus_per_node": gpn, "nodes": nodes, "layers": layers, "bounds": bounds, "gpus": gpus,
                      "ranks": ranks})
    return cases


def uniform_rows(layers):
    return [{"forward": 1.0, "backward": 2.0, "allreduce_in_node": {str(g): 0.1 for g in range(1, 9)},
             "allreduce_across_nodes": {"1": 0.1}, "mem_required": [8, 8]} for _ in range(layers)]


def random_profile_case(seed):
    """(gpus per node, (min nodes, max nodes), profile rows) of one seeded random planner input."""
    rnd = random.Random(seed)
    gpn = rnd.choice([1, 1, 2, 4])
    layers = rnd.randint(3, 11)
    lo = rnd.randint(1, 3)
    hi = rnd.randint(lo, min(layers, lo + 4))
    return gpn, (lo, hi), profile_rows(seed, layers, gpn, rnd.choice([1, 1, 10, 40]))


RANDOM_PROFILE_SEEDS = range(100, 124)
STAGE_OBJECT_BOUNDS = [(0, 9, 1), (2, 5, 2), (4, 9, 4), (0, 1, 1)]     # (begin, end, GPUs) over profile_rows(3, 9, 4)
SAVED_PROFILE = (21, 7, 4, "gpt2", "b200_saved_profile_test", 3)      # profile_rows(seed, layers, gpn), name, tag, mb


def results_from_rows(mod, rows):
    return mod.LayerExecutionResults([
        mod.LayerExecutionResult(i, r["forward"], r["backward"], {int(k): v for k, v in r["allreduce_in_node"].items()},
                                 {int(k): v for k, v in r["allreduce_across_nodes"].items()}, tuple(r["mem_required"]))
        for i, r in enumerate(rows)])


def template_shape(t):
    return [t._num_nodes, [[list(s._layer_indices), s._num_gpus] for s in t.get_stages()]]


def more():
    import pipeline_template as R      # the reference's module
    sys.path.insert(0, ROOT)
    from oobleck_b200.planning import pipeline_template as P
    from oobleck_b200.planning.profiler import save_profile_results
    out = {"rank_grids": [], "random_profiles": [], "stage_objects": []}
    for c in hand_built_templates():
        prof = results_from_rows(R, uniform_rows(c["layers"]))
        t = R.PipelineTemplate([R.StageExecutionResult(prof, tuple(b), g) for b, g in zip(c["bounds"], c["gpus"])], 1.0,
                               c["layers"], c["nodes"], c["gpus_per_node"])
        out["rank_grids"].append({str(k): v for k, v in t.get_rank_grid(c["ranks"]).items()})
    for seed in RANDOM_PROFILE_SEEDS:
        gpn, node_range, rows = random_profile_case(seed)
        with redirect_stdout(io.StringIO()):
            templates = R.PipelineTemplateGenerator().create_pipeline_templates(results_from_rows(R, rows), node_range, gpn)
        out["random_profiles"].append({"seed": seed, "shapes": [template_shape(t) for t in templates],
                                       "iteration_times": [t._iteration_time for t in templates]})
    rows = profile_rows(3, 9, 4)
    for begin, end, gpus in STAGE_OBJECT_BOUNDS:
        s = R.StageExecutionResult(results_from_rows(R, rows), (begin, end), gpus)
        out["stage_objects"].append({"layer_indices": list(s._layer_indices), "num_gpus": s._num_gpus,
                                     "num_layers": s._num_layers, "forward": s._forward, "backward": s._backward,
                                     "mem_required": s._mem_required})
    out["stage_objects_profile_size"] = results_from_rows(R, rows).size
    seed, layers, gpn, name, tag, mb = SAVED_PROFILE
    # get_profile_results reads the fixed cache directory of the reference's profiler: the files go there
    directory = save_profile_results(results_from_rows(P, profile_rows(seed, layers, gpn)), name, tag, mb)
    back = R.get_profile_results(name, tag, mb)
    out["saved_profile"] = {
        "files": {f: json.load(open(os.path.join(directory, f))) for f in sorted(os.listdir(directory))},
        "read_back": [{"index": l._index, "forward": l._forward, "backward": l._backward,
                       "allreduce_in_node": {str(k): v for k, v in dict(l._allreduce_in_node).items()},
                       "allreduce_across_nodes": {str(k): v for k, v in dict(l._allreduce_across_nodes).items()},
                       "mem_required": list(l._mem_required)} for l in back.get()]}
    path = os.path.join(ROOT, "tests", "golden", "planner_more.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print(f"wrote {path}", file=sys.stderr)


def main():
    import pipeline_template as R      # the reference's module
    out = []
    for seed, layers, gpn, node_range, ar_scale in CASES:
        rows = profile_rows(seed, layers, gpn, ar_scale)
        prof = results_from_rows(R, rows)
        with redirect_stdout(io.StringIO()):      # python-level prints only; the module's std::cout chatter stays
            templates = R.PipelineTemplateGenerator().create_pipeline_templates(prof, node_range, gpn)
        case = {"seed": seed, "layers": layers, "gpus_per_node": gpn, "node_range": list(node_range), "profile": rows,
                "templates": []}
        for t in templates:
            stages = t.get_stages()
            ranks = list(range(100, 100 + sum(s._num_gpus for s in stages)))
            case["templates"].append({
                "num_nodes": t._num_nodes, "num_gpus_per_node": t._num_gpus_per_node,
                "iteration_time": t._iteration_time,
                "stages": [{"layer_indices": list(s._layer_indices), "num_gpus": s._num_gpus, "forward": s._forward,
                            "backward": s._backward, "mem_required": s._mem_required} for s in stages],
                "ranks": ranks, "rank_grid": {str(k): v for k, v in t.get_rank_grid(ranks).items()}})
        out.append(case)
    path = os.path.join(ROOT, "tests", "golden", "planner.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0)
    print(f"wrote {path}: {len(out)} cases, {sum(len(c['templates']) for c in out)} templates", file=sys.stderr)


if __name__ == "__main__":
    more() if "--more" in sys.argv else main()
