"""Product bookkeeping (oobleck_b200.execution.engine / pipeline / planning) bit-exact against golden vectors produced
by the reference's own Python and against the tables in the reference's tests.  No GPU, no process group."""
import json
import os
import types

import pytest

from oobleck_b200.execution import utils as U
from oobleck_b200.execution.dataloader import OobleckSampler
from oobleck_b200.execution.engine import DataParallelEngine, ReconfigurationEngine
from oobleck_b200.execution.pipeline import OobleckPipeline
from oobleck_b200.planning.pipeline_template import PipelineTemplate, StageExecutionResult
from oracle import bookkeeping as bk

G = os.path.join(os.path.dirname(__file__), "golden")
NUM_LAYERS = 34


def load(name):
    return json.load(open(os.path.join(G, name + ".json")))


def product_template(num_stages, gpn, nodes) -> PipelineTemplate:
    """tests/conftest.py:144-213 dummy template, expressed with the product's template classes."""
    o = bk.dummy_template(NUM_LAYERS, num_stages, gpn, nodes)
    stages = [StageExecutionResult(s._layer_indices, s._num_gpus) for s in o.get_stages()]
    return PipelineTemplate(stages, 0.1, NUM_LAYERS, nodes, gpn)


class FakeEngine:
    def __init__(self, gpn, templates):
        self._num_gpus_per_node = gpn
        self._pipeline_templates = templates
        self._agent_pipe = None


def fake_pipelines(gpn, templates):
    pipes, used = [], 0
    for pid, t in enumerate(templates):
        n = t._num_nodes * gpn
        pipes.append(OobleckPipeline(pid, t, list(range(used, used + n)), None, 0, None,
                                     layer_cls=types.SimpleNamespace(device_type="cpu")))
        used += n
    return pipes


def test_rank_grid_matches_oracle():
    for gpn, stages, nodes in [(1, 4, 4), (4, 2, 1), (4, 4, 3), (2, 5, 4), (4, 5, 5)]:
        t, o = product_template(stages, gpn, nodes), bk.dummy_template(NUM_LAYERS, stages, gpn, nodes)
        ranks = list(range(3, 3 + nodes * gpn))
        assert t.get_rank_grid(ranks) == o.get_rank_grid(ranks)


def test_reconfiguration_policy_golden():
    cases = load("reconfigure")
    for c in cases:
        gpn = c["gpus_per_node"]
        templates = [product_template(i, gpn, i) for i in range(2, 6)]
        eng = FakeEngine(gpn, templates)
        eng._pipeline = None
        re = ReconfigurationEngine(eng, fake_pipelines(gpn, templates), start_listener=False)
        got = re.plan_new_ranks(list(c["failed"]))
        assert got == c["result"]["ranks"], c


def test_reconfiguration_insufficient_ranks():
    templates = [product_template(2, 1, 2)]
    eng = FakeEngine(1, templates)
    re = ReconfigurationEngine(eng, fake_pipelines(1, templates), start_listener=False)
    with pytest.raises(RuntimeError, match="insufficient"):
        re.plan_new_ranks([1])


def test_dp_groups_golden():
    for c in load("dp_groups"):
        gpn = c["gpus_per_node"]
        templates = []
        for n, k, s in zip(c["nodes"], c["num_pipelines"], c["stages"]):
            templates += [product_template(s, gpn, n)] * k
        eng = FakeEngine(gpn, templates)
        created = []
        dpe = DataParallelEngine(eng, fake_pipelines(gpn, templates), new_group=lambda r: created.append(list(r)) or len(created))
        got = {str(l): {str(f): pg.ranks for f, pg in d.items()} for l, d in dpe._dp_process_groups.items()}
        assert got == c["groups"]
        # communicators are created once per distinct rank set, in the reference's first-use order
        dedup = []
        for r in c["order"]:
            if r not in dedup:
                dedup.append(r)
        assert created == dedup and len(created) <= len(c["order"])


def test_sampler_golden():
    for c in load("sampler"):
        for pi, want in enumerate(c["batches"]):
            s = OobleckSampler(range(c["num_samples"]), c["microbatch_size"], pi, c["num_microbatches"], 0, c["epoch"],
                               c["shuffle"])
            assert [list(b) for b in s] == want
            assert s.epoch == c["epoch"] + 1 and s.num_iterations_done == 0   # dataloader.py:99-100


def test_dtype_wire_ids_golden():
    want = load("dtype_ids")
    assert {str(k).replace("torch.", ""): v for k, v in U.DTYPE_TO_ID.items()} == want
    assert [U.DTYPE_TO_ID[d] for d in U.ID_TO_DTYPE] == list(range(len(U.ID_TO_DTYPE)))


def test_pipeline_wiring_matches_oracle():
    t = product_template(4, 1, 4)
    for me in range(4):
        import oobleck_b200.execution.pipeline as P
        orig = P._my_rank
        P._my_rank = lambda me=me: me
        try:
            p = OobleckPipeline(0, t, [0, 1, 2, 3], None, 0, None, layer_cls=types.SimpleNamespace(device_type="cpu"))
            p.initialize_distributed_fsdp()
            p.initialize_distributed_pipeline()
            _, prev, nxt = bk.pipeline_neighbours(p.rank_grid, me)
            assert (p.communication.prev_rank, p.communication.next_rank) == (prev, nxt)
            mine = [lid for lid, pg in p._per_layer_pgs.items() if pg.rank_index() >= 0]
            assert mine == bk.my_layers(p.rank_grid, me)
        finally:
            P._my_rank = orig


# ---- minimum node count (engine.py:490-512; golden table: tests/execution/test_engine.py:394-406) -------------------
@pytest.mark.parametrize(
    ["num_nodes", "num_gpus_per_node", "gpu_mem", "num_layers", "expected_min_num_nodes", "expect_fail"],
    [
        (1, 1, 1024 * 32 * 6, 32, 1, False),
        (1, 1, 1024 * 32 * 6, 64, 2, True),
        (1, 1, 1024 * 128 * 6, 64, 1, False),
        (4, 1, 1024 * 32 * 6, 64, 2, False),
        (4, 1, 1024 * 16 * 6, 64, 4, False),
        (4, 1, 1024 * 16 * 6, 128, 8, True),
        (1, 4, 1024 * 16 * 6, 128, 2, True),
        (1, 4, 1024 * 32 * 6, 128, 1, False),
        (4, 4, 1024 * 16 * 6, 128, 2, False),
        (4, 4, 1024 * 1 * 6, 32, 8, True),
    ],
)
def test_multi_nodes_template_configuration(num_nodes, num_gpus_per_node, gpu_mem, num_layers, expected_min_num_nodes,
                                            expect_fail):
    """The reference's own table, with its fake profile (every layer: 1024 bytes of parameters, no activations)."""
    import re

    from oobleck_b200.execution.engine import node_range
    from oobleck_b200.planning.pipeline_template import LayerExecutionResult, LayerExecutionResults
    fake_profile = LayerExecutionResults([
        LayerExecutionResult(i, 0.1, 0.1, {g + 1: 0.1 for g in range(8)}, {n + 1: 0.1 for n in range(64)}, (1024, 0))
        for i in range(num_layers)])
    if expect_fail:
        with pytest.raises(AssertionError) as e:
            node_range(fake_profile, num_nodes, num_gpus_per_node, gpu_mem)
        assert e.value.args[0].startswith("Minimum required number of nodes")
        match = re.search(r"minimum required: (\d+),", e.value.args[0])
        assert int(match[1]) == expected_min_num_nodes
    else:
        assert node_range(fake_profile, num_nodes, num_gpus_per_node, gpu_mem) == (expected_min_num_nodes, num_nodes)


def test_node_range_counts_the_largest_activation_once():
    from oobleck_b200.execution.engine import node_range
    from oobleck_b200.planning.pipeline_template import LayerExecutionResult, LayerExecutionResults
    prof = LayerExecutionResults([LayerExecutionResult(i, 1.0, 1.0, {}, {}, (100, a)) for i, a in enumerate((5, 700, 30))])
    # 6 * 300 + max(5, 700, 30) = 2500 bytes
    assert node_range(prof, 4, 1, 2500) == (1, 4)
    assert node_range(prof, 4, 1, 2499) == (2, 4)
    assert node_range(prof, 4, 2, 1250) == (1, 4)


def test_measured_profile_feeds_node_range_and_template_search(monkeypatch):
    """The branch of ``instantiate_pipelines`` that only runs on a GPU box (profile -> node range -> template search,
    engine.py:453-523 in the reference), driven here with a fake profile and a fake device."""
    import torch

    from oobleck_b200.execution import engine as E
    from oobleck_b200.execution.dataloader import SyntheticTokenDataset
    from oobleck_b200.planning import profiler as P
    from oobleck_b200.planning.pipeline_template import LayerExecutionResult, LayerExecutionResults

    margs = dict(n_embd=64, n_head=1, num_hidden_layers=6, n_positions=32, vocab_size=211)
    args = E.OobleckArguments(job=E.JobArguments(microbatch_size=1, global_microbatch_size=8, steps=1),
                              model=E.ModelArguments(model_name="gpt2", model_tag="t", model_args=margs))
    ds = SyntheticTokenDataset(num_samples=64, seq_len=32, vocab_size=211, pin_memory=False)
    eng = E.OobleckEngine(0, 4, 1, None, args, dataset=ds)
    assert not eng._templates_injected and eng.layer_costs_source == "FLOP model"

    cost = {"embed": (0.05, 0.1), "block": (1.0, 2.0), "head": (2.5, 5.0)}

    def fake_results(model, microbatch, device=None):
        return LayerExecutionResults([
            LayerExecutionResult(i, cost[l.kind][0], cost[l.kind][1], {}, {}, (4 * l.num_params, l.activation_bytes(1)))
            for i, l in enumerate(model.layers)])

    class Props:
        total_memory = 178 * 2 ** 30

    class Stop(Exception):
        pass

    def stop(self):
        raise Stop

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda d: Props)
    monkeypatch.setattr(P, "measured_layer_results", fake_results)
    monkeypatch.setattr(E.OobleckEngine, "choose_plan", stop)
    with pytest.raises(Stop):
        eng.instantiate_pipelines(8)
    assert eng.min_num_nodes == 1
    assert eng.layer_costs == [sum(cost[l.kind]) for l in eng._model.layers]
    assert "template search" in eng.layer_costs_source
    assert [t._num_nodes for t in eng._pipeline_templates] == [1, 2, 3, 4]
    four = eng._pipeline_templates[-1]
    splits = [list(s._layer_indices) for s in four.get_stages()]
    assert [i for s in splits for i in s] == list(range(8))                  # contiguous, complete
    stage_cost = [sum(eng.layer_costs[i] for i in s) for s in splits]
    assert max(stage_cost) <= 9.0 + 1e-9                                      # 25.65 ms over 4 stages: best max is 3 blocks

    # a device too small for the model on the nodes at hand: the reference's assertion, from the same place
    class Tiny:
        total_memory = 1 << 20
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda d: Tiny)
    eng2 = E.OobleckEngine(0, 2, 1, None, args, dataset=ds)
    with pytest.raises(AssertionError, match="Minimum required number of nodes"):
        eng2.instantiate_pipelines(8)


_LIVE = {}


def live_reference_run():
    """What the reference's own classes produced on random inputs beyond the committed tables, shared by the tests below:
    tests/golden/live_reference.json.gz, recorded by ``gen_golden.py --live 20260923 80 150 13`` (its Python, its C++
    planner objects from oracle/_ref; the last stdout line, gzipped)."""
    import gzip
    if "data" not in _LIVE:
        with gzip.open(os.path.join(G, "live_reference.json.gz"), "rt") as f:
            _LIVE["data"] = json.load(f)
    return _LIVE["data"]


def test_reconfiguration_policy_live_against_the_reference():
    """Beyond the 120 committed failure sets: 450 fresh ones (up to 13 of the 14 nodes lost, so that "Ranks are
    insufficient" and the reference's own failure modes occur too) go through the reference's ``on_reconfigure`` in a child
    process (tests/golden/gen_golden.py --live-reconfigure; the reference's Python with its own C++ planner objects when
    oracle/_ref is built) and through this package's ``plan_new_ranks``."""
    cases = live_reference_run()["reconfigure"]
    assert len(cases) == 450
    outcomes = {"ranks": 0, "error": 0}
    for c in cases:
        gpn = c["gpus_per_node"]
        templates = [product_template(i, gpn, i) for i in range(2, 6)]
        eng = FakeEngine(gpn, templates)
        eng._pipeline = None
        re = ReconfigurationEngine(eng, fake_pipelines(gpn, templates), start_listener=False)
        want = c["result"]
        if "ranks" in want:
            assert re.plan_new_ranks(list(c["failed"])) == want["ranks"], c
            outcomes["ranks"] += 1
        elif want["error"] == "Ranks are insufficient":
            with pytest.raises(RuntimeError, match="insufficient"):
                re.plan_new_ranks(list(c["failed"]))
            outcomes["error"] += 1
        else:
            # the reference dereferenced a missing template (no template of the merged size): the rank lists this
            # package plans must still be well formed -- every survivor exactly once
            try:
                got = re.plan_new_ranks(list(c["failed"]))
            except (RuntimeError, IndexError):
                continue
            alive = sorted(set(range(sum(i * gpn for i in range(2, 6)))) - set(c["failed"]))
            assert sorted(r_ for ranks in got for r_ in ranks) == alive, c
    assert outcomes["ranks"] > 300 and outcomes["error"] > 0, outcomes


def test_dp_groups_and_sampler_live_against_the_reference():
    """80 random heterogeneous data-parallel layouts through the reference's ``DataParallelEngine.__init__`` (engine.py:
    363-398) and 80 random sampler configurations through its ``OobleckSampler`` (dataloader.py:13-100), generated in a
    child process (tests/golden/gen_golden.py --live), against this package's classes."""
    live = live_reference_run()
    assert len(live["dp_groups"]) == 80 and len(live["sampler"]) == 80
    for c in live["dp_groups"]:
        gpn = c["gpus_per_node"]
        templates = []
        for n, k, s in zip(c["nodes"], c["num_pipelines"], c["stages"]):
            templates += [product_template(s, gpn, n)] * k
        eng = FakeEngine(gpn, templates)
        created = []
        dpe = DataParallelEngine(eng, fake_pipelines(gpn, templates),
                                 new_group=lambda r_: created.append(list(r_)) or len(created))
        got = {str(l): {str(f): pg.ranks for f, pg in d.items()} for l, d in dpe._dp_process_groups.items()}
        assert got == c["groups"], c
        dedup = []
        for ranks in c["order"]:
            if ranks not in dedup:
                dedup.append(ranks)
        assert created == dedup
    for c in live["sampler"]:
        for pi, want in enumerate(c["batches"]):
            s = OobleckSampler(range(c["num_samples"]), c["microbatch_size"], pi, c["num_microbatches"], 0, c["epoch"],
                               c["shuffle"])
            assert [list(b) for b in s] == want, c


def test_pipeline_wiring_live_against_the_reference():
    """The reference's unmodified ``OobleckPipeline.__init__`` / ``initialize_distributed_fsdp`` /
    ``initialize_distributed_pipeline`` (pipeline.py:431-456, 565-617), run for every rank of 80 random templates in a child
    process (gen_golden.py --live), against this package's methods of the same names: membership of the pipeline, previous /
    next stage rank, per-layer holders, per-shard-column groups in the reference's ``list(set(ranks))`` order.  Templates
    whose stages own different numbers of GPUs are the stated limit (the reference leaves sends without a receiver there,
    pipeline.py:602-610): this package refuses them, and says so."""
    import oobleck_b200.execution.pipeline as P
    cases = live_reference_run()["wiring"]
    assert len(cases) == 80
    compared = refused = 0
    orig = P._my_rank
    try:
        for c in cases:
            t = product_template(c["stages"], c["gpus_per_node"], c["nodes"])
            widths = {s._num_gpus for s in t.get_stages()}
            for me_s, want in c["per_rank"].items():
                me = int(me_s)
                P._my_rank = lambda me=me: me
                p = OobleckPipeline(0, t, list(c["ranks"]), None, 0, None, layer_cls=types.SimpleNamespace(device_type="cpu"),
                                    stage_group_factory=lambda ranks: ("comm", tuple(ranks)))
                assert p.my_pipeline == want["my_pipeline"]
                if len(widths) > 1:
                    with pytest.raises(NotImplementedError, match="different widths"):
                        p.initialize_distributed_fsdp()
                    refused += 1
                    continue
                p.initialize_distributed_fsdp()
                p.initialize_distributed_pipeline()
                assert [sorted(pg.ranks) for pg in p._per_layer_pgs.values()] == [sorted(g) for g in want["layer_groups"]]
                assert [pg.ranks for pg in p._per_sharded_pp_pgs.values()] == want["shard_groups"]
                assert (p.communication is not None) == want["has_comm"]
                if want["has_comm"]:
                    assert (p.communication.prev_rank, p.communication.next_rank) == (want["prev"], want["next"]), (c, me)
                compared += 1
    finally:
        P._my_rank = orig
    assert compared > 100 and refused > 0, (compared, refused)
