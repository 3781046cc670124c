"""SURVEY 8f N4: the reference's REST layer (api.py, UNMODIFIED) bound to this package.  tests/golden/make_rest_trace.py
ran api.py's routes over this package and recorded every `messaging_system.*` call they made, with its arguments and
result (tests/golden/rest_api_calls.json); replaying that trace checks that each call still exists here and still
answers what the routes got.  The device is the oracle-backed stand-in of tests/fake_shard.py.

The recorded results are this package's own answers, so the replay is a regression snapshot; the route-level
expectations are asserted by the generator while it records.  When the package's answers change on purpose, regenerate
the trace with tests/golden/make_rest_trace.py (which re-checks those expectations) - never edit it by hand.  Attribute
reads are replayed as hasattr checks only: api.py creates the attributes it finds missing, so a read recorded as missing
may exist here later without changing what the routes do."""
import json

from tests import rest_trace


def test_rest_routes_run_on_this_package(golden_dir, tmp_path):
    import swarmdb_b200 as sdb
    from tests.fake_shard import OracleShard

    trace = json.loads((golden_dir / "rest_api_calls.json").read_text())
    init = rest_trace.decode(trace["init"])
    assert init["save_dir"] == rest_trace.SAVE_DIR
    init["save_dir"] = str(tmp_path / "history")
    db = sdb.SwarmsDB(**init, _shard=OracleShard(256, 16, 0, 1),
                      gpu_config=sdb.GpuConfig(max_agents=256, max_groups=16, deterministic_ids=True))
    assert type(db).__module__ == "swarmdb_b200.core"
    methods = set()
    for i, step in enumerate(trace["calls"]):
        if step.get("op") == "set":
            setattr(db, step["attr"], rest_trace.decode(step["value"]))
            continue
        if "attr" in step:
            assert step.get("missing") or hasattr(db, step["attr"]), step
            continue
        methods.add(step["method"])
        got = getattr(db, step["method"])(*rest_trace.decode(step["args"]), **rest_trace.decode(step["kwargs"]))
        assert json.loads(json.dumps(rest_trace.result(got))) == step["result"], (i, step["method"])
    # what the routes rely on beyond the recorded results
    assert {"send_message", "receive_messages", "send_to_group", "broadcast_message", "get_stats", "close"} <= methods
    assert db.get_message("00000000-0000-0000-0000-000000000001").status.value == "processed"
    assert list((tmp_path / "history").glob("message_history_*.json"))          # trigger_save wrote the history file
    db2 = sdb.SwarmsDB(save_dir=str(tmp_path / "probe"), auto_save=False, _shard=OracleShard(4, 1, 0, 1),
                       gpu_config=sdb.GpuConfig(max_agents=4, max_groups=1, deterministic_ids=True))
    assert db2.admin_client.list_topics(timeout=2).topics           # the health route's liveness probe (A:798)
    db2.close()
