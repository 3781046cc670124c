"""Generate tests/golden/rest_api_calls.json: the reference's REST layer (api.py, UNMODIFIED) run over this package.

Needs the reference checkout (SWARMDB_REFERENCE_ROOT, as oracle/ref_loader.py) plus fastapi and PyJWT:

    python tests/golden/make_rest_trace.py

The device is the oracle-backed stand-in of tests/fake_shard.py.  Route coroutines are called directly (no HTTP
client), the scenario's expectations are asserted while it runs, and every call the routes make on
`messaging_system` is written out (tests/rest_trace.py) for tests/test_rest_layer_cpu.py to replay."""
import asyncio
import importlib.util
import json
import os
import sys
import tempfile
import warnings
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle import ref_loader  # noqa: E402
from tests import rest_trace  # noqa: E402

REF_API = ref_loader.REFERENCE_ROOT / "api.py"
OUT = Path(__file__).resolve().parent / "rest_api_calls.json"


def run(coro):
    return asyncio.run(coro)


def drive_routes(api):
    """The REST scenario: auth, registration, p2p / group / broadcast sends, receives, status update, admin routes."""
    db = api.messaging_system._db                # the package object itself: these checks are not route calls
    tok = run(api.login_for_access_token(api.UserCredentials(username="a1", password="x")))
    from fastapi.security import HTTPAuthorizationCredentials
    assert api.get_current_agent(HTTPAuthorizationCredentials(scheme="Bearer", credentials=tok["access_token"])) == "a1"

    for a in ("a1", "a2", "a3"):
        r = run(api.register_agent(api.AgentRegistrationRequest(agent_id=a, description="d", capabilities=["c"]), agent_id=a))
        assert r == {"status": "success", "agent_id": a}
    assert db.agent_metadata["a2"]["capabilities"] == ["c"]

    sent = run(api.send_message(api.MessageRequest(content={"q": 1}, receiver_id="a2", priority=api.MessagePriorityEnum.HIGH,
                                                   metadata={"k": "v"}), current_agent="a1"))
    assert sent.sender_id == "a1" and sent.receiver_id == "a2" and sent.status.value == "delivered"
    got = run(api.receive_messages(max_messages=10, timeout=0.1, current_agent="a2"))
    assert [m.id for m in got] == [sent.id] and got[0].content == {"q": 1} and got[0].status.value == "read"
    assert got[0].metadata == {"k": "v"} and got[0].priority.value == 2

    assert run(api.create_agent_group(api.AgentGroupRequest(group_name="team", agent_ids=["a1", "a2", "a3"]), current_agent="a1"))["status"] == "success"
    ids = run(api.send_group_message(api.GroupMessageRequest(group_name="team", content="stand-up"), current_agent="a1"))
    assert len(ids) == 2
    assert [m.content for m in run(api.receive_messages(current_agent="a3"))] == ["stand-up"]
    bid = run(api.broadcast_message(api.BroadcastRequest(content="all hands", exclude_agents=["a3"]), current_agent="a1"))
    assert [m.content for m in run(api.receive_messages(current_agent="a2"))] == ["stand-up", "all hands"]
    assert run(api.receive_messages(current_agent="a3")) == []

    one = run(api.get_message(sent.id, current_agent="a2"))
    assert one.id == sent.id
    assert run(api.update_message_status(sent.id, api.MessageStatusEnum.PROCESSED, current_agent="a2"))["status"] == "success"
    assert db.get_message(sent.id).status.value == "processed"

    health = run(api.health_check())
    assert health.status == "ok" and health.kafka_connected is True          # admin_client.list_topics liveness probe
    stats = run(api.system_stats(current_agent="admin"))
    assert stats["total_messages"] == db.message_count and stats["active_agents"] == 3
    assert run(api.trigger_save(current_agent="admin"))["status"] == "success"
    assert run(api.resend_failed_messages(current_agent="admin"))["status"] == "success"
    assert run(api.flush_old_messages(older_than=None, current_agent="admin"))["status"] == "success"
    assert run(api.auto_scale_partitions(current_agent="admin"))["status"] == "success"
    assert run(api.deregister_agent("a3", current_agent="a3")) == {"status": "success", "agent_id": "a3"}
    assert bid["message_id"] in db.messages          # (the route returns a dict although it declares List[str], A:507/530)


def main() -> None:
    import swarmdb                      # the alias package the reference imports (api.py:29-36)
    import swarmdb_b200 as sdb
    from tests.fake_shard import OracleShard

    with tempfile.TemporaryDirectory() as tmp:
        save_dir = str(Path(tmp) / "history")
        trace = {"init": None, "calls": []}

        def make_db(*args, **kwargs):
            assert not args
            init = rest_trace.encode(kwargs)
            init["save_dir"] = rest_trace.SAVE_DIR if kwargs.get("save_dir") == save_dir else init.get("save_dir")
            init["config"]["__kafka_config__"]["group_id"] = "api_server"          # api.py appends a random uuid4 suffix
            trace["init"] = init
            db = sdb.SwarmsDB(**kwargs, _shard=OracleShard(256, 16, 0, 1),
                              gpu_config=sdb.GpuConfig(max_agents=256, max_groups=16, deterministic_ids=True))
            return rest_trace.Recorder(db, trace["calls"])

        swarmdb.SwarmsDB = make_db
        os.environ["MESSAGE_HISTORY_DIR"] = save_dir
        spec = importlib.util.spec_from_file_location("reference_api_under_test", str(REF_API))
        api = importlib.util.module_from_spec(spec)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            spec.loader.exec_module(api)
        drive_routes(api)
        assert list(Path(save_dir).glob("message_history_*.json"))
        api.shutdown_event()
    OUT.write_text(json.dumps(trace, indent=1, sort_keys=True) + "\n")
    print(f"{OUT.name}: {len(trace['calls'])} calls and attribute uses")


if __name__ == "__main__":
    main()
