"""The calls the reference's REST layer (api.py, run UNMODIFIED) makes on its `messaging_system`, as a JSON trace.

tests/golden/make_rest_trace.py drives api.py's routes over this package and records, through `Recorder`, every
constructor argument, method call (arguments and result) and attribute the routes touch; tests/test_rest_layer_cpu.py
replays the trace against the package and expects the same results.  Message timestamps and the save time are wall
clock and are left out of the recorded results."""
from enum import Enum

CLOCK_KEYS = ("timestamp", "last_save_time")
SAVE_DIR = "<save_dir>"


def _enum_types():
    from swarmdb_b200 import core
    return {c.__name__: c for c in (core.MessageType, core.MessagePriority, core.MessageStatus)}


def encode(v):
    """JSON form of a call argument."""
    from swarmdb_b200.core import KafkaConfig
    if isinstance(v, Enum):
        return {"__enum__": type(v).__name__, "value": v.value}
    if isinstance(v, KafkaConfig):
        return {"__kafka_config__": dict(vars(v))}
    if isinstance(v, (list, tuple)):
        return [encode(x) for x in v]
    if isinstance(v, dict):
        return {k: encode(x) for k, x in v.items()}
    return v


def decode(v):
    from swarmdb_b200.core import KafkaConfig
    if isinstance(v, list):
        return [decode(x) for x in v]
    if isinstance(v, dict):
        if "__enum__" in v:
            return _enum_types()[v["__enum__"]](v["value"])
        if "__kafka_config__" in v:
            return KafkaConfig(**v["__kafka_config__"])
        return {k: decode(x) for k, x in v.items()}
    return v


def result(v):
    """JSON form of a call's result, wall-clock fields dropped."""
    from swarmdb_b200.core import Message
    if isinstance(v, Message):
        v = v.to_dict()
    if isinstance(v, Enum):
        return v.value
    if isinstance(v, (list, tuple)):
        return [result(x) for x in v]
    if isinstance(v, dict):
        return {str(k): result(x) for k, x in v.items() if k not in CLOCK_KEYS}
    if hasattr(v, "item"):                                  # numpy scalars
        return v.item()
    return v


class Recorder:
    """Stands in for the SwarmsDB instance api.py builds; forwards everything to `db` and logs what it was asked."""

    def __init__(self, db, log):
        object.__setattr__(self, "_db", db)
        object.__setattr__(self, "_log", log)

    def __getattr__(self, name):
        try:
            v = getattr(self._db, name)
        except AttributeError:
            self._log.append({"attr": name, "op": "get", "missing": True})        # api.py probes with hasattr first
            raise
        if not callable(v):
            self._log.append({"attr": name, "op": "get"})
            return v

        def call(*args, **kwargs):
            out = v(*args, **kwargs)
            self._log.append({"method": name, "args": encode(list(args)), "kwargs": encode(kwargs), "result": result(out)})
            return out
        return call

    def __setattr__(self, name, v):
        self._log.append({"attr": name, "op": "set", "value": encode(v)})
        setattr(self._db, name, v)
