"""Load the UNMODIFIED reference `SwarmsDB` class for oracle pinning (TEST INFRASTRUCTURE ONLY).

Loads /root/reference/swarmdb/" main.py" where that exists (the build container) and otherwise the
byte-identical copy that `oracle/build_ref.py` staged under oracle/_ref/ (git-ignored; it travels to
the GPU box with the snapshot).  It is used by `tests/golden/make_golden.py` to generate the committed
golden fixtures, by the CPU tests that re-check the restatement (`oracle/cpu_ref.c`, `oracle/pyref.py`)
against the live reference, and by `bench.py`'s reference-python timing leg.

The reference cannot run as shipped (SURVEY.md section 0.3); exactly two shims are applied and
nothing else:

  1. `Message.to_dict` (M:91-98) calls `dataclasses.asdict` on a pydantic model and raises
     TypeError before `producer.produce` is reached (M:466).  The evident intent - pydantic
     dump with the three enum fields flattened to `.value` - is substituted.
  2. Optional deterministic `uuid.uuid4` / `time.time` through the module globals bound at
     M:4-5, so message ids and timestamps are reproducible in fixtures.

The Kafka client (`confluent_kafka`, absent from this image) is provided by the in-memory
partition-log stub in `oracle/kafka_stub/`.
"""
from __future__ import annotations

import importlib.util
import itertools
import os
import sys
import types
import uuid as _uuid
from pathlib import Path

REFERENCE_ROOT = Path(os.environ.get("SWARMDB_REFERENCE_ROOT", "/root/reference"))
REFERENCE_MAIN = REFERENCE_ROOT / "swarmdb" / " main.py"   # the filename really starts with a space
STAGED_MAIN = Path(__file__).resolve().parent / "_ref" / "swarmdb_reference_main.py"    # oracle/build_ref.py
_STUB_DIR = Path(__file__).resolve().parent / "kafka_stub"


def readable_file(path: Path) -> bool:
    """True when `path` is a file this user can read; a directory it may not enter counts as absent."""
    try:
        return path.is_file() and os.access(path, os.R_OK)
    except OSError:
        return False


def reference_path():
    """The unmodified reference file: in place when /root/reference exists, else the staged copy, else None."""
    if readable_file(REFERENCE_MAIN):
        return REFERENCE_MAIN
    if readable_file(STAGED_MAIN):
        return STAGED_MAIN
    return None


def reference_available() -> bool:
    return reference_path() is not None


class _DetUuid(types.ModuleType):
    """`uuid` look-alike whose uuid4() counts 1, 2, 3 ... (shim 2)."""

    def __init__(self) -> None:
        super().__init__("uuid")
        self._ctr = itertools.count(1)
        self.UUID = _uuid.UUID

    def uuid4(self):
        return _uuid.UUID(int=next(self._ctr))


class _DetTime(types.ModuleType):
    """`time` look-alike whose time() advances by 1 microsecond per call from 1.0e9 (shim 2)."""

    def __init__(self) -> None:
        super().__init__("time")
        self._t = 1.0e9

    def time(self) -> float:
        self._t += 1.0e-6
        return self._t


def load_reference(deterministic: bool = True, module_name: str = "swarmdb_reference_main"):
    """Return the reference module object (fresh load each call, fresh stub broker)."""
    src = reference_path()
    if src is None:
        raise FileNotFoundError(f"reference not present at {REFERENCE_MAIN} and not staged at {STAGED_MAIN}")
    if str(_STUB_DIR) not in sys.path:
        sys.path.insert(0, str(_STUB_DIR))
    import confluent_kafka  # the stub

    confluent_kafka.reset_broker()
    spec = importlib.util.spec_from_file_location(module_name, str(src))
    mod = importlib.util.module_from_spec(spec)
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # pydantic v1-style @validator deprecation
        spec.loader.exec_module(mod)

    # shim 1: Message.to_dict, intent of M:93-98
    def to_dict(self):
        d = self.model_dump()
        d["type"] = self.type.value
        d["priority"] = self.priority.value
        d["status"] = self.status.value
        return d

    mod.Message.to_dict = to_dict

    # shim 2: deterministic ids / timestamps through the globals bound at M:4-5
    if deterministic:
        mod.uuid = _DetUuid()
        mod.time = _DetTime()
    return mod


def make_reference_db(mod, save_dir: str, num_partitions: int = 1, quiet: bool = True, **kw):
    """Construct the reference SwarmsDB over the stub broker with autosave off."""
    cfg = mod.KafkaConfig(num_partitions=num_partitions)
    db = mod.SwarmsDB(config=cfg, save_dir=save_dir, auto_save=False, **kw)
    if quiet:
        # the per-message loguru file sink (M:486) is >50% of send cost and irrelevant to parity
        mod.logger.remove()
    return db
