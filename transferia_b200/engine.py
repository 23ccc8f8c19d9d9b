"""Host-side mirror of the reference's plug-in surface for the hot path, bound to the C-ABI.

    Engine                  ~ the Sinker middleware instance            pkg/abstract/middleware.go:3
    Engine.plan()           ~ transformation.AddTablePlan               pkg/transformer/transformation.go:46-85
    Engine.push_encode()    ~ transformation.Push + sink encode         transformation.go:122-158,
                                                                        providers/clickhouse/sink_table.go:605-704
    PushResult.errors       ~ TransformerResult.Errors                  pkg/abstract/transformer.go:40-48

Everything computes in libtfgpu.so (hand-written sm_100a kernels).  There is NO CPU fallback: if the
library is missing or no CUDA device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from dataclasses import dataclass
from typing import List, Optional, Tuple

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TFGPU_LIB_PATH") or os.path.join(_HERE, "libtfgpu.so")      # TFGPU_LIB_PATH: a build variant under test

TF_E_FATAL_NODEVICE = -4


class EngineError(RuntimeError):
    """rc > 0: retriable (Push may be retried); rc < 0: fatal (abstract.NewFatalError)."""

    def __init__(self, rc: int, msg: str):
        super().__init__(f"tfgpu rc={rc}: {msg}")
        self.rc = rc
        self.retriable = rc > 0


_lib = None


def _signatures() -> dict:
    """symbol -> (argument types, result type) of every engine entry point of include/tfgpu.h; buffers of numpy arrays and
    bytes objects are passed as void*."""
    vp, cp, i, u32, u64, P = C.c_void_p, C.c_char_p, C.c_int, C.c_uint32, C.c_uint64, C.POINTER
    batch, out = P(abi.TfBatch), P(vp)
    validate_out = [cp, u64, cp, u64]          # describe_out, cap, err_out, err_cap
    sig = {
        "tfgpu_version": ([], cp),
        "tfgpu_engine_create": ([cp, P(C.c_int), i, out], i),
        "tfgpu_engine_destroy": ([vp], i),
        "tfgpu_last_error": ([vp], cp),
        "tfgpu_engine_set_stream": ([vp, vp], i),
        "tfgpu_plan": ([vp, cp, cp, cp, cp, cp, P(C.c_int)], i),
        "tfgpu_plan_validate": ([cp] * 5 + validate_out, i),
        "tfgpu_plan_describe": ([vp, i], cp),
        "tfgpu_push_columns": ([vp, i, batch, out], i),
        "tfgpu_push_encode": ([vp, i, i, batch, out], i),
        "tfgpu_push_encode_selective": ([vp, i, i, batch, i, out], i),
        "tfgpu_engine_h2d_bytes": ([vp], u64),
        "tfgpu_emit_debezium": ([vp, i, cp, batch, P(abi.TfRowMeta), out], i),
        "tfgpu_emit_debezium_crud": ([vp, i, cp, batch, P(abi.TfOldKeys), P(abi.TfRowMeta), out], i),
        "tfgpu_emit_debezium_validate": ([cp] * 5 + validate_out, i),
        "tfgpu_measure": ([vp, batch, vp, P(u64)], i),
        "tfgpu_parse_csv": ([vp, i, cp, vp, u64, i, i, out], i),
        "tfgpu_parse_json": ([vp, i, cp, vp, u64, i, P(abi.TfMsg), u32, i, out], i),
        "tfgpu_parse_debezium": ([vp, i, cp, vp, u64, i, vp, u32, i, out], i),
        "tfgpu_debezium_schema_validate": ([cp] + validate_out, i),
        "tfgpu_push_encode_resident": ([vp, i, i, batch], i),
        "tfgpu_resident_stats": ([vp, P(u64), P(u64), P(u64), P(u64)], i),
        "tfgpu_resident_fetch": ([vp, i, vp, u64], i),
        "tfgpu_debug_lz4_phases": ([vp, i, P(u64)], i),
        "tfgpu_queue_json_batches": ([vp, u64, u64, u64, vp, u64, P(u64)], i),
        "tfgpu_queue_debezium_batches": ([vp, u64, u64, vp, u64, P(u64)], i),
        "tfgpu_result_errors": ([vp], P(abi.TfRowErr)),
        "tfgpu_result_batch": ([vp], batch),
        "tfgpu_result_bytes": ([vp], vp),
        "tfgpu_result_meta_kinds": ([vp], P(C.c_uint8)),
        "tfgpu_result_meta_lsn": ([vp], P(u64)),
        "tfgpu_result_meta_commit_time": ([vp], P(u64)),
        "tfgpu_result_release": ([vp], None),
        "tfgpu_engine_launch_count": ([vp], u64),
        "tfgpu_profile_enable": ([vp, i], i),
        "tfgpu_profile_read": ([vp], cp),
    }
    for name in ("rows_in", "rows_out", "n_errors", "bytes_len", "raw_len", "n_frames", "consumed"):
        sig["tfgpu_result_" + name] = ([vp], u64)
    for name in ("row_sizes", "key_sizes", "dbz_msg_sizes", "part_ids", "selection", "meta_tx_id"):
        sig["tfgpu_result_" + name] = ([vp], P(u32))
    return sig


_SIGNATURES = _signatures()
EXPORTED_SYMBOLS = list(_SIGNATURES)


def load_library():
    """dlopen transferia_b200/libtfgpu.so and declare every symbol of include/tfgpu.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` — "
                           "the engine has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    for name, (argtypes, restype) in _SIGNATURES.items():
        fn = getattr(L, name)
        fn.argtypes, fn.restype = argtypes, restype
    _lib = L
    return L


def debezium_table_schema(schema_text: str):
    """The table schema the reference derives from a Kafka Connect envelope schema's `after` struct with the default receivers
    (pkg/debezium/receiver.go:46-62, receiver_engine.go:104-141, common/field_receiver_default.go:15-30): key = !optional."""
    sch = json.loads(schema_text)
    node = next((f for f in sch.get("fields", []) if f.get("field") == "after"), None)
    if node is None:
        raise EngineError(-1, "debezium schema has no 'after' struct")
    out = []
    for f in node.get("fields", []):
        kt, nm = f.get("type"), f.get("name", "")
        if kt in ("int8", "int16", "int32", "int64", "boolean"): yt = kt
        elif kt == "string": yt = "utf8"
        elif kt in ("float", "double"): yt = "double"
        elif kt == "bytes": yt = "utf8" if nm == "org.apache.kafka.connect.data.Decimal" else "string"
        elif kt == "struct" and nm == "io.debezium.data.geometry.Point": yt = "utf8"
        elif kt == "struct" and nm == "io.debezium.data.VariableScaleDecimal": yt = "double"
        else: raise EngineError(-1, f"debezium: kafka type {kt} / {nm} has no default receiver on the device")
        out.append({"name": f["field"], "type": yt, "key": not f.get("optional", False)})
    return out


def queue_debezium_batches(value_sizes, max_message_size: int = 0):
    """MergeWithMaxMessageSize of the queue Debezium serializer (host only): first row of every merged message, then n."""
    import numpy as np
    L = load_library()
    a = np.asarray(value_sizes, dtype=np.uint32); st = np.zeros(len(a) + 1, dtype=np.uint64); k = C.c_uint64()
    rc = L.tfgpu_queue_debezium_batches(a.ctypes.data, len(a), max_message_size, st.ctypes.data, len(st), C.byref(k))
    if rc != 0:
        raise EngineError(rc, "tfgpu_queue_debezium_batches")
    return [int(x) for x in st[:k.value + 1]]


def queue_json_batches(json_row_sizes, max_message_size: int = 0, max_change_items: int = 0):
    """BatchJSON of the queue JSON serializer (host only): first row of every message, then n."""
    import numpy as np
    L = load_library()
    a = np.asarray(json_row_sizes, dtype=np.uint32); st = np.zeros(len(a) + 1, dtype=np.uint64); k = C.c_uint64()
    rc = L.tfgpu_queue_json_batches(a.ctypes.data, len(a), max_message_size, max_change_items, st.ctypes.data, len(st), C.byref(k))
    if rc != 0:
        raise EngineError(rc, "tfgpu_queue_json_batches")
    return [int(x) for x in st[:k.value + 1]]


def json_result_schema(fields, opts: Optional[dict] = None):
    """The generic parser's result schema for declared `fields` (addAuxFields, pkg/parsers/generic/generic_parser.go:115-164):
    `_rest` when add_rest, then _timestamp/_partition/_offset/_idx when add_dedupe_keys (system keys unless
    mark_dedupe_keys_as_system and a declared field is a key); a name already taken gets the `_delivery_` prefix (:93-100)."""
    opts = opts or {}
    out = [dict(f, required=bool(f.get("required") or f.get("key"))) for f in fields]

    def dedup(name):
        while any(c["name"] == name for c in out):
            name = "_delivery_" + name
        return name
    if opts.get("add_rest"):
        out.append({"name": dedup("_rest"), "type": "any"})
    if opts.get("add_dedupe_keys"):
        sys_key = not (opts.get("mark_dedupe_keys_as_system") and any(f.get("key") for f in fields))
        for n, t in (("_timestamp", "timestamp"), ("_partition", "string"), ("_offset", "uint64"), ("_idx", "uint32")):
            out.append({"name": dedup(n), "type": t, "key": sys_key, "required": sys_key})
    return out


def _schema_json(schema) -> str:
    """A table schema as the C-ABI takes it: JSON text as given, or the column dicts without their `_`-prefixed keys."""
    return schema if isinstance(schema, str) else json.dumps([{k: v for k, v in c.items() if not k.startswith("_")} for c in schema])


def _host_validate(fn_name: str, *args, out_cap: int = 1 << 20):
    """Calls a host-only validator with its leading arguments and the describe / error buffers: the describe JSON, or EngineError."""
    out = C.create_string_buffer(out_cap); err = C.create_string_buffer(4096)
    rc = getattr(load_library(), fn_name)(*args, out, len(out), err, len(err))
    if rc != 0:
        raise EngineError(rc, err.value.decode(errors="replace"))
    return json.loads(out.value.decode())


def debezium_schema_validate(schema_text: str) -> list:
    """Host-only: [{"name","type","key","recv","scale"}] the C++ side derives from an envelope schema (no GPU needed), or raises EngineError."""
    return _host_validate("tfgpu_debezium_schema_validate", schema_text.encode())


def emit_debezium_validate(namespace: str, name: str, schema, transformers, opts: dict) -> dict:
    """Host-only set-up of the Debezium emitter (no GPU needed): {"forms", "keys", "template"} or raises EngineError."""
    return _host_validate("tfgpu_emit_debezium_validate", namespace.encode(), name.encode(), _schema_json(schema).encode(),
                          json.dumps(transformers or []).encode(), json.dumps(opts).encode(), out_cap=1 << 22)


def plan_validate(namespace: str, name: str, schema, transformers=None, sink=None) -> dict:
    """Host-only plan construction (no GPU needed): returns the describe JSON or raises EngineError."""
    return _host_validate("tfgpu_plan_validate", namespace.encode(), name.encode(), _schema_json(schema).encode(),
                          json.dumps(transformers or []).encode(), None if sink is None else json.dumps(sink).encode())


@dataclass
class PushResult:
    rows_in: int
    rows_out: int
    raw_len: int
    n_frames: int
    wire: bytes                            # empty when the call was asked not to copy the bytes
    errors: List[Tuple[int, int, int]]     # (input row, TF_ROWERR_*, transformer index)
    wire_len: int = 0
    # per output row (numpy uint32; row_sizes of push_encode: a list), None when the result has none: row bytes of the row-text
    # formats, key message bytes and (rows_out x 7) message sizes of the Debezium emitter, ChangeItem.PartID with a sharder
    row_sizes: Optional["np.ndarray | List[int]"] = None
    key_sizes: Optional["np.ndarray"] = None
    msg_sizes: Optional["np.ndarray"] = None
    part_ids: Optional["np.ndarray"] = None


class Engine:
    def __init__(self, device: int = 0, frame_bytes: int = 15360):
        self._L = load_library()
        self._h = C.c_void_p()
        dev = (C.c_int * 1)(device)
        cfg = json.dumps({"frame_bytes": frame_bytes}).encode()
        rc = self._L.tfgpu_engine_create(cfg, dev, 1, C.byref(self._h))
        if rc != 0:
            msg = "no CUDA device — this engine has no CPU fallback" if rc == TF_E_FATAL_NODEVICE else "engine_create failed"
            raise EngineError(rc, msg)
        self.device = device
        self.frame_bytes = frame_bytes

    def close(self):
        if self._h:
            self._L.tfgpu_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise EngineError(rc, (self._L.tfgpu_last_error(self._h) or b"").decode(errors="replace"))

    def set_stream(self, cuda_stream_ptr: Optional[int]):
        self._check(self._L.tfgpu_engine_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))

    def plan(self, namespace: str, name: str, schema, transformers=None, sink=None) -> int:
        sj = _schema_json(schema)
        tj = json.dumps(transformers or [])
        kj = None if sink is None else json.dumps(sink).encode()
        pid = C.c_int(-1)
        self._check(self._L.tfgpu_plan(self._h, namespace.encode(), name.encode(), sj.encode(), tj.encode(), kj, C.byref(pid)))
        return pid.value

    def describe(self, plan_id: int) -> dict:
        s = self._L.tfgpu_plan_describe(self._h, plan_id)
        return json.loads(s.decode()) if s else {}

    def push_encode(self, plan_id: int, batch: abi.Batch, wire_fmt: int = abi.TF_WIRE_CH_NATIVE_LZ4, copy_bytes: bool = True, selective: Optional[int] = None) -> PushResult:
        """selective=N: tfgpu_push_encode_selective with N host threads for the gather (0 = default) — two phases, fewer PCIe bytes when
        the plan's filter_rows keeps a fraction of the rows; same result."""
        tb = batch.as_struct()
        res = C.c_void_p()
        if selective is None:
            self._check(self._L.tfgpu_push_encode(self._h, plan_id, wire_fmt, C.byref(tb), C.byref(res)))
        else:
            self._check(self._L.tfgpu_push_encode_selective(self._h, plan_id, wire_fmt, C.byref(tb), int(selective), C.byref(res)))
        try:
            out = self._read_wire(res, copy_bytes)
            if out.row_sizes is not None:      # push_encode gives the row sizes as a list of ints
                out.row_sizes = out.row_sizes.tolist()
            return out
        finally:
            self._L.tfgpu_result_release(res)

    def h2d_bytes(self) -> int:
        return int(self._L.tfgpu_engine_h2d_bytes(self._h))

    @staticmethod
    def _per_row(ptr, shape):
        """A copy of the result array `ptr` points at, None when the result has none."""
        import numpy as np
        return np.ctypeslib.as_array(ptr, shape=shape).copy() if (ptr and shape[0]) else None

    def _errors(self, res) -> List[Tuple[int, int, int]]:
        ep = self._L.tfgpu_result_errors(res)
        return [(ep[k].row, ep[k].code, ep[k].term) for k in range(self._L.tfgpu_result_n_errors(res))]

    def _read_wire(self, res, copy_bytes: bool, per_row: bool = True) -> PushResult:
        """PushResult of a wire-format result; copy_bytes=False leaves the wire bytes in the engine's pinned landing buffer and
        only reports their length. per_row=False skips the per-row arrays: the parsers' callers take the bytes only, and copying
        the row sizes of 400 k JSONEachRow rows cost 3 % of tfgpu_parse_json on a B200 (1000 W power limit)."""
        L = self._L
        n = L.tfgpu_result_bytes_len(res)
        out = PushResult(L.tfgpu_result_rows_in(res), L.tfgpu_result_rows_out(res), L.tfgpu_result_raw_len(res), L.tfgpu_result_n_frames(res),
                         C.string_at(L.tfgpu_result_bytes(res), n) if (copy_bytes and n) else b"", self._errors(res), n)
        if not per_row:
            return out
        k = int(out.rows_out)
        out.row_sizes, out.key_sizes = self._per_row(L.tfgpu_result_row_sizes(res), (k,)), self._per_row(L.tfgpu_result_key_sizes(res), (k,))
        out.msg_sizes, out.part_ids = self._per_row(L.tfgpu_result_dbz_msg_sizes(res), (k, 7)), self._per_row(L.tfgpu_result_part_ids(res), (k,))
        return out

    def _result_batch(self, res):
        import numpy as np
        L = self._L
        ob = L.tfgpu_result_batch(res)
        n = int(L.tfgpu_result_rows_out(res))
        cols = []
        if ob:
            b = ob.contents
            for k in range(b.ncols):
                c = b.cols[k]
                def arr(ptr, nbytes, dtype):
                    if not ptr or nbytes == 0:
                        return None if not ptr else np.zeros(0, dtype=dtype)
                    return np.frombuffer(C.string_at(ptr, nbytes), dtype=dtype).copy()
                t = c.type
                if t in abi.VAR_TYPES:
                    cols.append(abi.Column(t, offsets=arr(c.offsets, 4 * (n + 1), np.uint32), heap=arr(c.heap, c.heap_len, np.uint8) if c.heap else np.zeros(0, np.uint8),
                                           validity=arr(c.validity, (n + 7) // 8, np.uint8), aux=arr(c.aux, n, np.uint8)))
                else:
                    dt = abi.FIXED_DTYPE[t]
                    cols.append(abi.Column(t, values=arr(c.values, n * np.dtype(dt).itemsize, dt), validity=arr(c.validity, (n + 7) // 8, np.uint8),
                                           aux=arr(c.aux, 4 * n, np.uint32)))
        self.last_part_ids = self._per_row(L.tfgpu_result_part_ids(res), (n,))      # of the batch just returned (push_columns / parsers)
        return abi.Batch(n, cols), self._errors(res)

    def push_columns(self, plan_id: int, batch: abi.Batch) -> Tuple[abi.Batch, List[Tuple[int, int, int]]]:
        """Transformer chain only: (Transformed rows as a host Batch, row errors) — abstract.TransformerResult."""
        tb = batch.as_struct()
        res = C.c_void_p()
        self._check(self._L.tfgpu_push_columns(self._h, plan_id, C.byref(tb), C.byref(res)))
        try:
            return self._result_batch(res)
        finally:
            self._L.tfgpu_result_release(res)

    @staticmethod
    def _host_bytes(data):
        """(pointer, length, keepalive) of a bytes object or a (pinned) torch uint8 tensor, without copying."""
        if hasattr(data, "data_ptr"):
            return C.c_void_p(data.data_ptr()), int(data.numel()), data
        buf = C.c_char_p(data if data else b"\0")              # the bytes object's own storage
        return C.cast(buf, C.c_void_p), len(data), buf

    def parse_csv(self, plan_id: int, data, opts: Optional[dict] = None, wire_fmt: int = 0, copy_bytes: bool = True):
        """CSV bytes (a bytes object or a pinned torch uint8 tensor, used in place) -> typed columns -> the plan's transformer chain, all on
        the device. wire_fmt 0: (Batch, row errors, consumed bytes); otherwise (PushResult, consumed bytes); copy_bytes=False leaves the
        wire bytes in the engine's pinned landing buffer and only reports their length."""
        ptr, total, keep = self._host_bytes(data)
        res = C.c_void_p()
        self._check(self._L.tfgpu_parse_csv(self._h, plan_id, json.dumps(opts or {}).encode(), ptr, total, abi.TF_MEM_HOST, wire_fmt, C.byref(res)))
        try:
            consumed = int(self._L.tfgpu_result_consumed(res))
            if wire_fmt == 0:
                b, errs = self._result_batch(res)
                return b, errs, consumed
            return self._read_wire(res, copy_bytes, per_row=False), consumed
        finally:
            self._L.tfgpu_result_release(res)

    def parse_debezium(self, plan_id: int, data, msg_ends, schema_text: str, schema_registry: bool = False, schema_id: int = 0,
                       check_table: bool = False, wire_fmt: int = 0, copy_bytes: bool = True):
        """Debezium messages -> typed columns (default receivers) -> the plan's chain, on the device; one row per message.
        wire_fmt 0: (Batch, row errors, meta) with meta = {"selection", "kinds", "tx_id", "lsn", "commit_time"} (numpy; the last four
        per MESSAGE, selection per output row); otherwise (PushResult, meta)."""
        import numpy as np
        ends = np.asarray(msg_ends, dtype=np.uint64)
        opts = {"schema_text": schema_text, "schema_registry": schema_registry, "schema_id": schema_id, "check_table": check_table}
        ptr, total, keep = self._host_bytes(data)
        res = C.c_void_p()
        self._check(self._L.tfgpu_parse_debezium(self._h, plan_id, json.dumps(opts).encode(), ptr, total, abi.TF_MEM_HOST, ends.ctypes.data, len(ends), wire_fmt, C.byref(res)))
        try:
            L = self._L
            nin, nout = int(L.tfgpu_result_rows_in(res)), int(L.tfgpu_result_rows_out(res))
            def arr(fn, n, dt):
                p = getattr(L, fn)(res)
                return np.ctypeslib.as_array(p, shape=(n,)).astype(dt).copy() if (p and n) else np.zeros(0, dtype=dt)
            meta = {"selection": arr("tfgpu_result_selection", nout, np.uint32), "kinds": arr("tfgpu_result_meta_kinds", nin, np.uint8), "tx_id": arr("tfgpu_result_meta_tx_id", nin, np.uint32),
                    "lsn": arr("tfgpu_result_meta_lsn", nin, np.uint64), "commit_time": arr("tfgpu_result_meta_commit_time", nin, np.uint64)}
            if wire_fmt == 0:
                b, errs = self._result_batch(res)
                return b, errs, meta
            return self._read_wire(res, copy_bytes, per_row=False), meta
        finally:
            self._L.tfgpu_result_release(res)

    def lz4_phases(self, enable: bool = True):
        """Cycles spent per k_lz4_frames phase (stage, match, parse, scan, emit) since the last read (profiling aid)."""
        out = (C.c_uint64 * 8)()
        self._check(self._L.tfgpu_debug_lz4_phases(self._h, 1 if enable else 0, out))
        return [int(x) for x in out]

    def emit_debezium(self, plan_id: int, batch: abi.Batch, opts: dict, meta: Optional[dict] = None, copy_bytes: bool = True, old: Optional[abi.Batch] = None,
                      old_present=None, old_row_has=None) -> PushResult:
        """Queue Debezium serializer (Emitter.EmitKV) over the rows that survive the plan's chain: PushResult whose `wire` holds the
        messages of every row (key, value; a delete adds its tombstone key; a key-changing update is delete + tombstone + insert);
        `key_sizes` / `row_sizes` give the first key and the total per row, `msg_sizes` (rows_out x 7) the message count and
        (key bytes, value bytes | 0xFFFFFFFF) per message. meta: {"id", "lsn", "commit_time", "txid_offsets", "txid_heap"} arrays in the
        memory space of the batch. old / old_present / old_row_has: ChangeItem.OldKeys (tf_old_keys)."""
        import numpy as np
        tb = batch.as_struct()
        meta = meta or {}
        m, keep = abi.make_row_meta(meta.get("id"), meta.get("lsn"), meta.get("commit_time"), meta.get("txid_offsets"), meta.get("txid_heap"))
        res = C.c_void_p()
        ok, okeep = (abi.make_old_keys(old, old_present or [], old_row_has) if old is not None else (None, None))
        self._check(self._L.tfgpu_emit_debezium_crud(self._h, plan_id, json.dumps(opts).encode(), C.byref(tb), C.byref(ok) if ok is not None else None,
                                                     C.byref(m), C.byref(res)))
        try:
            out = self._read_wire(res, copy_bytes)
            if not out.rows_out:           # no rows, no per-row arrays in the result: the emitter's are empty, not absent
                out.row_sizes, out.key_sizes, out.msg_sizes = np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros((0, 7), np.uint32)
            return out
        finally:
            self._L.tfgpu_result_release(res)

    def measure(self, batch: abi.Batch):
        """Measurer middleware: ChangeItem.Size.Values of every row (numpy uint64) and their sum."""
        import numpy as np
        tb = batch.as_struct(); per = np.zeros(batch.nrows, dtype=np.uint64); tot = C.c_uint64()
        self._check(self._L.tfgpu_measure(self._h, C.byref(tb), per.ctypes.data, C.byref(tot)))
        return per, tot.value

    def parse_json(self, plan_id: int, data: bytes, opts: Optional[dict] = None, msgs: Optional[list] = None, wire_fmt: int = 0, copy_bytes: bool = True):
        """JSON-lines messages -> typed columns of the parser's result schema -> the plan's transformer chain, on the device.
        msgs: [(end, offset, write_sec, write_nsec)] (default: one message = all of `data`).
        wire_fmt 0: (Batch, row errors, non-empty lines); otherwise PushResult (copy_bytes=False leaves the wire bytes in the
        engine's pinned landing buffer and only reports their length)."""
        ptr, total, keep = self._host_bytes(data)
        msgs = msgs if msgs is not None else [(total, 0, 0, 0)]
        ms = (abi.TfMsg * max(1, len(msgs)))()
        for k, (end, off, ws, wn) in enumerate(msgs):
            ms[k].end, ms[k].offset, ms[k].write_sec, ms[k].write_nsec = end, off, ws, wn
        res = C.c_void_p()
        self._check(self._L.tfgpu_parse_json(self._h, plan_id, json.dumps(opts or {}).encode(), ptr, total, abi.TF_MEM_HOST, ms, len(msgs), wire_fmt, C.byref(res)))
        try:
            if wire_fmt == 0:
                b, errs = self._result_batch(res)
                return b, errs, int(self._L.tfgpu_result_rows_in(res))
            return self._read_wire(res, copy_bytes, per_row=False)
        finally:
            self._L.tfgpu_result_release(res)

    def push_encode_resident(self, plan_id: int, batch: abi.Batch, wire_fmt: int = abi.TF_WIRE_CH_NATIVE_LZ4):
        """Asynchronous, HBM-resident: no copies, no host sync (kernel-only timing)."""
        tb = batch.as_struct()
        self._check(self._L.tfgpu_push_encode_resident(self._h, plan_id, wire_fmt, C.byref(tb)))

    def resident_stats(self) -> dict:
        a, b, c, d = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._check(self._L.tfgpu_resident_stats(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"rows_out": a.value, "raw_bytes": b.value, "wire_bytes": c.value, "n_errors": d.value}

    def resident_fetch(self, what: int, nbytes: int) -> bytes:
        buf = C.create_string_buffer(max(1, nbytes))           # (a c_uint8 array would come back as a list of ints when sliced)
        self._check(self._L.tfgpu_resident_fetch(self._h, what, buf, nbytes))
        return C.string_at(buf, nbytes)

    def profile_enable(self, on: bool = True):
        self._check(self._L.tfgpu_profile_enable(self._h, 1 if on else 0))

    def profile_read(self) -> list:
        """[{name, ms}] per kernel of the last call (synchronises the stream)."""
        s = self._L.tfgpu_profile_read(self._h)
        return json.loads(s.decode()) if s else []

    def launch_count(self) -> int:
        return int(self._L.tfgpu_engine_launch_count(self._h))
