#!/usr/bin/env python
"""bench.py — ChangeItems/sec on ClickBench-shaped 99-column batches (BASELINE.json metric).

A step = one pass of the hot path over one synthetic batch of `--rows` ChangeItems (default 1 M):
    filter_rows (counterid > K AND url ~ '://')  ->  typesystem cast  ->  ClickHouse native block
    ->  LZ4 frames + CityHash128          (BASELINE.json configs[2], the config the metric is quoted on)

  value   kernel-only: the batch is resident in HBM, tfgpu_push_encode_resident, CUDA events, max over ranks
  e2e     the same call a user makes (tfgpu_push_encode) with pinned HOST buffers: H2D of every column and
          D2H of the wire bytes are inside the timed region
  roofline  dominant kernel (k_lz4_frames): algorithmic bytes (raw block read + LZ4 bytes written) / its
          CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the C++ oracle port of the Go row loop, timed on the host cores (rank 0, N=1)

`--impl reference` times that CPU port instead (Go is not buildable here: no toolchain, deps not vendored).
Launch: python bench.py --gpus N --steps K --warmup W   (N>1 under torch.distributed.run, one rank per GPU).
`--dump-outputs DIR` writes what the last timed step computed on rank 0 to DIR/<name>.npy, so that two builds can be compared
output for output (the inputs are seeded: the same arguments give the same batch).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "ChangeItems/sec on ClickBench-shaped 99-col batches (filter_rows + cast + ClickHouse native block + LZ4 frames)"
FALLBACK_HBM_GBS = 6650.0


TRAFFIC_PROFILE = "profiles/r2h_traffic.json"   # written by scripts/ncu_summary.py from the capture under profiles/
CACHE_DIR = tempfile.gettempdir()                  # generated inputs are cached here, never in the tree (which may be read-only)

# --dump-outputs: bytes kept per output; each byte is stored as one float32, so 50 MB in all. Larger outputs are cut into
# DUMP_CHUNK-byte chunks and a fixed seeded set of them is kept (the same chunks for the same output length).
DUMP_BYTES = 6 << 20
DUMP_CHUNK = 4096


def bench_config(args, ncols: int) -> dict:
    """The `config` object both arms print, key for key (the driver compares them)."""
    return {"workload": "clickbench_hits_99col filter_rows+cast+ch_native+lz4 (BASELINE configs[2])", "rows_per_step_per_gpu": min(args.rows, 1_000_000) if args.impl == "reference" else args.rows,
            "columns": ncols, "frame_bytes": args.frame_bytes, "batch_seed": "workload.SEED + rank", "filter": "watchid > K AND url ~ '://' with K set for 28 % kept rows on every rank's batch"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback 6.65 TB/s (B200_PROFILING.md)"


def make_batch(rows: int, seed: int):
    """Seeded synthetic batch; cached in the temporary directory so the two arms and every N reuse one generation."""
    from transferia_b200 import abi, workload
    schema = workload.hits_schema()
    cache = os.path.join(CACHE_DIR, f"tfgpu_hits_{rows}_{seed}.npz")
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            cols = []
            for i, c in enumerate(schema):
                t = abi.YT_NAME_TO_TF[c["type"]]
                g = lambda k: z[f"{i}_{k}"] if f"{i}_{k}" in z.files else None
                cols.append(abi.Column(t, g("values"), g("validity"), g("offsets"), g("heap"), g("aux")))
            return abi.Batch(rows, cols), schema
        except Exception:
            pass
    batch, schema = workload.make_hits_batch(rows, seed)
    try:
        arrs = {}
        for i, c in enumerate(batch.columns):
            for k in ("values", "validity", "offsets", "heap", "aux"):
                a = getattr(c, k)
                if a is not None:
                    arrs[f"{i}_{k}"] = a
        tmp = f"{cache}.{os.getpid()}.tmp.npz"
        np.savez(tmp, **arrs); os.replace(tmp, cache)          # atomic: several ranks may generate the same batch at once
    except Exception:
        pass
    return batch, schema


def byte_sample(data: bytes, budget: int) -> np.ndarray:
    """`data` as float32 byte values: all of it up to `budget` bytes, above that a seeded choice of whole DUMP_CHUNK-byte chunks."""
    a = np.frombuffer(data, dtype=np.uint8)
    if len(a) > budget:
        pick = np.sort(np.random.default_rng(0).choice(len(a) // DUMP_CHUNK, budget // DUMP_CHUNK, replace=False))
        a = a[(pick[:, None] * DUMP_CHUNK + np.arange(DUMP_CHUNK)).ravel()]
    return a.astype(np.float32)


def decode_frames(wire: bytes, raw_len: int):
    """ClickHouse compressed frames ([16 checksum][0x82][u32 block size + 9][u32 raw size][LZ4 block]) decoded with stock liblz4:
    (the bytes they carry, the number of frames). Raises on a frame that does not decode."""
    import ctypes as C
    import struct
    lz = C.CDLL("liblz4.so.1")
    out = C.create_string_buffer(max(1, raw_len)); pos = got = nf = 0
    while pos < len(wire):
        cs, rs = struct.unpack_from("<II", wire, pos + 17)
        if wire[pos + 16] != 0x82 or got + rs > raw_len:
            raise RuntimeError(f"frame {nf} at wire byte {pos}: bad header")
        n = lz.LZ4_decompress_safe(wire[pos + 25: pos + 16 + cs], C.c_void_p(C.addressof(out) + got), cs - 9, rs)
        if n != rs:
            raise RuntimeError(f"frame {nf} at wire byte {pos}: liblz4 returned {n} of {rs} bytes")
        pos += 16 + cs; got += rs; nf += 1
    return out.raw[:got], nf


def dump_outputs(eng, out_dir: str) -> None:
    """What the last tfgpu_push_encode_resident call computed, as its caller fetches it: counts.npy (rows out, native block bytes,
    frames, row errors; float64), raw_block.npy (the native block the frames compress) and wire_decoded.npy (the LZ4 frames decoded).
    The compressed bytes themselves are not written: the match finder's hash-table inserts race, so which of several valid matches
    a frame uses, and with it the compressed size, differs from run to run; what the frames decode to does not."""
    st = eng.resident_stats()
    raw = eng.resident_fetch(0, st["raw_bytes"])
    decoded, n_frames = decode_frames(eng.resident_fetch(1, st["wire_bytes"]), st["raw_bytes"])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "counts.npy"), np.array([st["rows_out"], st["raw_bytes"], n_frames, st["n_errors"]], dtype=np.float64))
    np.save(os.path.join(out_dir, "raw_block.npy"), byte_sample(raw, DUMP_BYTES))
    np.save(os.path.join(out_dir, "wire_decoded.npy"), byte_sample(decoded, DUMP_BYTES))


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled while the benchmark runs (NVML; nvidia-smi query as a fallback).
    Samples carry timestamps; the reported figures use the samples inside [mark_start, mark_end]."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index; self.stop_flag = False; self.samples = []; self.sm_max = None
        self.t0 = self.t1 = None; self.nv = None; self.h = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv; self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _sample(self):
        if self.nv is not None:
            nv = self.nv
            clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            return float(clk), {nm for bit, nm in self.REASONS.items() if r & bit}
        import subprocess
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        o = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip().split(",")
        self.sm_max = float(o[1])
        return float(o[0]), {nm for nm, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), o[2:]) if val.strip().lower().startswith("active")}

    def run(self):
        while not self.stop_flag:
            try:
                clk, rs = self._sample()
                self.samples.append((time.perf_counter(), clk, rs))
            except Exception:
                pass
            time.sleep(0.002 if self.nv is not None else 0.1)

    def mark_start(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def result(self):
        inside = [x for x in self.samples if self.t0 is not None and self.t0 <= x[0] <= (self.t1 or 1e30)]
        use = inside or self.samples[-3:]
        if not use:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unavailable"], "samples": 0}
        reasons = set().union(*[x[2] for x in use])
        return {"sm_mhz": float(np.median([x[1] for x in use])), "sm_max_mhz": self.sm_max, "reasons": sorted(reasons),
                "samples": len(inside)}


def cpu_port_rate(batch, schema, transformers, frame_bytes, budget_s: float, threads: int):
    """Rows/s of the oracle port run as `threads` independent sink pipelines (the reference's sharded-snapshot
    parallelism, pkg/worker/tasks/load_snapshot.go:917-1041), each over its own row slice, for >= budget_s."""
    from transferia_b200 import abi
    from oracle import pyoracle as po
    plan = po.build_plan("public", "hits", schema, transformers)
    n = batch.nrows
    per = max(1, min(n // threads, 100_000))
    slices = [batch.slice(i * per, (i + 1) * per) for i in range(threads)]
    done = [0] * threads
    t_end = [0.0] * threads
    t0 = time.perf_counter()

    def work(i):
        while True:
            po.push_encode(slices[i], plan, abi.TF_WIRE_CH_NATIVE_LZ4, frame_bytes, want_bytes=False)
            done[i] += per
            t_end[i] = time.perf_counter()
            if t_end[i] - t0 >= budget_s:
                break
    ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    el = max(t_end) - t0
    return sum(done) / el, sum(done), el


def host_paths(res: dict) -> None:
    """The host-only legs (no device involved): the transposer in front of every push of boxed items, and the regex_replace host step."""
    # SURVEY §8f-1: the host transpose ([]ChangeItem in row form -> columns) that sits in front of every push in a real transfer. The row
    # image of 200 k hits rows is made by the inverse (tfgpu_batch_to_rows) and timed through tfgpu_rows_to_batch: host-only C++ threads.
    try:
        import ctypes as C
        from transferia_b200 import rows as rws, workload
        nb_rows = 200_000
        hb, hschema = make_batch(nb_rows, workload.SEED)
        image, off = rws.batch_to_rows(hb)
        items = (rws.TfItem * nb_rows)(); offs = off.astype(np.uint64)
        for r_ in range(nb_rows):
            it = items[r_]; it.values_off = int(offs[r_]); it.n_values = len(hschema); it.old_keys_off = rws.NO_OLD_KEYS
        img = rws.RowsImage([], [("public", "hits", hschema)])
        vals = np.frombuffer(image, dtype=np.uint8).copy()
        img.struct.n_items = nb_rows; img.struct.items = C.cast(items, C.POINTER(rws.TfItem)); img.struct.values = vals.ctypes.data; img.struct.values_len = len(image)
        pool = rws.Columnar(); rates = {}
        for th in (1, 8, 16, 64):
            if th > (os.cpu_count() or 1):
                continue
            pool.rows_to_batch(img, threads=th)
            t0 = time.perf_counter(); k = 3
            for _ in range(k):
                pool.rows_to_batch(img, threads=th)
            rates[str(th)] = nb_rows * k / (time.perf_counter() - t0)
        pool.close()
        best = max(rates.values())
        res["host_transpose_rows_to_columns"] = {"rows_per_s": best, "ms": nb_rows / best * 1e3, "rows": nb_rows, "image_bytes_per_row": len(image) / nb_rows, "rows_per_s_by_threads": rates,
                                                 "note": "tfgpu_rows_to_batch over the row image of ClickBench-shaped items (99 boxed values per row): what a shim pays per batch before any push; CPU only"}
    except Exception as ex:
        res["host_transpose_error"] = str(ex)
    # SURVEY §8f-4: regex_replace_transformer runs on the host inside tfgpu_sink_push (Go's regexp as a Pike machine over the row image,
    # then the transpose): 200 k hits rows, the two URL-like columns rewritten.
    try:
        from transferia_b200 import sink as snk
        if "host_transpose_error" in res:
            raise RuntimeError("no row image")
        tr = [{"regex_replace_transformer": {"regexMatch": r"^(https?)://([^/]+)", "replaceRule": "$2 via $1", "columns": {"includeColumns": ["^url$", "^referer$"]}}}]
        s_ = snk.Sink(transformers=tr, record="counts")
        s_.push(img); s_.events.clear()
        t0 = time.perf_counter(); k = 3
        for _ in range(k):
            s_.push(img); s_.events.clear()
        dt = (time.perf_counter() - t0) / k
        s_.close()
        res["host_regex_replace_then_transpose"] = {"rows_per_s": nb_rows / dt, "ms": dt * 1e3, "rows": nb_rows,
                                                    "note": "tfgpu_sink_push without a device plan: the transposer, then two string columns through Regexp.ReplaceAll on the host workers (up to 16 threads); CPU only"}
    except Exception as ex:
        res["host_regex_error"] = str(ex)


def extra_paths(eng, args):
    """Secondary §8 paths, measured end to end through the public call with HOST bytes (not the headline metric):
    BASELINE configs[1] JSON lines -> parse -> mask_field -> ClickHouse JSONEachRow / native+LZ4, and the batch serializers."""
    import torch
    from transferia_b200 import abi, engine, workload
    sys.path.insert(0, ROOT)
    res = {}
    cache = os.path.join(CACHE_DIR, f"tf_json_lines_{args.json_lines}.bin")
    if os.path.exists(cache):
        text = open(cache, "rb").read(); fields = [dict(f) for f in workload.JSON_FIELDS]
    else:
        text, fields = workload.make_json_lines(args.json_lines)
        open(cache, "wb").write(text)
    opts = {"add_rest": True, "add_dedupe_keys": True, "partition": '{"partition":0,"topic":"events"}'}
    schema = engine.json_result_schema(fields, opts)
    trs = [{"mask_field": {"columns": ["user"], "maskFunctionHash": {"userDefinedSalt": "pepper"}}}]
    pid = eng.plan("", "events", schema, trs, {"type": "clickhouse"})
    n = text.count(b"\n")
    pinned = torch.frombuffer(bytearray(text), dtype=torch.uint8).pin_memory()      # the message bytes as a consumer would hold them: pinned
    for name, fmt in (("json_parse_mask_ch_jsoneachrow", abi.TF_WIRE_CH_JSONEACHROW), ("json_parse_mask_ch_native_lz4", abi.TF_WIRE_CH_NATIVE_LZ4)):
        for _ in range(2):
            r = eng.parse_json(pid, pinned, opts, None, wire_fmt=fmt, copy_bytes=False)
        torch.cuda.synchronize(); t0 = time.perf_counter(); k = 5
        for _ in range(k):
            r = eng.parse_json(pid, pinned, opts, None, wire_fmt=fmt, copy_bytes=False)
        torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / k
        eng.profile_enable(True); eng.parse_json(pid, text, opts, None, wire_fmt=fmt); prof = {kk["name"]: round(kk["ms"], 4) for kk in eng.profile_read()}; eng.profile_enable(False)
        res[name] = {"rows_per_s": n / dt, "lines": n, "input_MB": len(text) / 1e6, "ms": dt * 1e3, "rows_out": r.rows_out, "out_bytes": int(r.wire_len), "kernels_ms": prof,
                     "note": "wall clock around the public call with the message bytes in a pinned host buffer: H2D of the bytes and D2H of the wire bytes into the pinned landing buffer included"}
    # queue Debezium serializer on the ClickBench-shaped table (every column carries a pg original type: the production AddPg path)
    try:
        hb, hschema = make_batch(100_000, workload.SEED)
        hpid = eng.plan("public", "hits", hschema, [])
        dopts = {"source_type": "pg", "version": "2.1.4", "topic_prefix": "clickbench", "database": "db", "snapshot": True}
        rngm = np.random.default_rng(1)
        meta = {"id": rngm.integers(0, 2**31, hb.nrows).astype(np.uint32), "lsn": rngm.integers(0, 2**60, hb.nrows).astype(np.uint64),
                "commit_time": rngm.integers(16 * 10**17, 17 * 10**17, hb.nrows).astype(np.uint64)}
        hp = hb.pin()
        for _ in range(2):
            r = eng.emit_debezium(hpid, hp, dopts, meta, copy_bytes=False)
        torch.cuda.synchronize(); t0 = time.perf_counter(); k = 3
        for _ in range(k):
            r = eng.emit_debezium(hpid, hp, dopts, meta, copy_bytes=False)
        torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / k
        eng.profile_enable(True); eng.emit_debezium(hpid, hp, dopts, meta, copy_bytes=False); prof = {kk["name"]: round(kk["ms"], 4) for kk in eng.profile_read()}; eng.profile_enable(False)
        res["debezium_emit_pg_hits"] = {"rows_per_s": hb.nrows / dt, "rows": hb.nrows, "ms": dt * 1e3, "out_bytes": int(r.wire_len), "errors": len(r.errors), "kernels_ms": prof,
                                        "note": "tfgpu_emit_debezium over pinned host columns (99 pg-typed columns per row): key + value message per row, D2H of the messages included"}
        try:
            from oracle import pyoracle as po
            sl = hb.slice(0, 2000); sm = {kk: vv[:2000] for kk, vv in meta.items()}
            t0 = time.perf_counter(); po.debezium_emit(sl, po.build_plan("public", "hits", hschema, []), dopts, sm); dtc = time.perf_counter() - t0
            res["debezium_emit_pg_hits"]["cpu_port_rows_per_s_1core"] = 2000 / dtc
        except Exception as ex:
            res["debezium_emit_pg_hits"]["cpu_port_error"] = str(ex)
    except Exception as ex:
        res["debezium_emit_error"] = str(ex)
    # BASELINE configs[3]: Debezium CDC envelopes (12-field payload, schema-registry framed) -> parse -> filter_rows -> cast -> native block + LZ4
    try:
        dcache = os.path.join(CACHE_DIR, f"tf_dbz_{args.dbz_msgs}.bin")
        if os.path.exists(dcache + ".npy"):
            ddata = open(dcache, "rb").read(); dends = np.load(dcache + ".npy"); dschema_text, dtable = workload.debezium_schema_text(), ("public", "events")
        else:
            ddata, dends, dschema_text, dtable = workload.make_debezium_messages(args.dbz_msgs)
            open(dcache, "wb").write(ddata); np.save(dcache + ".npy", dends)
        dschema = engine.debezium_table_schema(dschema_text); dtrs = workload.debezium_transformers()
        dpid = eng.plan(dtable[0], dtable[1], dschema, dtrs, {"type": "clickhouse"})
        kw = dict(schema_registry=True, schema_id=7, wire_fmt=abi.TF_WIRE_CH_NATIVE_LZ4, copy_bytes=False)
        dpin = torch.frombuffer(bytearray(ddata), dtype=torch.uint8).pin_memory()        # the message bytes as a consumer would hold them: pinned
        for _ in range(2):
            r, _m = eng.parse_debezium(dpid, dpin, dends, dschema_text, **kw)
        torch.cuda.synchronize(); t0 = time.perf_counter(); k = 5
        for _ in range(k):
            r, _m = eng.parse_debezium(dpid, dpin, dends, dschema_text, **kw)
        torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / k
        eng.profile_enable(True); eng.parse_debezium(dpid, ddata, dends, dschema_text, **kw); prof = {kk["name"]: round(kk["ms"], 4) for kk in eng.profile_read()}; eng.profile_enable(False)
        kern_ms = sum(prof.values())
        res["debezium_parse_filter_cast"] = {"rows_per_s": len(dends) / dt, "messages": int(len(dends)), "input_MB": len(ddata) / 1e6, "ms": dt * 1e3, "rows_out": r.rows_out, "row_errors": len(r.errors),
                                             "out_bytes": int(r.wire_len), "kernels_ms": prof, "kernels_GBps_of_input": {n: round(len(ddata) / 1e6 / v, 1) for n, v in prof.items() if v > 0.02},
                                             "kernel_only_rows_per_s": len(dends) / (kern_ms / 1e3) if kern_ms else None,
                                             "note": "wall clock around tfgpu_parse_debezium with the message bytes in a pinned host buffer: H2D, the fused chain and D2H of the frames into the pinned landing buffer included"}
        try:
            from oracle import pyoracle as po
            ns = 4000; sd = ddata[: int(dends[ns - 1])]
            t0 = time.perf_counter(); b, kinds, *_ = po.debezium_parse(sd, dends[:ns].tolist(), dschema_text, use_sr=True, schema_id=7)
            po.push_encode(abi.Batch(b.nrows, b.columns, np.asarray(kinds, dtype=np.uint8)), po.build_plan(dtable[0], dtable[1], dschema, dtrs), abi.TF_WIRE_CH_NATIVE_LZ4, args.frame_bytes); dtc = time.perf_counter() - t0
            res["debezium_parse_filter_cast"]["cpu_port_rows_per_s_1core"] = ns / dtc
        except Exception as ex:
            res["debezium_parse_filter_cast"]["cpu_port_error"] = str(ex)
    except Exception as ex:
        res["debezium_parse_error"] = str(ex)
    # BASELINE configs[4]: hits-shaped CSV -> parse -> cast -> ClickHouse native block (+ LZ4)
    try:
        ccache = os.path.join(CACHE_DIR, f"tf_csv_{args.csv_rows}.bin")
        cb, cschema = make_batch(args.csv_rows, workload.SEED)
        cschema = [dict(c, path=str(i)) for i, c in enumerate(cschema)]
        if os.path.exists(ccache):
            ctext = open(ccache, "rb").read()
        else:
            ctext = workload.render_hits_csv(cb, cschema); open(ccache, "wb").write(ctext)
        cpid = eng.plan("public", "hits", cschema, [], {"type": "clickhouse"})
        cpin = torch.frombuffer(bytearray(ctext), dtype=torch.uint8).pin_memory()
        for _ in range(2):
            r, _c = eng.parse_csv(cpid, cpin, wire_fmt=abi.TF_WIRE_CH_NATIVE_LZ4, copy_bytes=False)
        torch.cuda.synchronize(); t0 = time.perf_counter(); k = 5
        for _ in range(k):
            r, _c = eng.parse_csv(cpid, cpin, wire_fmt=abi.TF_WIRE_CH_NATIVE_LZ4, copy_bytes=False)
        torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / k
        eng.profile_enable(True); eng.parse_csv(cpid, ctext, wire_fmt=abi.TF_WIRE_CH_NATIVE_LZ4); prof = {kk["name"]: round(kk["ms"], 4) for kk in eng.profile_read()}; eng.profile_enable(False)
        kern_ms = sum(prof.values())
        res["csv_parse_cast_native"] = {"rows_per_s": args.csv_rows / dt, "rows": args.csv_rows, "input_MB": len(ctext) / 1e6, "ms": dt * 1e3, "rows_out": r.rows_out, "out_bytes": int(r.wire_len), "kernels_ms": prof,
                                        "kernels_GBps_of_input": {n: round(len(ctext) / 1e6 / v, 1) for n, v in prof.items() if v > 0.02},
                                        "kernel_only_rows_per_s": args.csv_rows / (kern_ms / 1e3) if kern_ms else None,
                                        "note": "wall clock around tfgpu_parse_csv with the text in a pinned host buffer: H2D, tokenise + cast + native block + LZ4 frames, D2H into the pinned landing buffer included"}
        try:
            from oracle import pyoracle as po
            cut = ctext.rfind(b"\n", 0, len(ctext) // 25) + 1; sample = ctext[:cut]
            t0 = time.perf_counter(); b, _e, _l, _c = po.csv_parse(sample, cschema); po.push_encode(b, po.build_plan("public", "hits", cschema, []), abi.TF_WIRE_CH_NATIVE_LZ4, args.frame_bytes); dtc = time.perf_counter() - t0
            res["csv_parse_cast_native"]["cpu_port_rows_per_s_1core"] = sample.count(b"\n") / dtc
        except Exception as ex:
            res["csv_parse_cast_native"]["cpu_port_error"] = str(ex)
    except Exception as ex:
        res["csv_parse_error"] = str(ex)
    host_paths(res)
    try:
        from oracle import pyoracle as po
        sample = text[: text.rfind(b"\n", 0, len(text) // 20) + 1]
        t0 = time.perf_counter(); b, _, _ = po.json_parse(sample, fields, opts); po.push_encode(b, po.build_plan("", "events", schema, trs), abi.TF_WIRE_CH_JSONEACHROW); dt = time.perf_counter() - t0
        res["json_parse_mask_ch_jsoneachrow"]["cpu_port_rows_per_s_1core"] = sample.count(b"\n") / dt
    except Exception as ex:  # the oracle is optional here
        res["cpu_port_error"] = str(ex)
    return res


def run_reference(args):
    """--impl reference: the reference's CPU algorithm for this path (oracle port) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from transferia_b200 import workload
    cores = os.cpu_count() or 1
    rows = min(args.rows, 1_000_000)
    batch, schema = make_batch(rows, workload.SEED)
    k = workload.headline_threshold(batch, schema)
    trs = workload.headline_transformers_watchid(k)
    per_step_budget = 2.0
    for _ in range(args.warmup):
        cpu_port_rate(batch, schema, trs, args.frame_bytes, 0.5, cores)
    tot_rows = 0; tot_t = 0.0
    for _ in range(args.steps):
        _, r, t = cpu_port_rate(batch, schema, trs, args.frame_bytes, per_step_budget, cores)
        tot_rows += r; tot_t += t
    v = tot_rows / tot_t
    sample = f"{cores} pipelines, each over its own {min(rows // cores, 100000)}-row slice of the {rows}-row batch, >= {per_step_budget}s per step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": bench_config(args, len(schema)),
        "note": "CPU restatement (C++ oracle port), not Go: no Go toolchain / module cache in this image",
        "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def bind_to_gpu_numa_node(local):
    """One process per GPU, bound to the CPUs of the NUMA node the GPU hangs off (its pinned host buffers are then allocated there and the
    DMA does not cross the socket interconnect). Returns the node, or None when the topology cannot be read."""
    try:
        node = None
        try:                                                    # the CUDA device of this rank (honours CUDA_VISIBLE_DEVICES, unlike an NVML index)
            import torch
            pr = torch.cuda.get_device_properties(local)
            node = int(open("/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).read())
        except Exception:
            import pynvml
            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
            bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
            if len(bus.split(":")[0]) == 8:
                bus = bus[4:]                                   # sysfs uses a 4-digit PCI domain
            node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-"); cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--frame-bytes", type=int, default=15360)
    ap.add_argument("--impl", default="tfgpu")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary paths (JSON-lines parse, serializers)")
    ap.add_argument("--json-lines", type=int, default=400_000)
    ap.add_argument("--dbz-msgs", type=int, default=200_000, help="messages of the Debezium leg (BASELINE configs[3])")
    ap.add_argument("--csv-rows", type=int, default=100_000, help="rows of the CSV leg (BASELINE configs[4])")
    ap.add_argument("--host-layout", default="narrow", choices=["narrow", "offsets"], help="end-to-end leg: var-width columns as uint8 / uint16 lengths (narrow) or uint32 offsets")
    ap.add_argument("--numa-bind", type=int, default=1, help="bind the process to the CPUs of its GPU's NUMA node before allocating pinned memory (0: leave the affinity alone)")
    ap.add_argument("--host-buffers", default="arena", choices=["arena", "separate"], help="end-to-end leg: the pinned host batch as one arena (one DMA) or one pinned buffer per column array")
    ap.add_argument("--e2e-mode", default="auto", choices=["auto", "one-phase", "two-phase"], help="end-to-end leg: tfgpu_push_encode (one-phase), tfgpu_push_encode_selective (two-phase), or both and report the faster (auto)")
    ap.add_argument("--gather-threads", type=int, default=0, help="host threads of the two-phase gather per pipeline (0: min(32, cores / pipelines / ranks))")
    ap.add_argument("--e2e-pipelines", type=int, default=4, help="host threads (one engine handle each) pushing batches concurrently in the end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the device path; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from transferia_b200 import abi, engine, workload

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if args.numa_bind else None      # before any pinned allocation: first touch places the pages
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = f"cuda:{local}"

    # weak scaling: every rank pushes its OWN seeded batch (seed + rank: other values, dictionaries and therefore a slightly different
    # selectivity / compressibility per GPU, as independent table parts have); no data-path collective (SURVEY §8e)
    batch, schema = make_batch(args.rows, workload.SEED + rank)
    k = workload.headline_threshold(batch, schema)              # the same selectivity (0.28) on every rank's own batch
    trs = workload.headline_transformers_watchid(k)
    eng = engine.Engine(local, args.frame_bytes)
    stream = torch.cuda.Stream()          # a real (non-default) stream: events below and every kernel share it
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    pid = eng.plan("public", "hits", schema, trs, {"type": "clickhouse"})
    dbatch = batch.to_device(dev)
    # narrow: uint8 / uint16 lengths instead of uint32 offsets (TF_COL_LENS8 / 16); one pinned arena laid out like the device staging (a single DMA per batch)
    hb0 = batch.narrow() if args.host_layout == "narrow" else batch
    hbatch = hb0.pin() if args.host_buffers == "separate" else hb0.pin_arena()
    in_bytes = batch.input_bytes()
    h2d_bytes = hbatch.input_bytes()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-only (resident) ----
    sampler = ClockSampler(local); sampler.start()
    for _ in range(args.warmup):
        eng.push_encode_resident(pid, dbatch, abi.TF_WIRE_CH_NATIVE_LZ4)
    torch.cuda.synchronize()
    st = eng.resident_stats()
    eng.profile_enable(True)
    barrier()
    sampler.mark_start()
    l0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = {}
    ev0.record()
    for _ in range(args.steps):
        eng.push_encode_resident(pid, dbatch, abi.TF_WIRE_CH_NATIVE_LZ4)
        # per-kernel events of this step are read after the loop for the last step only; to average over the
        # timed region without syncing inside it, the engine keeps one event pair per kernel per call and we
        # read them once per step boundary below (the read syncs the stream, so do it outside timing)
    eng.resident_stats()      # orders the stream after the last batch's checksum / gather tail (side streams): the K steps are complete
    ev1.record()
    torch.cuda.synchronize()
    sampler.mark_end()
    launches = eng.launch_count() - l0
    ms_total = ev0.elapsed_time(ev1)
    for kk in eng.profile_read():        # events of the LAST timed step
        kernel_ms[kk["name"]] = kernel_ms.get(kk["name"], 0.0) + kk["ms"]
    if args.dump_outputs and rank == 0:   # before any further call replaces the last timed step's outputs
        dump_outputs(eng, args.dump_outputs)
    # average the dominant kernel over a few more (untimed) steps for a stable duration
    extra = 5
    acc = {}
    for _ in range(extra):
        eng.push_encode_resident(pid, dbatch, abi.TF_WIRE_CH_NATIVE_LZ4)
        for kk in eng.profile_read():
            acc[kk["name"]] = acc.get(kk["name"], 0.0) + kk["ms"]
    kernel_avg = {n: (acc.get(n, 0.0) + kernel_ms.get(n, 0.0)) / (extra + 1) for n in set(acc) | set(kernel_ms)}
    eng.profile_enable(False)
    barrier()
    sampler.stop_flag = True; sampler.join(timeout=2)
    if os.environ.get("TF_BENCH_DEBUG"):
        print(f"[rank {rank}] resident region {ms_total:.3f} ms over {args.steps} steps; kernels {sorted(kernel_avg.items(), key=lambda kv: -kv[1])[:4]}", file=sys.stderr, flush=True)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * args.rows * args.steps / (ms_max / 1e3)

    # what stock liblz4 (LZ4_compress_default, the class of compressor the reference's driver uses) makes of the same block cut into the
    # same frames: the yardstick for `lz4_ratio` (a CPU call on a sample of the frames, outside every timed region)
    stock_ratio = None
    if rank == 0:
        try:
            import ctypes as C
            lz = C.CDLL("liblz4.so.1")
            eng.push_encode_resident(pid, dbatch, abi.TF_WIRE_CH_NATIVE_LZ4); st2 = eng.resident_stats()
            raw = eng.resident_fetch(0, st2["raw_bytes"])
            F = args.frame_bytes; nfr = (len(raw) + F - 1) // F; pick = range(0, nfr, max(1, nfr // 400))
            dst = C.create_string_buffer(F + F // 255 + 64); tot_in = tot_out = 0
            for f in pick:
                chunk = raw[f * F:(f + 1) * F]
                tot_out += lz.LZ4_compress_default(chunk, dst, len(chunk), len(dst)) + 25; tot_in += len(chunk)
            stock_ratio = tot_in / tot_out
        except Exception:
            stock_ratio = None

    # ---- end to end through the public call, host buffers ----
    # Each call is synchronous: H2D of every column, the chain, D2H of the wire bytes. The reference keeps several sink
    # pipelines busy at once (one flush in flight while the next batch collects, bufferer.go:225-242; N parallel sinkers per
    # snapshot, load_snapshot.go:986): `--e2e-pipelines P` host threads, each with its own engine handle on this GPU, push
    # alternate batches, so one pipeline's copies overlap another's kernels. P = 1 is the strictly serial call sequence.
    P = max(1, args.e2e_pipelines)
    engs = [eng]
    for _ in range(P - 1):
        try:
            engs.append(engine.Engine(local, args.frame_bytes))
        except Exception as ex:      # not enough memory for another set of arenas: fewer pipelines, reported as such
            print(f"bench: extra pipeline not created ({ex}); continuing with {len(engs)}", file=sys.stderr)
            break
    P = len(engs)
    e2e_steps = ((max(3, min(args.steps, 10)) + P - 1) // P) * P
    pids = [pid] + [e2.plan("public", "hits", schema, trs, {"type": "clickhouse"}) for e2 in engs[1:]]
    last = [None] * P
    cores = os.cpu_count() or 1
    gather_threads = args.gather_threads if args.gather_threads > 0 else max(2, min(32, cores // (2 * P * world)))     # physical cores (2 hardware threads each) shared by the pipelines of every rank

    def run_e2e(selective):
        """K public calls per pipeline over the pinned host batch: one phase (every column crosses PCIe) or two phases
        (tfgpu_push_encode_selective: predicate columns, keep flags back, host gather of the kept rows, then only those)."""
        def pipeline(i, nsteps):
            torch.cuda.set_device(local)
            for _ in range(nsteps):
                last[i] = engs[i].push_encode(pids[i], hbatch, abi.TF_WIRE_CH_NATIVE_LZ4, copy_bytes=False, selective=gather_threads if selective else None)
        ths = [threading.Thread(target=pipeline, args=(i, 2)) for i in range(P)]
        [t_.start() for t_ in ths]; [t_.join() for t_ in ths]
        barrier()
        h0 = sum(e2.h2d_bytes() for e2 in engs)
        ths = [threading.Thread(target=pipeline, args=(i, e2e_steps // P)) for i in range(P)]
        t0 = time.perf_counter()
        [t_.start() for t_ in ths]; [t_.join() for t_ in ths]
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3          # wall clock: every call has returned, its result bytes are in host memory
        h2d = (sum(e2.h2d_bytes() for e2 in engs) - h0) // e2e_steps
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return world * args.rows * e2e_steps / (float(tt.item()) / 1e3), int(h2d), int(last[0].wire_len)

    modes = {"one-phase": [False], "two-phase": [True], "auto": [False, True]}[args.e2e_mode]
    legs = {("two-phase" if m else "one-phase"): run_e2e(m) for m in modes}
    best = max(legs, key=lambda k_: legs[k_][0])
    e2e_value, h2d_bytes, d2h = legs[best]
    r = last[0]
    for e2 in engs[1:]:
        e2.close()

    if rank == 0:
        peak, peak_src = load_peaks()
        lz_ms = kernel_avg.get("k_lz4_frames", 0.0)
        lz_bytes = st["raw_bytes"] + (st["wire_bytes"] - 25 * ((st["raw_bytes"] + args.frame_bytes - 1) // args.frame_bytes))
        achieved = lz_bytes / (lz_ms / 1e3) / 1e9 if lz_ms else 0.0
        step_ms = sum(kernel_avg.values())
        traffic, traffic_src = None, None      # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
        try:
            tj = json.load(open(os.path.join(ROOT, TRAFFIC_PROFILE)))["k_lz4_frames"]
            traffic = int(tj["dram_bytes_read"] + tj["dram_bytes_write"]); traffic_src = TRAFFIC_PROFILE
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": bench_config(args, len(schema)),
            "workload_stats": {"selectivity": st["rows_out"] / args.rows, "lz4_ratio": st["raw_bytes"] / max(1, st["wire_bytes"]),
                               "lz4_ratio_blocks_only": st["raw_bytes"] / max(1, st["wire_bytes"] - 25 * ((st["raw_bytes"] + args.frame_bytes - 1) // args.frame_bytes)),
                               "lz4_ratio_stock_liblz4_same_frames": stock_ratio,
                               "input_bytes_per_row": in_bytes / args.rows, "block_bytes_per_kept_row": st["raw_bytes"] / max(1, st["rows_out"]),
                               "l2": "inputs larger than L2 (%.0f MB per step > 126 MB)" % (in_bytes / 1e6),
                               "parallelism": f"dp{world} (one batch stream per GPU, its own seeded batch on every rank, no collective)", "rank": 0},
            "clocks": sampler.result(),
            "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": d2h, "host_layout": args.host_layout, "host_buffers": args.host_buffers, "numa_node": numa,
                    "mode": best, "gather_threads": gather_threads if best == "two-phase" else 0,
                    "all_modes": {k_: {"value": v_[0], "h2d_bytes_per_step": v_[1]} for k_, v_ in legs.items()},
                    "steps": e2e_steps, "pipelines": P, "timing": "host wall clock over synchronous calls (tfgpu_push_encode / tfgpu_push_encode_selective over pinned host columns; H2D counted by the engine)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_lz4_frames", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(lz_bytes), "kernel_ms": lz_ms,
                         "kernel_share_of_step": lz_ms / step_ms if step_ms else None,
                         "kernel_share_basis": "sum of the per-kernel CUDA-event times (as in the serialised ncu launch list); k_frame_seal overlaps the next step on a side stream, so that sum exceeds ms_per_step",
                         "all_kernels_ms": {n: round(v, 4) for n, v in sorted(kernel_avg.items())}},
        }
        if world == 1 and not args.no_extra:
            out["other_paths"] = extra_paths(eng, args)
        if world == 1:
            cores = os.cpu_count() or 1
            try:
                os.sched_setaffinity(0, range(cores))      # the CPU baseline uses every host core, not just the GPU's NUMA node
            except OSError:
                pass
            v, rows_done, el = cpu_port_rate(batch, schema, trs, args.frame_bytes, args.cpu_budget, cores)
            out["cpu_baseline"] = {"value": v, "unit": "rows/s", "cores": cores, "kind": "port",
                                   "sample": f"{cores} pipelines, each over its own {min(args.rows // cores, 100000)}-row slice of the same batch, for {el:.1f}s ({rows_done} rows); C++ oracle port of the Go row loop, not Go"}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


if __name__ == "__main__":
    main()
