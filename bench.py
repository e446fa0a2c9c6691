#!/usr/bin/env python
"""bench.py — merged rows/s of the LSM merge hot path on B200 (BASELINE.json metric).

One "step" = one pass of the hot path over one bucket of synthetic sorted runs:
  --source parquet (default for c3):  Parquet file bytes in HBM -> column-chunk decode (one launch set for the
      section) -> sampled partition -> plan -> scan -> emit.  The 16 run files are written once, outside the timed
      region, by the device encoder (PLAIN data pages V1, 20 000-row pages, 400 000-row row groups, uncompressed).
  --source columns: the merge alone over pre-decoded columns resident in HBM (round 1's measurement; reported for
      c3 under "extra" as well).

Workloads (BASELINE.json configs, SURVEY.md §8d):
  c3 (default, the configuration the metric is quoted on): 16 runs x 6.25 M rows = 100 M rows, partial-update merge
      engine, 50-column wide row (pk + 20 BIGINT + 15 DOUBLE + 14 VARCHAR(8..24)), every non-pk cell NULL with p = 0.5
  c3agg: same rows, merge-engine aggregation (sum over the numeric columns: ordered left fold, bit-exact)
  c2: 8 runs x 12.5 M rows = 100 M rows, deduplicate, BIGINT pk + 10 BIGINT columns
  c1: 2 runs x 500 K rows, deduplicate, BIGINT pk + BIGINT value
  c4: one bucket of a full compaction rewrite (32 runs, VARCHAR(16) key, deletes, drop-delete, re-encode)

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c3agg|c2|c1|c4] [--rows R] [--source ...]
    python bench.py --impl reference ...     # the reference algorithm on the host cores (CPU)
    python bench.py --dump-outputs DIR ...   # also write a seeded sample of the last timed step's merged batch

`value`     whole-job merged (= input) rows/s with the inputs (file bytes / columns) already resident in HBM.
`e2e`       same metric through the public reader API with HOST buffers: every step copies the Parquet files
            host->device (pinned memory), decodes, merges, and copies the merged batch device->host; consecutive
            steps are pipelined (the D2H of bucket i overlaps the H2D of bucket i+1, like consecutive splits of a scan).
`roofline`  achieved HBM GB/s of the dominant kernel (emit) on the algorithmic bytes N_in*B + N_out*B (DESIGN.md),
            `roofline_decode` the same for the decode stage on encoded page bytes + decoded bytes, both against
            MEASURED_PEAKS.json.
`parity_sample`  a key range of the full-size result compared bit-for-bit with the CPU oracle.
`cpu_baseline`  the oracle (C restatement of LoserTree + MergeFunction) timed on this box's host cores.
Multi-GPU: one process per GPU (torchrun); buckets are independent, so every rank merges its own bucket and there
is no data-path collective ("weak" scaling).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import queue
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# decoded runs (48 GB per step on c3) are recycled through the library's buffer cache instead of the driver allocator
os.environ.setdefault("PG_RUN_CACHE_BYTES", str(150 << 30))

import numpy as np  # noqa: E402

WORKLOADS = {
    "c3": dict(n_runs=16, rows=100_000_000, engine="partial-update", null_prob=0.5,
               desc="16-run partial-update, 50-col wide row (pk+20 i64+15 f64+14 varchar), 100M rows"),
    # SURVEY §8d "C3-agg": same rows as C3, merge-engine aggregation: the 15 doubles and 20 bigints use `sum`
    # (ordered left fold, bit-exact), the strings last_non_null_value
    "c3agg": dict(n_runs=16, rows=100_000_000, engine="aggregate", null_prob=0.5,
                  desc="16-run aggregation (sum over 20 i64 + 15 f64, last_non_null_value over 14 varchar), 50-col wide "
                       "row, 100M rows"),
    "c2": dict(n_runs=8, rows=100_000_000, engine="deduplicate", null_prob=0.0,
               desc="8-run deduplicate, int64 pk + 10 int64 cols, 100M rows"),
    "c1": dict(n_runs=2, rows=1_000_000, engine="deduplicate", null_prob=0.0,
               desc="2-run deduplicate, int64 pk + int64 val, 1M rows"),
    # one bucket of the full-compaction config (SURVEY §8d C4): string key, deletes, drop-delete, then the
    # merged batch is re-encoded to Parquet on the device (reported under "rewrite")
    "c4": dict(n_runs=32, rows=16_000_000, engine="deduplicate", null_prob=0.5, delete_prob=0.05, drop_delete=True,
               desc="one bucket of a full compaction rewrite: 32 runs x 500K rows, varchar(16) pk + 4 i64 + 2 f64 + "
                    "2 i32 + 3 varchar, 5% deletes, drop-delete, output re-encoded to Parquet"),
}
PARQUET_PAGE_ROWS = 20_000          # parquet-mr's page row limit (RowDataParquetBuilder.java:63-99 pulls the defaults)
PARQUET_GROUP_ROWS = 400_000        # ~128 MiB row groups at c3's ~310 encoded bytes per row


def schema_c4():
    from paimon_b200.types import DataField, KeyValueSchema, RowType
    fields = [DataField("pk", "VARCHAR(16)", False)]
    fields += [DataField(f"i{i}", "BIGINT", True) for i in range(4)]
    fields += [DataField(f"d{i}", "DOUBLE", True) for i in range(2)]
    fields += [DataField(f"n{i}", "INT", True) for i in range(2)]
    fields += [DataField(f"s{i}", "VARCHAR(64)", True) for i in range(3)]
    return KeyValueSchema.of(RowType(tuple(fields)), ["pk"])


def make_schema(workload):
    from paimon_b200 import datagen
    return {"c1": datagen.schema_c1, "c2": datagen.schema_c2, "c3": datagen.schema_c3, "c3agg": datagen.schema_c3,
            "c4": schema_c4}[workload]()


def make_spec(workload, schema):
    from paimon_b200.merge_function import (AggregateMergeFunction, DeduplicateMergeFunction,
                                            PartialUpdateMergeFunction)
    if WORKLOADS[workload]["engine"] == "aggregate":
        opts = {f"fields.{f.name}.aggregate-function": "sum" for f in schema.value_type.fields
                if f.name != "pk" and f.physical.name in ("INT64", "DOUBLE")}
        return AggregateMergeFunction.factory(opts, schema.value_type, ["pk"]).create()
    if WORKLOADS[workload]["engine"] == "partial-update":
        return PartialUpdateMergeFunction.factory({}, schema.value_type, ["pk"]).create()
    spec = DeduplicateMergeFunction.factory().create()
    return spec.with_drop_delete() if WORKLOADS[workload].get("drop_delete") else spec


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's threads (and, by first touch, its page-locked buffers) to the CPUs of the NUMA node its GPU
    hangs off: the end-to-end leg moves tens of GB per step between host DRAM and the device."""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={local_rank}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not out:
            return None
        dom, rest = out.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception:
        return None


# ------------------------------------------------------------------ device-side synthetic runs

def _splitmix64(x):
    x = x + (-7046029254386353131)                       # 0x9E3779B97F4A7C15 as int64
    x = (x ^ ((x >> 30) & ((1 << 34) - 1))) * (-4658895280553007687)   # 0xBF58476D1CE4E5B9
    x = (x ^ ((x >> 27) & ((1 << 37) - 1))) * (-7723592293110705685)   # 0x94D049BB133111EB
    return x ^ ((x >> 31) & ((1 << 33) - 1))


def _hex_keys(keys, dev):
    """int64 keys -> 16-character lower-case hex strings (big endian: string order == integer order)."""
    import torch
    sh = torch.arange(60, -4, -4, device=dev, dtype=torch.int64)
    nib = ((keys[:, None] >> sh) & 15).to(torch.uint8)
    data = torch.where(nib < 10, nib + 48, nib + 87).flatten()
    data = torch.cat([data, torch.zeros(16, device=dev, dtype=torch.uint8)]).contiguous()
    offs = (torch.arange(keys.numel() + 1, device=dev, dtype=torch.int64) * 16).to(torch.int32).contiguous()
    return data, offs


def gen_device_run(schema, run_index, n, key_space, null_prob, seed, dev, delete_prob=0.0):
    """One sorted run generated directly in HBM.  Returns (columns, keepalive tensors, key tensor, bytes, kinds)."""
    import torch
    from paimon_b200.sort_merge_reader import DeviceColumn
    from paimon_b200.types import PhysicalType
    g = torch.Generator(device=dev)
    g.manual_seed(seed * 1000003 + run_index)
    keys = torch.randperm(key_space, device=dev, generator=g)[:n].sort().values.contiguous()
    keep = [keys]
    cols = []
    string_key = schema.key_type.fields[0].physical == PhysicalType.STRING
    if string_key:
        kdata, koffs = _hex_keys(keys, dev)
        keep += [kdata, koffs]
        key_col = DeviceColumn(kdata.data_ptr(), koffs.data_ptr())
        key_bytes = n * 16 + 4 * (n + 1)
    else:
        key_col = DeviceColumn(keys.data_ptr())
        key_bytes = n * 8
    for _ in schema.key_type.fields:
        cols.append(key_col)
    seq = (torch.arange(n, device=dev, dtype=torch.int64) + (run_index << 32)).contiguous()
    kind = torch.zeros(n, device=dev, dtype=torch.int8)
    if delete_prob > 0:
        kind[torch.rand(n, device=dev, generator=g) < delete_prob] = 3
    keep += [seq, kind]
    cols += [DeviceColumn(seq.data_ptr()), DeviceColumn(kind.data_ptr())]
    nbytes = key_bytes + seq.numel() * 8 + kind.numel()
    pk_names = {f.name[len("_KEY_"):] for f in schema.key_type.fields}
    for ci, f in enumerate(schema.value_type.fields):
        t = f.physical
        if f.name in pk_names:
            cols.append(key_col)
            nbytes += key_bytes
            continue
        h = _splitmix64(keys ^ ((run_index + 1) * 0x100 + ci << 40))
        valid_ptr = 0
        bits = None
        if f.nullable and null_prob > 0:
            assert null_prob == 0.5, "device generator draws validity bits with p = 0.5"
            vbytes = torch.randint(0, 256, ((n + 7) // 8 + 8,), device=dev, dtype=torch.uint8, generator=g)
            keep.append(vbytes)
            valid_ptr = vbytes.data_ptr()
            nbytes += (n + 7) // 8
            if t in (PhysicalType.STRING, PhysicalType.BINARY):
                sh = torch.arange(8, device=dev, dtype=torch.uint8)
                bits = ((vbytes[:, None] >> sh) & 1).flatten()[:n].to(torch.int64)
        if t == PhysicalType.INT64:
            keep.append(h)
            cols.append(DeviceColumn(h.data_ptr(), 0, valid_ptr))
            nbytes += n * 8
        elif t == PhysicalType.INT32:
            v = (h & 0x7fffffff).to(torch.int32).contiguous()
            keep.append(v)
            cols.append(DeviceColumn(v.data_ptr(), 0, valid_ptr))
            nbytes += n * 4
        elif t == PhysicalType.DOUBLE:
            d = ((h >> 11) & ((1 << 53) - 1)).to(torch.float64) * (2000.0 / (1 << 53)) - 1000.0
            keep.append(d)
            cols.append(DeviceColumn(d.data_ptr(), 0, valid_ptr))
            nbytes += n * 8
        elif t in (PhysicalType.STRING, PhysicalType.BINARY):
            lens = 8 + ((h >> 3) & 0xffff) % 17                       # U[8, 24]
            if bits is not None:
                lens = lens * bits                                     # NULL cells carry no payload
            offs = torch.zeros(n + 1, device=dev, dtype=torch.int64)
            torch.cumsum(lens, 0, out=offs[1:])
            total = int(offs[-1].item())
            offs32 = offs.to(torch.int32)
            data = torch.randint(48, 112, (max(total, 1) + 16,), device=dev, dtype=torch.uint8, generator=g)
            keep += [offs32, data]
            cols.append(DeviceColumn(data.data_ptr(), offs32.data_ptr(), valid_ptr))
            nbytes += total + 4 * (n + 1)
            del lens, offs, bits
        else:
            raise ValueError(f"bench generator: unsupported type {t}")
    return cols, keep, keys, nbytes, kind


def device_runs(workload, schema, rows, dev, seed):
    import torch
    from paimon_b200.sort_merge_reader import SortedRunReader
    w = WORKLOADS[workload]
    n_runs = w["n_runs"]
    per_run = rows // n_runs
    key_space = max(rows // 2, per_run)
    readers, all_keys, all_kinds, in_bytes = [], [], [], 0
    for r in range(n_runs):
        cols, keep, keys, nb, kind = gen_device_run(schema, r, per_run, key_space, w["null_prob"], seed, dev,
                                                    w.get("delete_prob", 0.0))
        readers.append(SortedRunReader.from_device(schema, per_run, cols, keepalive=keep))
        all_keys.append(keys)
        all_kinds.append(kind)
        in_bytes += nb
    torch.cuda.synchronize()
    return readers, all_keys, in_bytes, all_kinds


def device_parquet_files(workload, schema, rows, dev, seed, lib):
    """The bucket's runs as Parquet files whose bytes sit in HBM: every run is generated on the device, encoded by
    pg_parquet_encode (PLAIN, data page V1) and dropped; the file images stay.  Returns (encoded-file handles,
    [(device pointer, size)], key tensors, kind tensors)."""
    import torch
    from paimon_b200 import _native as N
    from paimon_b200.compact_rewriter import file_column_names
    from paimon_b200.sort_merge_reader import SortedRunReader, _SchemaHandle
    w = WORKLOADS[workload]
    n_runs = w["n_runs"]
    per_run = rows // n_runs
    key_space = max(rows // 2, per_run)
    names = file_column_names(schema)
    arr = (C.c_char_p * len(names))(*[nm.encode() for nm in names])
    sh = _SchemaHandle(schema, dev.index or 0)
    handles, images, all_keys, all_kinds = [], [], [], []
    try:
        for r in range(n_runs):
            cols, keep, keys, _, kind = gen_device_run(schema, r, per_run, key_space, w["null_prob"], seed, dev,
                                                       w.get("delete_prob", 0.0))
            rd = SortedRunReader.from_device(schema, per_run, cols, keepalive=keep)
            try:
                fh = C.c_uint64(0)
                opts = N.PgParquetWriteOptions(PARQUET_GROUP_ROWS, PARQUET_PAGE_ROWS)
                N.check(lib.pg_parquet_encode(rd._open(sh.handle), arr, 0, -1, C.byref(opts), C.byref(fh)))
                ptr, size = C.c_void_p(0), C.c_int64(0)
                N.check(lib.pg_parquet_file_device_image(fh.value, C.byref(ptr), C.byref(size)))
                handles.append(fh.value)
                images.append((ptr.value, size.value))
            finally:
                rd.close()
            all_keys.append(keys)
            all_kinds.append(kind)
            del cols, keep, rd
            torch.cuda.empty_cache()
    finally:
        sh.close()
    torch.cuda.synchronize()
    return handles, images, all_keys, all_kinds


# ------------------------------------------------------------------ C5: lineitem-shaped Parquet decode + merge

def schema_c5():
    """SURVEY §8d C5: pk (l_orderkey BIGINT, l_linenumber INT), 16 columns."""
    from paimon_b200.types import DataField, KeyValueSchema, RowType
    fields = [DataField("l_orderkey", "BIGINT", False), DataField("l_linenumber", "INT", False),
              DataField("l_partkey", "BIGINT", True), DataField("l_suppkey", "BIGINT", True),
              DataField("l_quantity", "DECIMAL(15,2)", True), DataField("l_extendedprice", "DECIMAL(15,2)", True),
              DataField("l_discount", "DECIMAL(15,2)", True), DataField("l_tax", "DECIMAL(15,2)", True),
              DataField("l_returnflag", "CHAR(1)", True), DataField("l_linestatus", "CHAR(1)", True),
              DataField("l_shipdate", "DATE", True), DataField("l_commitdate", "DATE", True),
              DataField("l_receiptdate", "DATE", True), DataField("l_shipinstruct", "CHAR(25)", True),
              DataField("l_shipmode", "CHAR(10)", True), DataField("l_comment", "VARCHAR(44)", True)]
    return KeyValueSchema.of(RowType(tuple(fields)), ["l_orderkey", "l_linenumber"])


def c5_bucket(schema, codec, seed=5):
    """One C5 bucket as parquet-mr-style files written by pyarrow on the host (dictionary on with parquet-mr's 1 MiB
    dictionary page limit, data page V1, ~128 MiB row groups; DECIMAL(15,2) / DATE in their physical INT64 / INT32
    form): 1 base run (83.3 %) + 4 update runs whose keys are resampled from the base.  parquet-mr closes a page at
    1 MiB OR 20 000 rows (parquet.page.row.count.limit, RowDataParquetBuilder.java:63-99 keeps the defaults), pyarrow
    only knows a byte limit: 160 KiB pages give the 20 000-row pages an 8-byte column gets from parquet-mr.
    Returns ([(file bytes, run)], rows in, expected columns)."""
    import pyarrow as pa
    import pyarrow.parquet as pq
    rng = np.random.default_rng(seed)
    total = 1_000_000_000 // 64
    n_base = int(total * 5 / 6)
    n_upd = (total - n_base) // 4
    names = [f.name for f in schema.file_fields()]
    flags = [np.array([b"A", b"N", b"R"]), np.array([b"F", b"O"])]
    instr = np.array([b"DELIVER IN PERSON", b"COLLECT COD", b"NONE", b"TAKE BACK RETURN"])
    modes = np.array([b"REG AIR", b"AIR", b"RAIL", b"SHIP", b"TRUCK", b"MAIL", b"FOB"])

    def run_table(idx, seq0):
        n = len(idx)
        ok_, ln_ = pa.array(idx // 4), pa.array((idx % 4 + 1).astype(np.int32))
        # (a Paimon value row carries the primary-key fields too: _KEY_* copies + the table's own columns)
        cols = [ok_, ln_, pa.array(seq0 + np.arange(n, dtype=np.int64)), pa.array(np.zeros(n, np.int8)), ok_, ln_]
        part = rng.integers(1, 20_000_000, n)
        cols += [pa.array(part), pa.array(rng.integers(1, 1_000_000, n))]
        cols += [pa.array(rng.integers(100, 5_000_000, n)) for _ in range(4)]
        cols += [pa.array(flags[0][rng.integers(0, 3, n)]).cast(pa.string()), pa.array(flags[1][rng.integers(0, 2, n)]).cast(pa.string())]
        ship = rng.integers(8000, 10600, n).astype(np.int32)
        cols += [pa.array(ship), pa.array(ship + 30), pa.array(ship + 45)]
        cols += [pa.array(instr[rng.integers(0, 4, n)]).cast(pa.string()), pa.array(modes[rng.integers(0, 7, n)]).cast(pa.string())]
        import pyarrow.compute as pc
        cols.append(pc.binary_join_element_wise(pa.array(rng.integers(0, 1 << 40, n)).cast(pa.string()),
                                                pa.array(rng.integers(0, 1 << 30, n)).cast(pa.string()), " carefully final "))
        fields = [pa.field(nm, c.type, nullable=i >= schema.n_key + 2) for i, (nm, c) in enumerate(zip(names, cols))]
        return pa.Table.from_arrays(cols, schema=pa.schema(fields)), part, ship

    files = []
    exp_part = exp_ship = exp_seq = None
    for r in range(5):
        idx = np.arange(n_base, dtype=np.int64) if r == 0 else np.sort(rng.choice(n_base, n_upd, replace=False))
        seq0 = 0 if r == 0 else n_base + (r - 1) * n_upd
        tb, part, ship = run_table(idx, seq0)
        if r == 0:
            exp_part, exp_ship, exp_seq = part.copy(), ship.copy(), np.arange(n_base, dtype=np.int64)
        else:
            exp_part[idx] = part; exp_ship[idx] = ship; exp_seq[idx] = seq0 + np.arange(n_upd, dtype=np.int64)
        sink = pa.BufferOutputStream()
        pq.write_table(tb, sink, compression=codec, use_dictionary=True, data_page_version="1.0", data_page_size=160 << 10,
                       row_group_size=800_000, write_statistics=False, **({"compression_level": 1} if codec == "zstd" else {}))
        files.append((np.frombuffer(sink.getvalue(), np.uint8), r))
    return files, n_base + 4 * n_upd, {"l_partkey": exp_part, "l_shipdate": exp_ship, "_SEQUENCE_NUMBER": exp_seq}


def extra_c5(local_rank, peak, steps=3, codecs=("none", "zstd")):
    """Decode + merge of a C5 bucket from file bytes resident in HBM, `none` and zstd-1 (run A / run B)."""
    from paimon_b200.format import FileUpload, read_section
    from paimon_b200.merge_function import DeduplicateMergeFunction
    from paimon_b200.sort_merge_reader import SortMergeReader
    schema = schema_c5()
    spec = DeduplicateMergeFunction.factory().create()
    out = {"what": "SURVEY C5: one bucket of lineitem-shaped Parquet (15.6 M rows: base run + 4 update runs; dictionary on, "
                   "page V1, 160 KiB pages = 20 000 rows of an 8-byte column) -> device decode -> 5-run deduplicate, timed from file bytes in HBM"}
    for codec in codecs:
        t0 = time.perf_counter()
        files, n_in, expect = c5_bucket(schema, codec)
        gen_s = time.perf_counter() - t0
        up = FileUpload(files, local_rank)
        rd = SortMergeReader([], spec, None, local_rank, schema=schema)
        try:
            dev_files = up.wait()
            ms_dec = ms_mrg = 0.0
            for it in range(2 + steps):
                readers, info = read_section(schema, dev_files, 5, local_rank)
                rd.rebind(readers)
                rd.execute()
                st = rd.stats()
                if it >= 2:
                    ms_dec += info.ms_decode / steps; ms_mrg += st.ms_total / steps
                if it < 1 + steps:
                    for r_ in readers:
                        r_.close()
                    rd.readers = []
            got = rd.fetch()
            names = [f.name for f in schema.file_fields()]
            ok = got.n_rows == len(expect["l_partkey"])
            for nm, want in expect.items():
                col = got.columns[names.index(nm)]
                n_ = got.n_rows
                ok = ok and bool(np.array_equal(np.asarray(col.data)[:n_], want))
                ok = ok and (col.valid is None or bool(np.unpackbits(np.asarray(col.valid, np.uint8), bitorder="little")[:n_].all()))
            for r_ in readers:
                r_.close()
            rd.readers = []
            step = ms_dec + ms_mrg
            out["run_A_none" if codec == "none" else "run_B_zstd1"] = {
                "rows_per_s": n_in / (step * 1e-3), "ms_per_step": step, "decode_ms": ms_dec, "merge_ms": ms_mrg,
                "rows_in": int(n_in), "rows_out": int(got.n_rows), "file_bytes": int(info.file_bytes),
                "encoded_page_bytes": int(info.page_bytes), "decoded_bytes": int(info.decoded_bytes),
                "dictionary_pages": int(info.n_dictionary_pages), "data_pages": int(info.n_data_pages),
                "decode_frac_of_hbm_peak": (info.page_bytes + info.decoded_bytes) / (ms_dec * 1e-3) / 1e9 / peak,
                "parity": "ok" if ok else "MISMATCH", "parity_what": "rows out, l_partkey, l_shipdate and _SEQUENCE_NUMBER of "
                "all merged rows against the generator's last-writer-wins arrays", "host_generation_s": round(gen_s, 1)}
        finally:
            rd.close()
            up.close()
    return out


# ------------------------------------------------------------------ clocks sampling

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            p = [x.strip() for x in s.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ CPU baseline (oracle)

def cpu_baseline(workload, total_sample_rows, threads, steps=1, seed=7):
    """The reference algorithm (oracle port) on the host cores: `threads` independent buckets, one thread
    per bucket exactly like the reference's one-thread-per-split readers."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle
    from paimon_b200 import datagen
    schema = make_schema(workload)
    spec = make_spec(workload, schema)
    w = WORKLOADS[workload]
    per_bucket = max(total_sample_rows // threads, w["n_runs"] * 64)
    n_distinct = min(threads, 8)        # distinct synthetic buckets; threads beyond that re-merge a copy's inputs
    buckets = [datagen.make_runs(schema, w["n_runs"], per_bucket, seed=seed + b, null_prob=w["null_prob"],
                                 delete_prob=w.get("delete_prob", 0.0))
               for b in range(n_distinct)]
    prepared = [pyoracle.prepare(schema, spec, buckets[b % n_distinct]) for b in range(threads)]

    def work(b):
        return pyoracle.run_prepared(prepared[b])          # C call only; the GIL is released

    times, outs = [], []
    with ThreadPoolExecutor(max_workers=threads) as ex:
        for _ in range(steps):
            t0 = time.perf_counter()
            outs = list(ex.map(work, range(threads)))
            times.append(time.perf_counter() - t0)
    rows = per_bucket // w["n_runs"] * w["n_runs"] * threads
    return rows, times, sum(outs)


def load_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    return peak, ("measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s")


def expected_rows(w, all_keys, all_kinds):
    """Size-independent sanity at full size: the number of rows the merge must produce."""
    import torch
    if w.get("drop_delete"):
        # the newest record of a key wins (sequence = run << 32 | row); keys whose winner is a DELETE drop out
        cat_k = torch.cat(all_keys)
        cat_r = torch.cat([torch.full_like(k, r) for r, k in enumerate(all_keys)])
        cat_d = torch.cat(all_kinds).to(torch.int64)
        order = torch.argsort(cat_k * 64 + cat_r)
        sk, sd = cat_k[order], cat_d[order]
        last = torch.ones_like(sk, dtype=torch.bool)
        last[:-1] = sk[1:] != sk[:-1]
        return int((last & (sd == 0)).sum().item())
    return torch.unique(torch.cat(all_keys)).numel()


def parity_sample(schema, spec, rd, run_handles, all_keys, n_out, target_rows=300_000):
    """Compare a key range from the middle of the FULL-size merged batch with the CPU oracle, bit for bit: the input
    rows of the range are read back from the device-resident runs, the oracle merges them, and the result must equal
    the rows of the big batch that carry those keys."""
    import torch
    from oracle import pyoracle
    from paimon_b200.sort_merge_reader import fetch_slice
    n_in = sum(k.numel() for k in all_keys)
    k0 = all_keys[0]
    i0 = int(k0.numel() * 0.37)
    c0 = int(k0[i0].item())
    span = max(1, int(target_rows / max(n_in, 1) * k0.numel()))
    c1 = int(k0[min(i0 + span, k0.numel() - 1)].item())
    bounds = [(int(torch.searchsorted(k, c0).item()), int(torch.searchsorted(k, c1).item())) for k in all_keys]
    slices = [fetch_slice(schema, h, lo, hi) for h, (lo, hi) in zip(run_handles, bounds)]
    want = pyoracle.merge(schema, spec, slices)

    def key_at(i):
        return int(fetch_slice(schema, rd._merge_h, i, i + 1).columns[0].data[0])

    def lower_bound(c):
        lo, hi = 0, n_out
        while lo < hi:
            mid = (lo + hi) // 2
            if key_at(mid) < c:
                lo = mid + 1
            else:
                hi = mid
        return lo
    o0, o1 = lower_bound(c0), lower_bound(c1)
    got = fetch_slice(schema, rd._merge_h, o0, o1)
    ok = got.equals(want)
    return {"result": "ok" if ok else "MISMATCH: " + got.first_difference(want), "rows_in": sum(hi - lo for lo, hi in bounds),
            "rows_out": int(o1 - o0), "key_range": [c0, c1],
            "checked": "every column of the merged rows with keys in the range, taken from the full-size batch, "
                       "bit-exact against the oracle's merge of the same input rows"}


DUMP_BLOCKS, DUMP_BLOCK_ROWS = 64, 256
DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(schema, merge_handle, n_out, out_dir, seed=0):
    """--dump-outputs: a fixed, seeded sample of the merged batch the last timed step left on the device, as the host
    columns SortMergeReader.fetch hands a caller, written as out_dir/<name>.npy so that two builds can be compared
    output for output.  The sample is DUMP_BLOCKS blocks of DUMP_BLOCK_ROWS consecutive rows at seeded positions
    (every row when the batch is smaller).  For each file column <name>:
      <name>.npy                      fixed-width values as float64, 0 under NULL; an INT64 column, which float64
                                      cannot hold exactly, becomes <name>.hi32.npy (signed upper 32 bits) and
                                      <name>.lo32.npy (unsigned lower 32 bits)
      <name>.len.npy, <name>.bytes.npy  var-len columns: byte length of every value (0 under NULL, float64) and the
                                      values' bytes back to back (float32)
      <name>.valid.npy                nullable columns: 1.0 where the value is present (float32)
    and row_index.npy (the sampled row positions) and rows_out.npy (the batch's row count)."""
    from paimon_b200.columnar import unpack_validity
    from paimon_b200.sort_merge_reader import fetch_slice
    from paimon_b200.types import PhysicalType, is_varlen, numpy_dtype
    if n_out <= DUMP_BLOCKS * DUMP_BLOCK_ROWS:
        starts, block = ([0] if n_out else []), n_out
    else:
        slots = np.random.default_rng(seed).choice(n_out // DUMP_BLOCK_ROWS, DUMP_BLOCKS, replace=False)
        starts, block = sorted(int(s) * DUMP_BLOCK_ROWS for s in slots), DUMP_BLOCK_ROWS
    parts = [fetch_slice(schema, merge_handle, s, s + block) for s in starts]

    def cat(arrays, dtype):
        return np.concatenate(arrays).astype(dtype) if arrays else np.zeros(0, dtype)
    out = {"row_index": cat([np.arange(s, s + block) for s in starts], np.float64),
           "rows_out": np.array([n_out], np.float64)}
    for ci, f in enumerate(schema.file_fields()):
        cols = [p.columns[ci].canonical() for p in parts]
        if f.nullable:
            out[f"{f.name}.valid"] = cat([unpack_validity(c.valid, len(c)) for c in cols], np.float32)
        if is_varlen(f.physical):
            out[f"{f.name}.len"] = cat([np.diff(c.offsets.astype(np.int64)) for c in cols], np.float64)
            out[f"{f.name}.bytes"] = cat([c.data for c in cols], np.float32)
        elif f.physical == PhysicalType.INT64:
            v = cat([c.data for c in cols], np.int64)
            out[f"{f.name}.hi32"] = (v >> 32).astype(np.float64)
            out[f"{f.name}.lo32"] = (v & 0xFFFFFFFF).astype(np.float64)
        else:
            out[f.name] = cat([c.data for c in cols], numpy_dtype(f.physical)).astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: the sample takes {total} bytes, more than {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print(f"--dump-outputs: {len(out)} arrays, {total} bytes, {len(out['row_index'])} of {n_out} merged rows -> {out_dir}",
          file=sys.stderr)


# ------------------------------------------------------------------ main

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--source", default=None, choices=["parquet", "columns"],
                    help="timed region starts from Parquet file bytes in HBM (default for c3) or from decoded columns")
    ap.add_argument("--rows", type=int, default=None, help="override total input rows per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-range-rows", type=int, default=8 << 20,
                    help="e2e (--source columns): input rows per key range of the streaming reader (0 = one batch)")
    ap.add_argument("--e2e-depth", type=int, default=3, help="e2e (--source columns): key ranges in flight")
    ap.add_argument("--e2e-frac", type=float, default=0.0,
                    help="e2e (--source columns): fraction of the key space to stream (0 = all if page-locked memory allows)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra sub-lines (merge-only c3, c3agg, c2, c4)")
    ap.add_argument("--no-parity-sample", action="store_true")
    ap.add_argument("--cpu-sample-rows", type=int, default=None)
    ap.add_argument("--cpu-threads", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of the last step's merged batch to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = WORKLOADS[args.workload]
    rows = args.rows or w["rows"]
    source = args.source or ("parquet" if args.workload == "c3" else "columns")
    metric = "merged rows/sec at 16 runs x 100M rows" if args.workload == "c3" else f"merged rows/sec ({args.workload})"
    threads = args.cpu_threads or min(os.cpu_count() or 1, 64)
    cpu_sample = min(args.cpu_sample_rows or threads * (250_000 if args.workload in ("c3", "c3agg") else 1_000_000), rows)
    config = {"workload": f"{args.workload}: {w['desc']}", "rows_per_gpu": rows, "n_runs": w["n_runs"],
              "merge_engine": w["engine"], "buckets_per_gpu": 1, "parallelism": f"bucket-per-gpu x{world}",
              "source": ("parquet: the timed step starts from the bucket's 16 Parquet files resident in HBM (PLAIN data pages "
                         f"V1, {PARQUET_PAGE_ROWS}-row pages, {PARQUET_GROUP_ROWS}-row row groups, uncompressed: the "
                         "synthetic values are random bits), decodes them on the device and merges")
              if source == "parquet" else "columns: decoded columns resident in HBM, merge only",
              "reference_arm_sample": f"the CPU arm merges a {cpu_sample}-row sample of this shape ({threads} buckets, one "
                                      "thread each) from decoded columns, no Parquet decode",
              "l2": "inputs (>30 GB) far exceed the 126 MB L2; no explicit flush" if rows >= 10_000_000
                    else "small input: L2-resident (not a headline configuration)"}

    # ---------------- reference arm: the reference's CPU algorithm on the host cores
    if args.impl == "reference":
        if rank != 0:
            return
        cpu_baseline(args.workload, min(cpu_sample, 200_000), threads, steps=max(args.warmup, 1) if args.warmup else 0)
        nrows, times, _ = cpu_baseline(args.workload, cpu_sample, threads, steps=args.steps)
        total = sum(times)
        val = nrows * len(times) / total
        line = {"impl": "reference", "metric": metric, "value": val, "unit": "rows/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "rows/s", "cores": threads, "kind": "port",
                                 "sample": f"{threads} buckets x {nrows // threads} rows of the same shape, one "
                                           f"thread per bucket (C restatement of LoserTree+MergeFunction over decoded "
                                           f"columns; no JVM in the image)"},
                "e2e": {"value": val, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ---------------- B200 arm
    numa = bind_to_gpu_numa_node(local_rank)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the merge path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from paimon_b200 import _native as N
    from paimon_b200.columnar import Column, KeyValueBatch
    from paimon_b200.format import read_section
    from paimon_b200.sort_merge_reader import RangeStreamingMergeReader, SortedRunReader, SortMergeReader

    schema = make_schema(args.workload)
    spec = make_spec(args.workload, schema)
    lib = N.init(local_rank)
    peak, peak_kind = load_peak()
    n_runs = w["n_runs"]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    extra = {}
    parity = None
    roofline_decode = None

    if source == "parquet":
        enc_handles, images, all_keys, all_kinds = device_parquet_files(args.workload, schema, rows, dev, 100 + rank, lib)
        n_in = sum(k.numel() for k in all_keys)
        files = [(img, r) for r, img in enumerate(images)]
        rd = SortMergeReader([], spec, None, local_rank, schema=schema)
        dstream = C.c_void_p(0)
        N.check(lib.pg_thread_stream(C.byref(dstream)))

        def one_step(keep_runs=False):
            readers, info = read_section(schema, files, n_runs, local_rank)
            rd.rebind(readers)
            rd.execute()
            st_ = rd.stats()
            if not keep_runs:
                for r_ in readers:
                    r_.close()
                rd.readers = []
            return info, st_, readers

        for _ in range(warm):
            info, st, _ = one_step()
        n_out = st.rows_out
        assert info.n_rows == n_in
        uniq = expected_rows(w, all_keys, all_kinds)
        assert n_out == uniq, f"merged rows {n_out} != expected rows {uniq}"
        in_bytes, out_bytes, page_bytes, file_bytes = info.decoded_bytes, st.bytes_out, info.page_bytes, info.file_bytes

        ext_dec = torch.cuda.ExternalStream(dstream.value or 0, device=dev)
        ext_mrg = torch.cuda.ExternalStream(rd.cuda_stream(), device=dev)
        sampler = ClockSampler(local_rank)
        barrier()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms_emit = ms_plan = ms_part = ms_tot = ms_alloc = ms_dec = 0.0
        launches = 0
        t0 = time.perf_counter()
        e0.record(ext_dec)
        for _ in range(args.steps):
            info, s, _ = one_step()
            ms_dec += info.ms_decode
            ms_emit += s.ms_emit; ms_plan += s.ms_plan; ms_part += s.ms_partition; ms_tot += s.ms_total
            ms_alloc += s.ms_alloc
            launches += s.launches + info.launches
        e1.record(ext_mrg)
        barrier()
        wall = time.perf_counter() - t0
        clocks = sampler.stop()
        dev_ms = e0.elapsed_time(e1)
        dec_ms = ms_dec / args.steps
        dec_alg = page_bytes + in_bytes
        dec_traffic = None
        try:
            tjd = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if args.workload == "c3" and rows == w["rows"]:
                dec_traffic = tjd["c3_decode"]["traffic"]
        except Exception:
            pass
        roofline_decode = {"bound": "hbm", "stage": "parquet decode (page walk + levels + value walk + expand)", "traffic": dec_traffic,
                           "achieved": dec_alg / (dec_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": dec_alg / (dec_ms * 1e-3) / 1e9 / peak, "stage_ms": dec_ms,
                           "algorithmic_bytes": int(dec_alg), "encoded_page_bytes": int(page_bytes),
                           "decoded_bytes": int(in_bytes), "file_bytes": int(file_bytes),
                           "pages": int(info.n_data_pages), "chunks": int(info.n_chunks), "launches": int(info.launches)}
    else:
        readers, all_keys, in_bytes, all_kinds = device_runs(args.workload, schema, rows, dev, seed=100 + rank)
        n_in = sum(r.n_rows for r in readers)
        rd = SortMergeReader.create_sort_merge_reader(readers, None, None, spec, device=local_rank)
        for _ in range(warm):
            rd.execute()
        st = rd.stats()
        n_out = st.rows_out
        uniq = expected_rows(w, all_keys, all_kinds)
        assert n_out == uniq, f"merged rows {n_out} != expected rows {uniq}"
        out_bytes = st.bytes_out
        ext = torch.cuda.ExternalStream(rd.cuda_stream(), device=dev)
        sampler = ClockSampler(local_rank)
        barrier()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms_emit = ms_plan = ms_part = ms_tot = ms_alloc = 0.0
        launches = 0
        t0 = time.perf_counter()
        e0.record(ext)
        for _ in range(args.steps):
            rd.execute()
            s = rd.stats()
            ms_emit += s.ms_emit; ms_plan += s.ms_plan; ms_part += s.ms_partition; ms_tot += s.ms_total
            ms_alloc += s.ms_alloc
            launches += s.launches
        e1.record(ext)
        barrier()
        wall = time.perf_counter() - t0
        clocks = sampler.stop()
        dev_ms = e0.elapsed_time(e1)

    if args.dump_outputs and rank == 0:
        dump_outputs(schema, rd._merge_h, int(s.rows_out), args.dump_outputs)

    t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    step_ms = float(t.item()) / args.steps
    value = world * n_in / (step_ms * 1e-3)

    alg_bytes = in_bytes + out_bytes
    emit_ms = ms_emit / args.steps
    # DRAM traffic of the dominant kernel from the committed ncu capture of this workload at its full size
    # (profiles/traffic.json; only meaningful for the default row count)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if args.workload in tj and rows == w["rows"]:
            traffic = tj[args.workload]["traffic"]
    except Exception:
        pass
    achieved = alg_bytes / (emit_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "k_emit", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "peak_source": peak_kind, "traffic": traffic,
                "algorithmic_bytes": int(alg_bytes), "kernel_ms": emit_ms,
                "step_frac": alg_bytes / (step_ms * 1e-3) / 1e9 / peak,
                "phase_ms": {"decode": (ms_dec / args.steps) if source == "parquet" else None,
                             "partition": ms_part / args.steps, "plan+scan": ms_plan / args.steps,
                             "size_readback+alloc": ms_alloc / args.steps, "emit": emit_ms,
                             "merge_total": ms_tot / args.steps, "step": step_ms}}
    if source == "parquet":
        # the whole decode+merge step on its minimal traffic: encoded pages in, merged batch out
        fused_alg = page_bytes + out_bytes
        roofline["step_frac_fused_definition"] = fused_alg / (step_ms * 1e-3) / 1e9 / peak
        roofline["fused_algorithmic_bytes"] = int(fused_alg)

    # ---------------- parity sample at full size + extras that reuse the decoded runs
    if source == "parquet":
        info, st, run_readers = one_step(keep_runs=True)       # decoded runs + the full-size batch stay on the device
        if not args.no_parity_sample and schema.n_key == 1 and not w.get("drop_delete"):
            t0p = time.perf_counter()
            parity = parity_sample(schema, spec, rd, [r_._handle for r_ in run_readers], all_keys, n_out)
            parity["seconds"] = round(time.perf_counter() - t0p, 2)
        if world == 1 and not args.no_extra:
            # round 1's measurement: the merge alone over the decoded runs
            tms = {"emit": 0.0, "total": 0.0, "plan": 0.0}
            for _ in range(5):
                rd.execute()
                s = rd.stats()
                tms["emit"] += s.ms_emit / 5; tms["total"] += s.ms_total / 5; tms["plan"] += s.ms_plan / 5
            extra[f"{args.workload}_merge_only"] = {
                "what": "merge of the decoded runs (columns resident in HBM), device-timed", "rows_per_s": n_in / (tms["total"] * 1e-3),
                "ms_per_step": tms["total"], "emit_ms": tms["emit"], "plan_scan_ms": tms["plan"],
                "emit_frac_of_hbm_peak": alg_bytes / (tms["emit"] * 1e-3) / 1e9 / peak}
            if args.workload == "c3":
                spec_agg = make_spec("c3agg", schema)
                ra = SortMergeReader([], spec_agg, None, local_rank, schema=schema)
                try:
                    ra.rebind(run_readers)
                    for _ in range(2):
                        ra.execute()
                    tm = {"emit": 0.0, "total": 0.0}
                    for _ in range(3):
                        ra.execute()
                        s = ra.stats()
                        tm["emit"] += s.ms_emit / 3; tm["total"] += s.ms_total / 3
                    extra["c3agg_merge_only"] = {
                        "what": WORKLOADS["c3agg"]["desc"], "rows_per_s": n_in / (tm["total"] * 1e-3), "ms_per_step": tm["total"],
                        "emit_ms": tm["emit"], "rows_out": int(s.rows_out),
                        "emit_frac_of_hbm_peak": (in_bytes + s.bytes_out) / (tm["emit"] * 1e-3) / 1e9 / peak}
                finally:
                    ra.readers = []
                    ra.close()
        for r_ in run_readers:
            r_.close()
        rd.readers = []

    # ---------------- compaction rewrite: encode the merged batch to Parquet on the device (C4)
    rewrite = None
    if w.get("drop_delete"):
        from paimon_b200.compact_rewriter import file_column_names
        names = file_column_names(schema)
        arr = (C.c_char_p * len(names))(*[nm.encode() for nm in names])
        enc_ms, fbytes, pages = [], 0, 0
        for _ in range(3):
            fh = C.c_uint64(0)
            N.check(lib.pg_parquet_encode(rd._merge_h, arr, 0, -1, None, C.byref(fh)))
            fm = N.PgFileMeta()
            N.check(lib.pg_parquet_file_meta(fh.value, C.byref(fm)))
            enc_ms.append(float(fm.ms_encode)); fbytes = int(fm.file_bytes); pages = int(fm.n_pages)
            lib.pg_parquet_file_free(fh.value)
        em = min(enc_ms)
        rewrite = {"encode_ms": em, "file_bytes": fbytes, "pages": pages, "encode_GBps": fbytes / (em * 1e-3) / 1e9,
                   "merge_plus_encode_rows_per_s": n_in / ((step_ms + em) * 1e-3)}

    # ---------------- e2e: host buffers in, host batch out, through the public reader API
    e2e = None
    if not args.no_e2e and source == "parquet":
        # the files move to page-locked host memory; the device copies are dropped
        host_files = []
        pinned = True
        try:                                  # every rank of the node locks its files + its output arena
            import psutil
            local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
            need_host = (sum(sz for _, sz in images) + int(out_bytes * 1.02)) * local_world
            if psutil.virtual_memory().available < 1.3 * need_host:
                pinned = False                # (pageable buffers: the copies get staged by the driver, slower but safe)
        except Exception:
            pass

        def host_buffer(nbytes):
            if pinned:
                try:
                    return torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
                except RuntimeError:
                    pass
            return torch.empty(nbytes, dtype=torch.uint8)
        for fh, (ptr, size) in zip(enc_handles, images):
            hb = host_buffer(size)
            N.check(lib.pg_parquet_file_fetch(fh, hb.data_ptr(), size))
            host_files.append(hb.numpy())
            lib.pg_parquet_file_free(fh)
        enc_handles = []
        rd.close()
        torch.cuda.empty_cache()
        lib.pg_trim()
        arena = host_buffer(int(out_bytes * 1.02) + (64 << 20))
        arena_np = arena.numpy()
        hfiles = [(hf, r) for r, hf in enumerate(host_files)]
        mrs = [SortMergeReader([], spec, None, local_rank, schema=schema) for _ in range(2)]
        free_q, full_q = queue.Queue(), queue.Queue()
        for m_ in mrs:
            free_q.put(m_)
        d2h_bytes = [0]
        rows_seen = []
        errors = []

        def consumer():
            try:
                while True:
                    m_ = full_q.get()
                    if m_ is None:
                        return
                    top = [0]

                    def alloc(nbytes):
                        a = (top[0] + 63) & ~63
                        top[0] = a + nbytes
                        return arena_np[a:a + nbytes]
                    out = m_.fetch(allocator=alloc)                   # D2H of the merged batch
                    d2h_bytes[0] = m_.stats().bytes_d2h
                    rows_seen.append(out.n_rows)
                    free_q.put(m_)                                    # (the handle keeps its output arena for the next bucket)
            except BaseException as e:                                # surfaced below
                errors.append(e)
                free_q.put(None)

        n_e2e = max(1, args.e2e_steps)
        from paimon_b200.format import FileUpload

        def run_buckets(n_steps, overlap_upload):
            """K consecutive buckets; with overlap_upload the files of bucket i + 1 are on their way to the device
            (FileUpload: the library's upload stream) while bucket i decodes and merges."""
            th = threading.Thread(target=consumer, daemon=True)
            th.start()
            barrier()
            t0 = time.perf_counter()
            up_next = FileUpload(hfiles, local_rank) if overlap_upload else None
            try:
                for i in range(n_steps):
                    m_ = free_q.get()
                    if m_ is None:
                        raise errors[0]
                    up, files_i = None, hfiles
                    if overlap_upload:
                        up, up_next = up_next, None
                        files_i = up.wait()
                        if i + 1 < n_steps:
                            up_next = FileUpload(hfiles, local_rank)
                    try:
                        rdrs, sec = read_section(schema, files_i, n_runs, local_rank)   # (H2D of the file bytes +) decode
                        m_.rebind(rdrs)
                        m_.execute()
                        for r_ in rdrs:
                            r_.close()
                        m_.readers = []
                    finally:
                        if up is not None:
                            up.close()
                    full_q.put(m_)
            finally:
                if up_next is not None:
                    up_next.close()
                full_q.put(None)
                th.join()
            torch.cuda.synchronize()
            if errors:
                raise errors[0]
            return time.perf_counter() - t0

        # what the link gives on this box: the file upload alone (the read-back alone is timed after the loop)
        t0u = time.perf_counter()
        up0 = FileUpload(hfiles, local_rank)
        up0.wait()
        h2d_only_ms = 1e3 * (time.perf_counter() - t0u)
        up0.close()
        overlap = True
        try:
            run_buckets(1, True)
        except N.PaimonGpuError as ex:
            # two file images + the decoded runs + two output batches did not fit: copy inside read_section instead
            if "memory" not in str(ex):
                raise
            overlap = False
            errors.clear(); rows_seen.clear()
            while not free_q.empty():
                free_q.get()
            for m_ in mrs:
                free_q.put(m_)
            lib.pg_trim()
            run_buckets(1, False)
        dt = run_buckets(n_e2e, overlap)
        # what the link gives on this box: the read-back alone, and one upload + one read-back issued together
        link = {}
        try:
            def fetch_again():
                top_ = [0]

                def alloc_(nbytes):
                    a = (top_[0] + 63) & ~63
                    top_[0] = a + nbytes
                    return arena_np[a:a + nbytes]
                mrs[0].fetch(allocator=alloc_)
            t0l = time.perf_counter()
            fetch_again()
            link["d2h_alone_ms"] = 1e3 * (time.perf_counter() - t0l)
            t0l = time.perf_counter()
            upl = FileUpload(hfiles, local_rank)
            fetch_again()
            upl.wait()
            link["h2d_and_d2h_together_ms"] = 1e3 * (time.perf_counter() - t0l)
            upl.close()
        except Exception as ex:                                          # a probe must not take the line down
            link["error"] = repr(ex)[:200]
        assert all(x == n_out for x in rows_seen), (rows_seen, n_out)
        tt = torch.tensor([dt / n_e2e], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        h2d = int(sum(len(hf) for hf in host_files))
        e2e = {"value": world * n_in / float(tt.item()), "unit": "rows/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": int(d2h_bytes[0]), "ms_per_step": 1e3 * float(tt.item()), "steps": n_e2e,
               "rows_in_per_step": int(n_in), "rows_out_per_step": int(n_out), "sample": "the whole bucket",
               "numa": numa,
               "api": "format.FileUpload(host Parquet file bytes) -> format.read_section -> SortMergeReader.rebind/execute -> "
                      "fetch() over the C ABI; wall clock of K consecutive buckets / K; the H2D of bucket i+1's files "
                      "(library upload stream) and the D2H of bucket i-1's batch (second merge handle) overlap the decode + "
                      "merge of bucket i; pinned buffers bound to the GPU's NUMA node",
               "upload_overlapped": overlap, "h2d_alone_ms": h2d_only_ms, "link_probes": link,
               "host_buffers": "page-locked" if pinned else "pageable (not enough free host memory to lock every rank's buffers)",
               "h2d_alone_gbs": sum(len(hf) for hf in host_files) / (h2d_only_ms * 1e-3) / 1e9,
               "pcie_floor_ms": 1e3 * max(h2d, int(d2h_bytes[0])) / 55e9}
        for m_ in mrs:
            m_.close()
        del arena, arena_np, host_files
    elif not args.no_e2e:
        ftypes = schema.physical_types()
        # device -> pinned host copies of every input buffer (the step's inputs live in page-locked memory)
        # Page-locked host memory is finite and every rank of the box needs its own copy of the inputs and room for
        # the outputs: when that does not fit comfortably, the end-to-end leg streams a key-range PREFIX of the
        # bucket (the first e2e_frac of the key space; same runs, same shape) and reports rows/s on it.
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
        e2e_frac = args.e2e_frac
        if e2e_frac <= 0:
            try:
                avail = next(int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable"))
            except Exception:
                avail = 256 << 30
            need = (in_bytes + out_bytes * 1.05) * local_world
            e2e_frac = 1.0 if need <= 0.5 * avail else max(0.05, 0.5 * avail / need)
        hi_rows = [r.n_rows for r in readers]
        e2e_rows_in, e2e_rows_out = n_in, n_out
        if e2e_frac < 1.0 and schema.n_key == 1 and not w.get("drop_delete"):
            cut = all_keys[0][min(int(e2e_frac * all_keys[0].numel()), all_keys[0].numel() - 1)]
            hi_rows = [int(torch.searchsorted(k_, cut).item()) for k_ in all_keys]
            hi_rows = [max(h, 1) for h in hi_rows]
            e2e_rows_in = sum(hi_rows)
            e2e_rows_out = torch.unique(torch.cat([k_[:h] for k_, h in zip(all_keys, hi_rows)])).numel()
        else:
            e2e_frac = 1.0
        host_runs = []
        e2e_out_bytes = int(out_bytes * (e2e_rows_in / max(n_in, 1)) * 1.1) if e2e_frac < 1.0 else int(out_bytes)
        for r, hi in zip(readers, hi_rows):
            cols = []
            byptr = {tt.data_ptr(): tt for tt in r.keepalive}
            cache = {}

            def to_host(ptr, count=None, byptr=byptr, cache=cache):
                if not ptr:
                    return None
                if ptr not in cache:
                    tt = byptr[ptr]
                    if count is not None:
                        tt = tt[:count]
                    hb = torch.empty(tt.shape, dtype=tt.dtype, pin_memory=True)
                    hb.copy_(tt)
                    cache[ptr] = hb.numpy()
                return cache[ptr]
            for ci, dc in enumerate(r.device_columns):
                t_ = ftypes[ci]
                offs = to_host(dc.offsets, hi + 1)
                if offs is not None:
                    data = to_host(dc.data, int(offs[hi]) + 16).view(np.uint8)
                else:
                    data = to_host(dc.data, hi)
                val = to_host(dc.validity, (hi + 7) // 8 + 8)
                cols.append(Column(t_, data[:hi] if offs is None else data, offs, val))
            host_runs.append(KeyValueBatch(schema, cols))
        torch.cuda.synchronize()
        rd.close()
        del readers, all_keys
        torch.cuda.empty_cache()
        arena = torch.empty(int(e2e_out_bytes * 1.02) + (64 << 20), dtype=torch.uint8, pin_memory=True)
        arena_np = arena.numpy()
        e2e_times, h2d_b, d2h_b = [], 0, 0
        single_key = schema.n_key == 1
        for it_ in range(max(args.e2e_steps, 2)):
            top = [0]
            lock = threading.Lock()

            def alloc(nbytes):
                with lock:
                    a = (top[0] + 63) & ~63
                    top[0] = a + nbytes
                return arena_np[a:a + nbytes]
            barrier()
            t0 = time.perf_counter()
            rows_out = 0
            if single_key and args.e2e_range_rows > 0:
                # batches of key ranges: H2D of range i+1 | merge of range i | D2H of range i-1
                mr = RangeStreamingMergeReader(schema, host_runs, spec, target_rows=args.e2e_range_rows,
                                               depth=args.e2e_depth, device=local_rank,
                                               allocator_factory=lambda: alloc)
                while True:
                    out = mr.read_batch()
                    if out is None:
                        break
                    rows_out += out.n_rows
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                h2d_b, d2h_b = mr.bytes_h2d, mr.bytes_d2h
                mr.close()
            else:
                hr = [SortedRunReader(schema, b) for b in host_runs]
                mr = SortMergeReader.create_sort_merge_reader(hr, None, None, spec, device=local_rank)   # H2D
                mr.execute()
                out = mr.fetch(allocator=alloc)                                                           # D2H
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                s = mr.stats()
                h2d_b, d2h_b = s.bytes_h2d, s.bytes_d2h
                rows_out = out.n_rows
                mr.close()
            assert rows_out == e2e_rows_out, (rows_out, e2e_rows_out)
            if it_ > 0:
                e2e_times.append(dt)
        tt = torch.tensor([sum(e2e_times) / len(e2e_times)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * e2e_rows_in / float(tt.item()), "unit": "rows/s", "h2d_bytes_per_step": int(h2d_b),
               "d2h_bytes_per_step": int(d2h_b), "ms_per_step": 1e3 * float(tt.item()), "steps": len(e2e_times),
               "rows_in_per_step": int(e2e_rows_in), "rows_out_per_step": int(e2e_rows_out), "numa": numa,
               "sample": ("the whole bucket" if e2e_frac >= 1.0 else
                          f"key-range prefix of the bucket ({e2e_frac:.2f} of the key space): page-locked host memory "
                          f"for {local_world} ranks' full inputs + outputs was not available"),
               "api": ("RangeStreamingMergeReader(host runs).read_batch() loop over the C ABI: key ranges of "
                       f"~{args.e2e_range_rows} rows, {args.e2e_depth} in flight (H2D | merge | D2H overlap)")
               if single_key and args.e2e_range_rows > 0 else
               "SortMergeReader.create_sort_merge_reader(host runs).execute()+fetch() over the C ABI"}
    else:
        rd.close()
        if source == "parquet":
            for fh in enc_handles:
                lib.pg_parquet_file_free(fh)

    # ---------------- extra sub-lines: other BASELINE configs in the same invocation (merge of decoded columns)
    if world == 1 and not args.no_extra and args.workload == "c3" and rows == w["rows"]:
        torch.cuda.empty_cache()
        lib.pg_trim()
        for wl in ("c2", "c4"):
            try:
                sc2 = make_schema(wl)
                sp2 = make_spec(wl, sc2)
                rds2, keys2, inb2, kinds2 = device_runs(wl, sc2, WORKLOADS[wl]["rows"], dev, seed=100)
                r2 = SortMergeReader.create_sort_merge_reader(rds2, None, None, sp2, device=local_rank)
                try:
                    for _ in range(3):
                        r2.execute()
                    assert r2.stats().rows_out == expected_rows(WORKLOADS[wl], keys2, kinds2)
                    tm = {"emit": 0.0, "total": 0.0, "plan": 0.0, "part": 0.0}
                    for _ in range(5):
                        r2.execute()
                        s = r2.stats()
                        tm["emit"] += s.ms_emit / 5; tm["total"] += s.ms_total / 5; tm["plan"] += s.ms_plan / 5
                        tm["part"] += s.ms_partition / 5
                    n2 = sum(x.n_rows for x in rds2)
                    alg2 = inb2 + s.bytes_out
                    extra[f"{wl}_merge_only"] = {
                        "what": WORKLOADS[wl]["desc"], "rows_per_s": n2 / (tm["total"] * 1e-3), "ms_per_step": tm["total"],
                        "emit_ms": tm["emit"], "plan_scan_ms": tm["plan"], "partition_ms": tm["part"],
                        "rows_in": int(n2), "rows_out": int(s.rows_out),
                        "emit_frac_of_hbm_peak": alg2 / (tm["emit"] * 1e-3) / 1e9 / peak,
                        "step_frac_of_hbm_peak": alg2 / (tm["total"] * 1e-3) / 1e9 / peak}
                finally:
                    r2.close()
                    del rds2, keys2, kinds2
                    torch.cuda.empty_cache()
                    lib.pg_trim()
            except Exception as e:                                   # an extra must not take the headline line down
                extra[f"{wl}_merge_only"] = {"error": repr(e)[:300]}

    if world == 1 and not args.no_extra and args.workload == "c3" and rows == w["rows"]:
        try:
            extra["c5"] = extra_c5(local_rank, peak)
        except Exception as e:
            extra["c5"] = {"error": repr(e)[:300]}
        lib.pg_trim()

    # ---------------- extra: C4's bucket scheduling on hardware — many buckets per GPU, longest-processing-time
    # assignment by input bytes (paimon_b200/bucket_scheduler.py), every rank merging its own buckets back to back
    if not args.no_extra and args.workload == "c3" and rows == w["rows"]:
        try:
            from paimon_b200.bucket_scheduler import assign_buckets, reduce_stats
            n_buckets = 8 * world
            rng_b = np.random.default_rng(7)
            bucket_rows = [int(x) for x in rng_b.integers(1_000_000, 3_000_000, n_buckets)]     # skewed bucket sizes
            mine = assign_buckets(n_buckets, world, weights=bucket_rows)[rank]
            sc4 = make_schema("c4")
            sp4 = make_spec("c4", sc4)
            t_ms, r_in, r_out = 0.0, 0, 0
            for b in mine:
                rds4, keys4, _, kinds4 = device_runs("c4", sc4, bucket_rows[b], dev, seed=1000 + b)
                r4 = SortMergeReader.create_sort_merge_reader(rds4, None, None, sp4, device=local_rank)
                try:
                    r4.execute()
                    r4.execute()
                    s4 = r4.stats()
                    assert s4.rows_out == expected_rows(WORKLOADS["c4"], keys4, kinds4)
                    t_ms += s4.ms_total; r_in += s4.rows_in; r_out += s4.rows_out
                finally:
                    r4.close()
                    del rds4, keys4, kinds4
                    torch.cuda.empty_cache()
            agg = reduce_stats({"rows_in": float(r_in), "rows_out": float(r_out), "device_ms": t_ms}, device=dev)
            extra["c4_bucket_schedule"] = {
                "what": f"{n_buckets} C4-shaped buckets of 1-3 M rows (32 runs each) over {world} GPU(s), LPT assignment by "
                        "input rows, device-timed merges back to back; device_ms is the slowest rank's sum",
                "buckets_of_rank0": mine if rank == 0 else None, "rows_in": int(agg["rows_in"]), "rows_out": int(agg["rows_out"]),
                "device_ms": agg["device_ms"], "rows_per_s": agg["rows_in"] / (agg["device_ms"] * 1e-3)}
            lib.pg_trim()
        except Exception as e:
            extra["c4_bucket_schedule"] = {"error": repr(e)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        nrows, times, _ = cpu_baseline(args.workload, cpu_sample, threads, steps=2)
        cpu = {"value": nrows / min(times), "unit": "rows/s", "cores": threads, "kind": "port",
               "sample": f"{threads} buckets x {nrows // threads} rows of the same shape, one thread per bucket; "
                         f"oracle = C restatement of LoserTree+MergeFunction over decoded columns (no JVM in the image)"}

    if rank == 0:
        line = {"metric": metric, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": config,
                "rows_in_per_gpu": int(n_in), "rows_out_per_gpu": int(n_out), "wall_ms_per_step": 1e3 * wall / args.steps,
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}
        if roofline_decode is not None:
            line["roofline_decode"] = roofline_decode
        if parity is not None:
            line["parity_sample"] = parity["result"]
            line["parity_sample_detail"] = parity
        if rewrite is not None:
            line["rewrite"] = rewrite
        if extra:
            line["extra"] = extra
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
