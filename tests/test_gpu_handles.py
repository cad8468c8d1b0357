"""Wide schemas, several live handles and input lifetimes, every result against the CPU oracle.

  * schema widths from 1 to the ABI's 4096 fields, across the 32-field warp, the 128-field tile-decode cut and the shared-memory
    lines of the encoder's size pass (48 KiB without opt-in, 227 KiB with it): encode, decode (synchronising and pipelined, full
    and pruned reader schema) and schema inference;
  * decoders and encoders alive at the same time whose launches need different amounts of dynamic shared memory, on one
    thread and on eight threads whose first launches coincide (tfrgpu.h: one handle per Spark task thread, many task threads
    per executor process);
  * input lifetimes: a device buffer overwritten as soon as tfr_decode returns, a host-input batch redone from its lane's
    device copy while the next batch is copied into that lane, and columns the encoder reads straight from device memory at
    arbitrary alignment and first offsets.

Reference semantics: M/TFRecordFileReader.scala:49-81, M/TFRecordDeserializer.scala:21-61, M/TFRecordSerializer.scala:20-60,
M/TensorFlowInferSchema.scala:35-58."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from util import assert_columns_equal, record_offsets
from spark_tfrecord_b200 import _cabi as A
from spark_tfrecord_b200.sqltypes import *  # noqa

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    from spark_tfrecord_b200 import _native
    _native.lib()
    return _native


def _encode(oracle, sch, cols, record_type=0):
    data, rc, _ = oracle.encode(cols, sch, record_type)
    assert rc == 0
    return np.frombuffer(data, dtype=np.uint8)


def _check(batch, want, sch, what):
    """a decoded batch against an oracle result: status, row count, consumed bytes and every column, bit for bit"""
    info = batch.info
    for k in ("error_code", "error_row", "n_rows", "consumed_bytes"):
        assert info[k] == want.info[k], (what, k, info, want.info)
    assert_columns_equal(batch.to_host(), want.columns, sch.names, what)


def _cuda(data):
    import torch
    return torch.from_numpy(np.array(data, dtype=np.uint8, copy=True)).cuda()


# ------------------------------------------------------------------------------------------------------------------------
# A. schema width sweep
# ------------------------------------------------------------------------------------------------------------------------
# The Example size pass (encode_tile_size_kernel) stages the schema's fields (DevField, 36 B) and column pointers (EncCol,
# 40 B) in dynamic shared memory, each array rounded up to 16 B (enc_tile_meta_bytes), next to 32 words of static
# accumulators.  A launch needs the opt-in attribute above 48 KiB and cannot exceed 227 KiB on sm_100 at all.
_DEVFIELD_BYTES, _ENCCOL_BYTES, _SIZE_PASS_STATIC = 36, 40, 32 * 4


def _size_pass_smem(nf):
    r16 = lambda b: (b + 15) & ~15  # noqa: E731
    return r16(nf * _DEVFIELD_BYTES) + r16(nf * _ENCCOL_BYTES) + _SIZE_PASS_STATIC


def _last_width_within(limit):
    nf = 1
    while _size_pass_smem(nf + 1) <= limit:
        nf += 1
    return nf


W48 = _last_width_within(48 * 1024)
W227 = _last_width_within(227 * 1024)
WIDTHS = sorted({1, 31, 32, 33, 127, 128, 129, 646, 647, 648, W48, W48 + 1, 1000, W227, W227 + 1, 4096})
SWEEP_ROWS = 97                 # three full 32-row tiles and a partial one


def _field_name(i, rng):
    """unique names of 1 to 200 bytes: the field's index in base 36, padded with characters that are not base-36 digits"""
    tag = np.base_repr(i, 36).lower()
    n = max(len(tag), int(rng.integers(1, 201)))
    return tag + "".join("-_~."[(i + k) % 4] for k in range(n - len(tag)))


def _wide_schema(nf, seed, seq=False):
    """mostly scalar long and float columns, array<string> every fifth field, DoubleType and IntegerType among them, about
    10 % nulls; with seq, every tenth field is a FeatureList of floats instead"""
    rng = np.random.default_rng(seed)
    fields, gens = [], []
    for i in range(nf):
        name = _field_name(i, rng)
        if seq and i % 10 == 4:
            dt, gen = ArrayType(ArrayType(FloatType())), lambda r: [[float(x) for x in r.standard_normal(int(r.integers(0, 4))).astype(np.float32)]
                                                                  for _ in range(int(r.integers(0, 4)))]
        elif i % 5 == 4:
            dt, gen = ArrayType(StringType()), lambda r: ["".join(chr(97 + int(c)) for c in r.integers(0, 26, int(r.integers(0, 13))))
                                                        for _ in range(int(r.integers(0, 4)))]
        elif i % 10 == 1:
            dt, gen = DoubleType(), lambda r: float(np.float32(r.standard_normal()))
        elif i % 10 == 2:
            dt, gen = IntegerType(), lambda r: int(r.integers(-2**31, 2**31))
        elif i % 2 == 0:
            dt, gen = LongType(), lambda r: int(r.integers(-2**63, 2**63 - 1)) if r.random() < 0.3 else int(r.integers(0, 1000))
        else:
            dt, gen = FloatType(), lambda r: float(np.float32(r.standard_normal()))
        fields.append(StructField(name, dt, True))
        gens.append(gen)
    return StructType(fields), gens


def _wide_rows(gens, n, seed):
    r = np.random.default_rng(seed)
    return [tuple(None if r.random() < 0.1 else g(r) for g in gens) for _ in range(n)]


def test_sweep_widths_cover_the_shared_memory_lines():
    """the sweep straddles both limits of the size pass, computed from the layout above (no GPU needed)"""
    assert _size_pass_smem(W48) <= 48 * 1024 < _size_pass_smem(W48 + 1)
    assert _size_pass_smem(W227) <= 227 * 1024 < _size_pass_smem(W227 + 1)
    assert 600 < W48 < 700 and 2900 < W227 < 3100 and max(WIDTHS) == 4096


@pytest.mark.parametrize("nf", WIDTHS)
def test_width_sweep_example(native, oracle, nf):
    sch, gens = _wide_schema(nf, seed=nf)
    rows = _wide_rows(gens, SWEEP_ROWS, seed=10_000 + nf)
    cols = A.columns_from_rows(sch, rows)
    data = _encode(oracle, sch, cols)
    # (a) encode: two calls of one encoder (the second reuses its buffers and size history)
    enc = native.Encoder(sch)
    try:
        for it in range(2):
            assert enc.encode(cols) == data.tobytes(), f"{nf} fields: encode call {it + 1} differs from the oracle writer"
    finally:
        enc.close()
    # (b) decode: synchronising, then twice pipelined
    want = oracle.decode(data, sch)
    assert want.info["error_code"] == 0 and want.n_rows == SWEEP_ROWS
    dev = _cuda(data)
    dec = native.Decoder(sch)
    try:
        b, used = dec.decode(data)
        assert used == len(data)
        _check(b, want, sch, f"{nf} fields: decode"); b.release()
        for it in range(2):
            b = dec.submit(dev)
            _check(b, want, sch, f"{nf} fields: submit {it + 1}"); b.release()
    finally:
        dec.close()
    # (c) a reader schema of every other field, in reverse order
    rsch = StructType(list(reversed(sch.fields[::2])))
    want_r = oracle.decode(data, rsch)
    dec = native.Decoder(rsch)
    try:
        b, _ = dec.decode(dev)
        _check(b, want_r, rsch, f"{nf} fields: pruned and reversed reader schema"); b.release()
    finally:
        dec.close()
    # (d) schema inference; a record with more than 1024 features in its map exceeds the GPU tables by design
    rc, want_inf = oracle.infer(data, 0)
    assert rc == 0
    most = max(sum(v is not None for v in row) for row in rows)
    inf = native.Infer(0)
    try:
        if most <= 1024:
            inf.update(data)
            assert inf.result() == want_inf, f"{nf} fields: inferred schema differs"
        else:
            with pytest.raises(native.TfrError) as ei:
                inf.update(data)
            assert ei.value.code == A.TFR_E_BATCH_TOO_LARGE and "1024" in str(ei.value)
    finally:
        inf.close()


@pytest.mark.parametrize("nf", [129, 1000, 4096])
def test_width_sweep_sequence_example(native, oracle, nf):
    sch, gens = _wide_schema(nf, seed=50_000 + nf, seq=True)
    cols = A.columns_from_rows(sch, _wide_rows(gens, SWEEP_ROWS, seed=60_000 + nf), 1)
    data = _encode(oracle, sch, cols, 1)
    enc = native.Encoder(sch, 1)
    try:
        for it in range(2):
            assert enc.encode(cols) == data.tobytes(), f"{nf} fields, SequenceExample: encode call {it + 1} differs"
    finally:
        enc.close()
    want = oracle.decode(data, sch, 1)
    assert want.info["error_code"] == 0 and want.n_rows == SWEEP_ROWS
    dec = native.Decoder(sch, 1)
    try:
        b, _ = dec.decode(data)
        _check(b, want, sch, f"{nf} fields, SequenceExample: decode"); b.release()
        b = dec.submit(_cuda(data))
        _check(b, want, sch, f"{nf} fields, SequenceExample: submit"); b.release()
    finally:
        dec.close()


def test_more_than_4096_fields_is_rejected(native):
    sch = StructType([StructField(f"c{i}", LongType()) for i in range(4097)])
    with pytest.raises(native.TfrError) as ei:
        native.Schema(sch)
    assert ei.value.code == A.TFR_E_INVALID_ARG


# ------------------------------------------------------------------------------------------------------------------------
# B. several live handles
# ------------------------------------------------------------------------------------------------------------------------
def _narrow(n, seed, str_len=(0, 12)):
    """three scalar columns: long, float, string"""
    r = np.random.default_rng(seed)
    sch = StructType([StructField("id", LongType()), StructField("x", FloatType()), StructField("s", StringType())])
    rows = [(int(r.integers(-2**40, 2**40)), float(np.float32(r.standard_normal())),
             "".join(chr(97 + int(c)) for c in r.integers(0, 26, int(r.integers(str_len[0], str_len[1] + 1))))) for _ in range(n)]
    return sch, A.columns_from_rows(sch, rows)


def _alternate(oracle, jobs, rounds, what):
    """jobs: [(name, encoder, schema, columns)] -- encode them in turn, `rounds` times over, each against the oracle"""
    wants = {name: _encode(oracle, sch, cols).tobytes() for name, _, sch, cols in jobs}
    for k in range(rounds):
        for name, enc, sch, cols in jobs:
            if k == rounds - 1 and name != jobs[0][0]:
                break                                        # the sequence ends on the first job: W, N, W, N, W
            assert enc.encode(cols) == wants[name], f"{what}: {name}, round {k + 1}"


@pytest.mark.parametrize("fused", [False, True])
def test_live_encoders_do_not_lower_each_others_shared_memory(native, oracle, monkeypatch, fused):
    """W (cfg2 rows: 64 fields, about 77 KiB for the tile emit) and N (3 scalars, about 9 KiB) alive together: W, N, W, N, W.
    With TFR_FUSED_ENCODE=1 the later calls take the one-kernel encoder, whose launch needs the same care."""
    from oracle.corpus import cfg2_columns
    if fused:
        monkeypatch.setenv("TFR_FUSED_ENCODE", "1")
    sch_w, cols_w = cfg2_columns(1000, seed=3)
    sch_n, cols_n = _narrow(1000, seed=4)
    ew, en = native.Encoder(sch_w), native.Encoder(sch_n)
    try:
        _alternate(oracle, [("W", ew, sch_w, cols_w), ("N", en, sch_n, cols_n)], 4 if fused else 3, f"fused={fused}")
    finally:
        ew.close(); en.close()
    # one schema, two encoders: the slot size (and with it the shared memory) differs by the data alone
    sch_l, cols_l = _narrow(700, seed=5, str_len=(1500, 1500))
    sch_s, cols_s = _narrow(700, seed=6, str_len=(10, 10))
    el, es = native.Encoder(sch_l), native.Encoder(sch_s)
    try:
        _alternate(oracle, [("1500-byte strings", el, sch_l, cols_l), ("10-byte strings", es, sch_s, cols_s)], 4 if fused else 3,
                   f"fused={fused}, one schema")
    finally:
        el.close(); es.close()


def _frame_payloads(payloads):
    from oracle import pyref
    return np.frombuffer(b"".join(pyref.frame_fast(p) for p in payloads), dtype=np.uint8)


def test_live_decoders_interleaved(native, oracle):
    """four decoders alive at once, steady-state submits interleaved across them: cfg2 records (12 + 3 warp tiles), 220-byte
    string records (4 + 1 warp tiles, eight per SM), and ByteArray records of 5 KiB (one bytes tile of about 200 KiB per SM)
    and of 1 KiB (the same kernel instantiation with a fifth of that shared memory)"""
    from oracle.corpus import cfg2_columns

    def small_strings(n, seed):
        r = np.random.default_rng(seed)
        sch = StructType([StructField("k", LongType()), StructField("s", StringType())])
        rows = [(int(r.integers(0, 2**31)), "".join(chr(97 + int(c)) for c in r.integers(0, 26, int(r.integers(195, 206))))) for _ in range(n)]
        return sch, A.columns_from_rows(sch, rows)

    def blobs(n, lo, hi, seed):
        r = np.random.default_rng(seed)
        return _frame_payloads([r.integers(0, 256, int(s), dtype=np.uint8).tobytes() for s in r.integers(lo, hi, n)])

    jobs = []                                   # (name, schema, record type, [data of each batch])
    sch, _ = cfg2_columns(1, seed=1)
    jobs.append(("cfg2", sch, 0, [_encode(oracle, sch, cfg2_columns(6000 + 13 * i, seed=70 + i)[1]) for i in range(3)]))
    sch, _ = small_strings(1, 0)
    jobs.append(("220-byte records", sch, 0, [_encode(oracle, sch, small_strings(20000 + 11 * i, 80 + i)[1]) for i in range(3)]))
    jobs.append(("ByteArray 5 KiB", byte_array_schema(), 2, [blobs(1500 + 7 * i, 4600, 5600, 90 + i) for i in range(3)]))
    jobs.append(("ByteArray 1 KiB", byte_array_schema(), 2, [blobs(6000 + 7 * i, 900, 1100, 95 + i) for i in range(3)]))
    wants = {(name, i): oracle.decode(d, sch, rt) for name, sch, rt, datas in jobs for i, d in enumerate(datas)}
    devs = {(name, i): _cuda(d) for name, sch, rt, datas in jobs for i, d in enumerate(datas)}
    decs = {name: native.Decoder(sch, rt) for name, sch, rt, _ in jobs}
    try:
        for name, sch, rt, _ in jobs:                              # learn, then one pipelined batch each
            b, _ = decs[name].decode(devs[(name, 0)]); _check(b, wants[(name, 0)], sch, f"{name}: learning batch"); b.release()
        for rnd in range(4):
            inflight = []
            for name, sch, rt, _ in jobs:
                for i in (1, 2):
                    inflight.append((name, sch, i, decs[name].submit(devs[(name, (i + rnd) % 3)])))
            for name, sch, i, b in inflight:
                _check(b, wants[(name, (i + rnd) % 3)], sch, f"{name}: round {rnd + 1}, batch {(i + rnd) % 3}"); b.release()
        for name, _, _, _ in jobs:
            st = decs[name].stats()
            assert st["speculative_submits"] >= 6 and st["speculative_redone"] == 0 and st["general_path_batches"] == 0, (name, st)
    finally:
        for d in decs.values():
            d.close()


_THREADS_SCRIPT = r'''
import sys, threading, traceback
ROOT, TESTS = sys.argv[1], sys.argv[2]
sys.path[:0] = [ROOT, TESTS]
import numpy as np
import torch
from oracle import oracle
from oracle.corpus import cfg2_columns, mixed_columns
from spark_tfrecord_b200 import _native
from util import assert_columns_equal

N_THREADS = 8
oracle.build()


def corpus(k, i):
    """thread k's i-th batch: a schema and record size of its own (cfg2-like records of 0.1 to 4 KB, or ragged mixed rows)"""
    if k % 4 == 3:
        return mixed_columns(2500 + 11 * i, seed=100 * k + i, null_frac=0.05 * (k // 4 + 1))
    return cfg2_columns(3000 + 7 * i, seed=100 * k + i, n_int=4 + 4 * k, n_float=2 + 2 * k, n_bytes=1 + k, float_len=1 + k,
                        bytes_len=8 + 60 * k)


jobs = []
for k in range(N_THREADS):
    datas, wants, cols0, sch = [], [], None, None
    for i in range(3):
        sch, cols = corpus(k, i)
        data, rc, _ = oracle.encode(cols, sch)
        assert rc == 0
        datas.append(np.frombuffer(data, dtype=np.uint8))
        wants.append(oracle.decode(datas[-1], sch))
        cols0 = cols0 or cols
    jobs.append(dict(sch=sch, datas=datas, devs=[torch.from_numpy(d.copy()).cuda() for d in datas], wants=wants, cols0=cols0,
                     dec=_native.Decoder(sch), enc=_native.Encoder(sch)))
torch.cuda.synchronize()
barrier = threading.Barrier(N_THREADS)
errors = []


def check(b, want, sch, what):
    for key in ("error_code", "error_row", "n_rows", "consumed_bytes"):
        assert b.info[key] == want.info[key], (what, key, b.info, want.info)
    assert_columns_equal(b.to_host(), want.columns, sch.names, what)


def work(k):
    try:
        J = jobs[k]
        dec, enc, sch = J["dec"], J["enc"], J["sch"]
        barrier.wait()
        b, _ = dec.decode(J["devs"][0])
        check(b, J["wants"][0], sch, f"thread {k}: learning decode"); b.release()
        inflight = [(i, dec.submit(J["devs"][i])) for i in (1, 2, 1, 2)]
        for i, b in inflight:
            check(b, J["wants"][i], sch, f"thread {k}: pipelined batch {i}"); b.release()
        b = dec.submit(J["datas"][0])
        check(b, J["wants"][0], sch, f"thread {k}: host-input batch"); b.release()
        got = enc.encode(J["cols0"])
        assert got == J["datas"][0].tobytes(), f"thread {k}: encoded bytes differ from the oracle writer"
    except BaseException as e:          # noqa: BLE001
        errors.append((k, e, traceback.format_exc()))
        barrier.abort()


threads = [threading.Thread(target=work, args=(k,)) for k in range(N_THREADS)]
for t in threads:
    t.start()
for t in threads:
    t.join()
for J in jobs:
    J["dec"].close(); J["enc"].close()
if errors:
    errors.sort(key=lambda x: isinstance(x[1], threading.BrokenBarrierError))
    k, e, tb = errors[0]
    print(f"thread {k} failed ({len(errors)} thread(s) in all):\n{tb}", file=sys.stderr)
    sys.exit(1)
print("threads ok")
'''


def test_eight_threads_first_launches_coincide(tmp_path):
    """eight threads of one fresh process, each with its own decoder and encoder (a different schema and record size per
    thread), make their first launches together behind a barrier; everything they decode and encode is checked against
    results the oracle computed before the barrier.  A fresh interpreter: the library's per-process state has not been
    warmed by earlier tests."""
    script = tmp_path / "threads.py"
    script.write_text(textwrap.dedent(_THREADS_SCRIPT))
    r = subprocess.run([sys.executable, str(script), ROOT, os.path.join(ROOT, "tests")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "threads ok" in r.stdout, f"exit {r.returncode}\n{r.stdout[-4000:]}\n{r.stderr[-8000:]}"


# ------------------------------------------------------------------------------------------------------------------------
# C. input lifetimes
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mixed_256mib(oracle):
    """about 256 MiB of ragged rows (strings, binary, arrays of every type, nulls), written by the oracle"""
    from oracle.corpus import mixed_columns
    sch, cols = mixed_columns(2000, seed=17)
    per_row = len(_encode(oracle, sch, cols)) / 2000
    n = int((256 << 20) / per_row)
    sch, cols = mixed_columns(n, seed=18)
    data = _encode(oracle, sch, cols)
    return sch, data, oracle.decode(data, sch)


def _overwritten_after_decode(dec, src):
    """decode from the device tensor `src`, overwrite it on torch's stream the moment tfr_decode returns, then read the rows"""
    import torch
    b, _ = dec.decode(src)
    src.fill_(0xA5)
    torch.cuda.synchronize()
    return b


def test_decode_is_complete_when_it_returns(native, oracle, mixed_256mib):
    """tfr_decode returns when the batch is complete: the caller may reuse the device buffer at once.  A fresh decoder's
    first batch (count mode), a batch that takes the general kernels, a steady-state batch redone after a flipped payload
    bit, and a non-contiguous tensor whose contiguous copy dies with the call."""
    import torch
    from oracle import pyref
    sch, data, want = mixed_256mib
    assert want.info["error_code"] == 0
    # a non-canonical record (the `features` field repeated, empty) in the middle: the general path
    offs = record_offsets(data)
    k = len(offs) // 2
    rec = bytes(data[offs[k] + 12: offs[k + 1] - 4])
    odd = np.concatenate([data[: offs[k]], np.frombuffer(pyref.frame_fast(rec + b"\x0a\x00"), np.uint8), data[offs[k + 1]:]])
    want_odd = oracle.decode(odd, sch)
    assert want_odd.info["error_code"] == 0 and want_odd.n_rows == want.n_rows
    # a flipped payload bit in the last tenth
    j = len(offs) * 9 // 10
    bad = data.copy()
    bad[offs[j] + 20] ^= 0x10
    want_bad = oracle.decode(bad, sch)
    assert want_bad.info["error_code"] == A.TFR_E_CRC_DATA

    dec = native.Decoder(sch)
    try:
        b = _overwritten_after_decode(dec, _cuda(data))
        assert dec.stats()["count_mode_batches"] == 1, dec.stats()
        _check(b, want, sch, "fresh decoder (count mode), input overwritten after tfr_decode"); b.release()
    finally:
        dec.close()
    dec = native.Decoder(sch)
    try:
        b = _overwritten_after_decode(dec, _cuda(odd))
        assert dec.stats()["general_path_batches"] == 1, dec.stats()
        _check(b, want_odd, sch, "general path, input overwritten after tfr_decode"); b.release()
    finally:
        dec.close()
    dec = native.Decoder(sch)
    try:
        b, _ = dec.decode(_cuda(data)); b.release()
        b = dec.submit(_cuda(data)); _check(b, want, sch, "steady state"); b.release()
        s0 = dec.stats()
        b = _overwritten_after_decode(dec, _cuda(bad))
        s1 = dec.stats()
        assert s1["speculative_submits"] == s0["speculative_submits"] + 1 and s1["speculative_redone"] == s0["speculative_redone"] + 1, (s0, s1)
        _check(b, want_bad, sch, "steady-state batch redone inside tfr_decode, input overwritten after it"); b.release()
    finally:
        dec.close()
    # a strided view: Decoder.decode hands the library a contiguous copy that is freed when the call returns; the caching
    # allocator gives its block to the next tensor of that size on the same stream
    dec = native.Decoder(sch)
    try:
        wide = torch.empty((len(data), 2), dtype=torch.uint8, device="cuda")
        wide[:, 0] = _cuda(data)
        view = wide[:, 0]
        assert not view.is_contiguous()
        b, _ = dec.decode(view)
        scribble = torch.full((len(data),), 0xA5, dtype=torch.uint8, device="cuda")
        wide.fill_(0x5A)
        torch.cuda.synchronize()
        _check(b, want, sch, "non-contiguous input, its copy's memory reused after tfr_decode"); b.release()
        del scribble
    finally:
        dec.close()


def test_host_input_redo_finishes_before_its_lane_is_refilled(native, oracle):
    """pageable host input in the steady state goes through the lanes round-robin.  Batch A has a flipped payload bit in its
    last tenth and is held unresolved; the next TFR_LANES batches (other contents) bring the pipeline back to A's lane, whose
    reuse redoes A from the lane's device copy first -- that redo must be over before the lane's copy-in overwrites it."""
    from oracle.corpus import mixed_columns
    lanes = native.Decoder.num_staging_slots()
    sch, _ = mixed_columns(1, seed=1)
    datas = [_encode(oracle, sch, mixed_columns(60000 + 17 * i, seed=200 + i)[1]) for i in range(lanes + 2)]
    offs = record_offsets(datas[1])
    bad = datas[1].copy()
    bad[offs[len(offs) * 19 // 20] + 40] ^= 0x04
    datas[1] = bad
    wants = [oracle.decode(d, sch) for d in datas]
    assert wants[1].info["error_code"] == A.TFR_E_CRC_DATA
    dec = native.Decoder(sch)
    try:
        b, _ = dec.decode(datas[0]); _check(b, wants[0], sch, "learning batch"); b.release()
        b = dec.submit(datas[0]); _check(b, wants[0], sch, "steady state"); b.release()
        s0 = dec.stats()
        held = [(1, dec.submit(datas[1]))]                      # A: not resolved until its lane comes round again
        for i in range(2, lanes + 2):
            held.append((i, dec.submit(datas[i])))
        s1 = dec.stats()
        assert s1["speculative_submits"] == s0["speculative_submits"] + lanes + 1, (s0, s1)
        assert s1["speculative_redone"] == s0["speculative_redone"] + 1, ("A was redone when its lane was reused", s0, s1)
        for i, b in held:
            _check(b, wants[i], sch, f"host-input batch {i}" + (" (redone from its lane)" if i == 1 else "")); b.release()
    finally:
        dec.close()


def _device_column(hc, rng, keep):
    """a tfr_column over device memory holding `hc` the way a slice of a larger Arrow array does: every offsets array starts
    at k > 0 (junk entries in front of the ones it uses), byte values start at an odd address, scalar values at row k of
    their buffer"""
    import torch
    from spark_tfrecord_b200._cabi import tfr_column

    def dev(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        keep.append(t)
        return t

    c = hc.to_ctypes()
    t = tfr_column()
    for f, _ in tfr_column._fields_:
        setattr(t, f, getattr(c, f))
    if hc.validity is not None:
        t.validity = dev(hc.validity).data_ptr()
    shift = int(rng.integers(1, 40))                   # junk entries in front of the current level's array
    for lvl, o in enumerate(hc.offsets):
        k_next = int(rng.integers(1, 40))               # junk in front of what this level points into
        a = np.concatenate([rng.integers(-1000, 1000, shift).astype(np.int32), o.astype(np.int32) + k_next])
        # the outermost offsets begin at the slice's first row; a child array is not sliced, its parent's offsets skip the junk
        t.offsets[lvl] = dev(a).data_ptr() + (4 * shift if lvl == 0 else 0)
        shift = k_next
    vals = hc.values.view(np.uint8)
    width = hc.values.dtype.itemsize
    if hc.offsets:                                     # the innermost offsets index values[shift:]
        front = shift * width
    else:                                              # scalars: a sliced array's values begin at row k of the buffer
        front = int(rng.integers(1, 40)) * width
    odd = 1 if width == 1 else 0
    buf = dev(np.concatenate([np.zeros(odd, np.uint8), rng.integers(0, 256, front, dtype=np.uint8), vals]))
    t.values = buf.data_ptr() + odd + (0 if hc.offsets else front)
    if width == 1:
        assert t.values % 2 == 1 or not hc.offsets
    return t


def test_encode_from_device_columns(native, oracle, monkeypatch):
    """tfr_encode with columns_on_device=1 for Example and SequenceExample: the columns of a decoded batch re-encode to the
    file they came from; columns that are slices of larger device arrays (offsets starting at k > 0, string bytes at odd
    addresses) encode to the oracle's bytes for the same rows"""
    import torch
    from test_gpu_fuzz import _schema, _batch
    from oracle.corpus import cfg4_columns, mixed_columns
    for seed in range(6):
        rt = seed % 2
        rng = np.random.default_rng(40_000 + seed)
        sch, gens = _schema(rng, seq=bool(rt))
        data = _batch(oracle, sch, gens, int(rng.choice([33, 700, 3000])), 41_000 + seed, rt)
        dec, enc = native.Decoder(sch, rt), native.Encoder(sch, rt)
        try:
            b, _ = dec.decode(_cuda(data))
            assert b.info["error_code"] == 0
            cols = b.device_columns()
            for it in range(2):
                enc.encode_columns(cols, on_device=True)
                assert enc.result_host() == data.tobytes(), f"seed {seed} (record type {rt}): decoded columns re-encoded, call {it + 1}"
            b.release()
        finally:
            dec.close(); enc.close()
    rng = np.random.default_rng(7)
    for rt, (sch, hcols) in ((0, mixed_columns(3000, seed=31)), (1, cfg4_columns(800, seed=32, mean_steps=6))):
        want = _encode(oracle, sch, hcols, rt).tobytes()
        keep = []
        dcols = [_device_column(c, rng, keep) for c in hcols]
        torch.cuda.synchronize()
        enc = native.Encoder(sch, rt)
        try:
            for it in range(3):
                if it == 2:
                    monkeypatch.setenv("TFR_FUSED_ENCODE", "1")
                enc.encode_columns(dcols, on_device=True)
                assert enc.result_host() == want, f"record type {rt}: sliced device columns, call {it + 1}"
        finally:
            monkeypatch.delenv("TFR_FUSED_ENCODE", raising=False)
            enc.close()
