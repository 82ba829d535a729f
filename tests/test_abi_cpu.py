"""CPU-side checks of the product library: it loads, exports every symbol include/*.h declares,
refuses to run without a GPU (no CPU fallback), and its host-side SST writer/reader agree with the
oracle byte for byte."""
import importlib
import os
import random
import re

import numpy as np
import pytest

import oracle_py as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return importlib.import_module("yugabyte-db_b200")


def test_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, "include", "ybgpu_compaction.h")).read()
    names = set(re.findall(r"\b(ybgpu_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 25
    L = pkg.lib()
    for n in sorted(names):
        assert hasattr(L, n), "libybgpu.so does not export %s" % n


def test_status_codes_are_the_reference_numbers(pkg):
    """ybgpu_status values must equal yb::Status::Code (util/status_codes.h) because the adapter casts them; the
    committed table was extracted from the reference header (tests/golden/extract_status_codes.py)."""
    import json
    tab = json.load(open(os.path.join(ROOT, "tests", "golden", "status_codes_table.json")))["codes"]
    hdr = open(os.path.join(ROOT, "include", "ybgpu_compaction.h")).read()
    enum = dict((n, int(v)) for n, v in re.findall(r"YBGPU_([A-Z_]+)\s*=\s*(\d+)", hdr.split("typedef enum ybgpu_status")[1].split("}")[0]))
    want = {"OK": "Ok", "NOT_FOUND": "NotFound", "CORRUPTION": "Corruption", "NOT_SUPPORTED": "NotSupported",
            "INVALID_ARGUMENT": "InvalidArgument", "IO_ERROR": "IOError", "RUNTIME_ERROR": "RuntimeError",
            "ILLEGAL_STATE": "IllegalState", "TRY_AGAIN": "TryAgain", "SHUTDOWN_IN_PROGRESS": "ShutdownInProgress"}
    assert set(enum) == set(want)
    for k, ref_name in want.items():
        assert enum[k] == tab[ref_name], (k, enum[k], tab[ref_name])
    adapter = open(os.path.join(ROOT, "yugabyte-db_b200", "csrc", "adapter", "gpu_compaction_job.h")).read()
    for name, v in re.findall(r"\bk(\w+) = (\d+)", adapter.split("enum Code {")[1].split("}")[0]):
        assert tab[name if name != "Ok" else "Ok"] == int(v), name
    for v, name in pkg.STATUS_NAMES.items():
        assert tab["Ok" if name == "OK" else name] == v


def test_no_cpu_fallback_without_gpu(pkg):
    if pkg.device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(pkg.YbGpuError) as e:
        pkg.GpuCompactionJob()
    assert "no CPU fallback" in str(e.value)


def _rand_kvs(rng, n, klen=(1, 40), vlen=(0, 200)):
    keys = set()
    while len(keys) < n:
        keys.add(bytes(rng.randrange(256) for _ in range(rng.randrange(*klen))))
    return [(o.ikey(k, 77 + i), bytes(rng.randrange(256) for _ in range(rng.randrange(*vlen)))) for i, k in enumerate(sorted(keys))]


@pytest.mark.parametrize("n,bs,ibs,mk", [(1, 4096, 4096, 100), (300, 512, 256, 4), (5000, 1024, 512, 8), (20000, 4096, 32768, 100)])
def test_host_table_builder_matches_oracle_bytes(pkg, n, bs, ibs, mk):
    rng = random.Random(n)
    kvs = _rand_kvs(rng, n)
    ref = o.Sst.build(kvs, o.TableOptions(block_size=bs, index_block_size=ibs, min_keys_per_index_block=mk))
    b = pkg.HostTableBuilder(block_size=bs, index_block_size=ibs, min_keys_per_index_block=mk)
    for k, v in kvs:
        b.add(k, v)
    data, meta = b.finish()
    assert data == ref.data
    assert meta == ref.meta


def test_host_table_builder_docdb_shape(pkg):
    cfg = o.GenConfig(seed=4, num_rows=3000, cols=2, versions=3, num_files=1, value_len=120)
    ref = o.Sst.generate(cfg, 0, o.TableOptions(block_size=4096, index_block_size=1024, min_keys_per_index_block=10))
    b = pkg.HostTableBuilder(block_size=4096, index_block_size=1024, min_keys_per_index_block=10)
    for k, v in ref.read_all():
        b.add(k, v)
    data, meta = b.finish()
    assert data == ref.data and meta == ref.meta


@pytest.mark.parametrize("shape", ["random", "docdb", "counter"])
def test_host_table_builder_three_shared_parts(pkg, shape):
    """kKeyDeltaEncodingThreeSharedParts through the host writer (the planner is the code the GPU
    encoder runs, compiled for the host) against the oracle's ThreeSharedPartsEncoder."""
    if shape == "random":
        kvs = _rand_kvs(random.Random(5), 4000, klen=(1, 60))
    elif shape == "docdb":
        cfg = o.GenConfig(seed=6, num_rows=2500, cols=3, versions=3, num_files=1, value_len=60, tombstone_per_1024=40)
        kvs = o.Sst.generate(cfg, 0, o.TableOptions(block_size=4096)).read_all()
    else:
        # same user-key length, consecutive sequence numbers / equal suffixes: last-component reuse and "+1"
        kvs = [(o.ikey(b"row%07d" % (i // 3) + bytes([65 + i % 3]), 1000 + (i if i % 5 else 0)), b"x" * (i % 9)) for i in range(6000)]
    topt = dict(block_size=2048, index_block_size=1024, min_keys_per_index_block=8)
    ref = o.Sst.build(kvs, o.TableOptions(key_encoding=2, **topt))
    b = pkg.HostTableBuilder(key_encoding=2, **topt)
    for k, v in kvs:
        b.add(k, v)
    data, meta = b.finish()
    assert data == ref.data
    assert meta == ref.meta
    assert [kv for kv in ref.read_all()] == kvs


@pytest.mark.parametrize("fbs,enc", [(256, 1), (4096, 2), (65536, 1)])
def test_host_table_builder_bloom_filter_blocks(pkg, fbs, enc):
    """DocKeyV3Filter fixed-size bloom blocks, filter index, metaindex entry and properties written by the
    host writer are byte-identical to the oracle's BlockBasedTableBuilder restatement."""
    cfg = o.GenConfig(seed=12, num_rows=4000, cols=2, versions=2, num_files=1, value_len=50, tombstone_per_1024=30)
    kvs = o.Sst.generate(cfg, 0, o.TableOptions(block_size=4096)).read_all()
    kvs += [(o.ikey(b"~plain-key-%d" % i, 5), b"v") for i in range(3)]           # not DocKeys: never in the filter
    topt = dict(block_size=2048, index_block_size=512, min_keys_per_index_block=6, key_encoding=enc, filter_policy=1, filter_block_size=fbs)
    ref = o.Sst.build(kvs, o.TableOptions(**topt))
    b = pkg.HostTableBuilder(**topt)
    for k, v in kvs:
        b.add(k, v)
    data, meta = b.finish()
    assert data == ref.data
    assert meta == ref.meta


def test_product_generator_matches_oracle_generator(pkg):
    """bench.py's inputs come from the product's generator; the oracle has an independent one.
    Same spec (SURVEY.md 8d) => same bytes."""
    kw = dict(seed=21, num_rows=4000, cols=2, versions=3, num_files=4, value_len=100, tombstone_per_1024=50)
    a = pkg.generate_ssts(pkg.GenConfig(**kw), block_size=4096)
    b = o.Sst.generate_all(o.GenConfig(**kw), o.TableOptions(block_size=4096))
    for x, y in zip(a, b):
        assert x.data_view().tobytes() == y.data and x.meta_view().tobytes() == y.meta
        assert x.num_entries == y.num_entries and x.raw_bytes == y.raw_bytes


def test_meta_reader_handles_and_separators(pkg):
    cfg = o.GenConfig(seed=6, num_rows=5000, cols=1, versions=2, num_files=1, value_len=50)
    sst = o.Sst.generate(cfg, 0, o.TableOptions(block_size=1024, index_block_size=512, min_keys_per_index_block=4))
    off, sz, enc = pkg.sst_block_handles(sst.meta_view())
    eo, es = sst.block_handles()
    assert enc == 1 and list(off) == list(eo) and list(sz) == list(es)
    seps = pkg.sst_separators(sst.meta_view())
    assert len(seps) == len(off)
    kvs = sst.read_all()
    # separator i is >= every key of block i and < first key of block i+1 (index_builder.cc:61-90)
    assert seps == sorted(seps, key=lambda k: (k[:-8], -int.from_bytes(k[-8:], "little")))
    assert seps[-1][:-8] >= kvs[-1][0][:-8]


@pytest.mark.parametrize("enc", [1, 2])
def test_sst_last_key_both_encodings(pkg, enc):
    """FileMetaData::largest of an input, read on the host from its last data block (the seqno-zeroing
    exception key of a compaction cut into subcompactions: db/compaction.cc:318)."""
    cfg = o.GenConfig(seed=8, num_rows=1500, cols=2, versions=3, num_files=3, value_len=40, tombstone_per_1024=60)
    for s in o.Sst.generate_all(cfg, o.TableOptions(block_size=1024)):
        kvs = s.read_all()
        sst = o.Sst.build(kvs, o.TableOptions(block_size=700, key_encoding=enc))
        assert pkg.sst_last_key(sst.meta_view(), sst.data_view()) == kvs[-1][0]
    one = o.Sst.build([(o.ikey(b"only", 9), b"v")], o.TableOptions(key_encoding=enc))
    assert pkg.sst_last_key(one.meta_view(), one.data_view()) == o.ikey(b"only", 9)


def test_plan_subcompactions_row_aligned_and_balanced(pkg):
    """GenSubcompactionBoundaries analogue (compaction_job.cc:409-519): splitters are complete DocKeys
    (no row straddles two ranges), strictly increasing, and the ranges carry similar numbers of entries."""
    cfg = o.GenConfig(seed=17, num_rows=6000, cols=3, versions=4, num_files=5, value_len=60)
    ssts = o.Sst.generate_all(cfg, o.TableOptions(block_size=2048))
    files = [(s.meta_view(), s.data_view()) for s in ssts]
    sp = pkg.plan_subcompactions(files, 6)
    assert 3 <= len(sp) <= 5 and sp == sorted(set(sp))
    users = sorted(k[:-8] for s in ssts for k, _ in s.read_all())
    rows = {u[:32] for u in users}                      # the generator's DocKeys are 32 bytes
    for s in sp:
        # no row straddles a splitter: that needs an existing row's DocKey as a proper prefix of it
        assert all(not (s != r and s.startswith(r)) for r in rows)
    assert any(len(s) == 32 and s[-2:] == b"!!" for s in sp)   # separators inside a row are cut back to its DocKey
    import bisect
    cuts = [0] + [bisect.bisect_left(users, s) for s in sp] + [len(users)]
    sizes = [b - a for a, b in zip(cuts, cuts[1:])]
    assert min(sizes) > 0.4 * len(users) / len(sizes) and max(sizes) < 2.0 * len(users) / len(sizes)
    # plain RocksDB keys: the whole user key is the row
    kvs = [(o.ikey(b"key%06d" % i, 100 + i), b"v" * 30) for i in range(20000)]
    plain = o.Sst.build(kvs, o.TableOptions(block_size=1024))
    sp2 = pkg.plan_subcompactions([(plain.meta_view(), plain.data_view())], 4, docdb_keys=False)
    assert len(sp2) == 3 and sp2 == sorted(sp2)
    assert pkg.plan_subcompactions(files, 1) == []
    # bench shape: one entry per row, so FindShortestSeparator shortens every index key to a string that
    # is no DocKey — such a separator is used whole (it cannot have a complete DocKey as a prefix)
    cfg1 = o.GenConfig(seed=3, num_rows=60000, cols=1, versions=1, num_files=4, value_len=40)
    ssts1 = o.Sst.generate_all(cfg1, o.TableOptions(block_size=8192))
    sp3 = pkg.plan_subcompactions([(s.meta_view(), s.data_view()) for s in ssts1], 8)
    assert len(sp3) == 7 and sp3 == sorted(set(sp3))
    users1 = sorted(k[:-8] for s in ssts1 for k, _ in s.read_all())
    rows1 = {u[:32] for u in users1}
    for s in sp3:
        assert all(not (s != r and s.startswith(r)) for r in rows1)
    cuts = [0] + [bisect.bisect_left(users1, s) for s in sp3] + [len(users1)]
    sizes = [b - a for a, b in zip(cuts, cuts[1:])]
    assert min(sizes) > 0.6 * len(users1) / 8 and max(sizes) < 1.5 * len(users1) / 8


def test_compact_files_fails_loudly_without_gpu(pkg):
    """The subcompaction entry point plans on the host but never compacts there: without a CUDA device
    it fails like ybgpu_job_create does."""
    if pkg.device_count() > 0:
        pytest.skip("GPU present")
    cfg = o.GenConfig(seed=5, num_rows=500, cols=2, versions=2, num_files=2, value_len=30)
    ssts = o.Sst.generate_all(cfg, o.TableOptions(block_size=1024))
    with pytest.raises(pkg.YbGpuError) as e:
        pkg.compact_files([(s.meta_view(), s.data_view()) for s in ssts], max_subcompactions=3, max_in_flight=2)
    assert "no CPU fallback" in str(e.value) and e.value.status_name == "RuntimeError"
    with pytest.raises(pkg.YbGpuError) as e:      # range bounds belong to the planner
        pkg.compact_files([(s.meta_view(), s.data_view()) for s in ssts], max_subcompactions=3, range_lower=b"x")
    assert e.value.status_name == "InvalidArgument"


@pytest.mark.parametrize("enc,with_filter", [(1, True), (2, True), (1, False)])
def test_sst_concat_meta_builds_one_valid_table(pkg, enc, with_filter):
    """ybgpu_sst_concat_meta: the key-disjoint range outputs of one compaction (here: the oracle's
    compaction of each key range — byte-identical to what ybgpu_compact_files returns per range, see
    test_subcompactions_pipelined) become ONE split SST. The oracle's independent reader must find every
    key/value of the single-pass compaction in it, walk the rebased multi-level index, and every key's
    bloom filter key must hit the filter block the filter index routes it to."""
    import bisect
    import test_oracle_bloom as ob
    cfg = o.GenConfig(seed=29, num_rows=7000, cols=2, versions=3, num_files=5, value_len=70, tombstone_per_1024=40)
    ssts = o.Sst.generate_all(cfg, o.TableOptions(block_size=2048))
    cutoff = o.ht_from_micros(cfg.base_micros + 1500)
    topt = dict(block_size=2048, index_block_size=512, min_keys_per_index_block=4, key_encoding=enc,
                filter_policy=int(with_filter), filter_block_size=1024)
    exp = o.compact(ssts, o.CompactionParams(cutoff_ht=cutoff), o.TableOptions(**topt))
    splitters = pkg.plan_subcompactions([(s.meta_view(), s.data_view()) for s in ssts], 6)
    assert len(splitters) >= 3
    all_kvs = [s.read_all() for s in ssts]
    largest = max(kvs[-1][0][:-8] for kvs in all_kvs)
    pieces, datas = [], []
    bounds = [b""] + splitters + [b""]
    for lo, hi in zip(bounds, bounds[1:]):
        part = [[kv for kv in kvs if (not lo or kv[0][:-8] >= lo) and (not hi or kv[0][:-8] < hi)] for kvs in all_kvs]
        ref = o.compact([o.Sst.build(p, o.TableOptions(block_size=2048)) for p in part if p],
                        o.CompactionParams(cutoff_ht=cutoff, largest_user_key=largest), o.TableOptions(**topt))
        sst = ref.sst()
        if sst is None:
            continue
        kvs = ref.kv_list()
        pieces.append((sst.meta_view().copy(), len(sst.data), kvs[0][0], kvs[-1][0]))
        datas.append(sst.data)
    assert len(pieces) >= 3
    meta = pkg.sst_concat_meta(pieces, block_size=2048, index_block_size=512, min_keys_per_index_block=4,
                               output_key_encoding=enc, filter_policy=int(with_filter), filter_block_size=1024)
    data = b"".join(datas)
    whole = o.Sst.from_bytes(meta, data)
    assert whole.read_all() == exp.kv_list()                 # checksums verified, index walked by the oracle's reader
    props = whole.properties()
    assert o.varint(props["rocksdb.num.entries"]) == len(exp.kv_list())
    assert o.varint(props["rocksdb.data.size"]) == len(data)
    assert o.varint(props["rocksdb.raw.key.size"]) == exp.stats.out_key_bytes
    assert o.varint(props["rocksdb.raw.value.size"]) == exp.stats.out_val_bytes
    # the product's own reader agrees on the block list
    off, sz, e2 = pkg.sst_block_handles(np.frombuffer(meta, np.uint8))
    assert e2 == enc and len(off) == o.varint(props["rocksdb.num.data.blocks"]) and int(off[-1] + sz[-1]) + 5 == len(data)
    if with_filter:
        fb = whole.filter_blocks()
        assert len(fb) == sum(len(o.Sst.from_bytes(p[0].tobytes(), d).filter_blocks()) for p, d in zip(pieces, datas))
        index_keys = [k for k, _ in fb]
        assert index_keys == sorted(index_keys)
        for k, _ in exp.kv_list()[::7]:
            fk = ob.filter_key(k[:-8])
            i = bisect.bisect_left(index_keys, fk)           # FixedSizeFilterBlockReader: first index entry >= key
            assert i < len(fb) and ob.may_match(fb[i][1], fk)
    # rejected: pieces out of order, options that do not match the pieces
    with pytest.raises(pkg.YbGpuError):
        pkg.sst_concat_meta(pieces[::-1], block_size=2048, output_key_encoding=enc, filter_policy=int(with_filter), filter_block_size=1024)
    with pytest.raises(pkg.YbGpuError):
        pkg.sst_concat_meta(pieces, block_size=2048, output_key_encoding=3 - enc, filter_policy=int(with_filter), filter_block_size=1024)


def test_ctypes_structs_match_the_header(pkg, tmp_path):
    """The Python binding mirrors the C structs by hand: sizes and the offsets of the trailing fields must
    agree with what a C compiler makes of include/ybgpu_compaction.h (ybgpu_job_options_init memsets the
    whole struct)."""
    import ctypes as C
    import subprocess
    b = importlib.import_module("yugabyte-db_b200.binding")
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\n'
                   'int main(void) { printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu\\n", sizeof(ybgpu_job_options), sizeof(ybgpu_job_stats),'
                   ' sizeof(ybgpu_sub_output), sizeof(ybgpu_sst_piece), sizeof(ybgpu_input_file), offsetof(ybgpu_job_options, yield_fn),'
                   ' offsetof(ybgpu_job_options, cuda_stream), offsetof(ybgpu_sub_output, smallest_key)); return 0; }\n'
                   % os.path.join(ROOT, "include", "ybgpu_compaction.h"))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(b.JobOptions), C.sizeof(b.JobStats), C.sizeof(b.SubOutput), C.sizeof(b.SstPiece), C.sizeof(b.InputFile),
            b.JobOptions.yield_fn.offset, b.JobOptions.cuda_stream.offset, b.SubOutput.smallest_key.offset]
    assert got == want


def test_sst_verify_blocks_detects_corruption(pkg):
    cfg = o.GenConfig(seed=9, num_rows=3000, cols=2, versions=2, num_files=1, value_len=60)
    sst = o.Sst.generate(cfg, 0, o.TableOptions(block_size=1024))
    nb = len(sst.block_handles()[0])
    assert pkg.sst_verify_blocks(sst.meta_view(), sst.data_view()) == (nb, 0)
    assert pkg.sst_verify_blocks(sst.meta_view(), sst.data_view(), stride=7) == ((nb + 6) // 7, 0)
    bad = sst.data_view().copy()
    off, sz = sst.block_handles()
    bad[int(off[3]) + 10] ^= 0x40                    # one flipped bit inside block 3
    assert pkg.sst_verify_blocks(sst.meta_view(), bad) == (nb, 1)
    assert pkg.sst_verify_blocks(sst.meta_view(), bad, stride=2) == ((nb + 1) // 2, 0)      # block 3 is not sampled
    assert pkg.sst_verify_blocks(sst.meta_view(), sst.data_view()[:int(off[-1])].copy())[1] == 1   # truncated data file: last block missing


def test_meta_reader_snappy_compressed_index_blocks(pkg):
    """Production tables are Snappy-compressed (docdb_rocksdb_util.cc:184) and index blocks go through WriteBlock like data
    blocks (block_based_table_builder.cc:586,790,823,869): the host-side reader of the metadata file must uncompress the
    multi-level index and the filter index. Same handles and separators as for the uncompressed twin of the table."""
    cfg = o.GenConfig(seed=16, num_rows=6000, cols=2, versions=2, num_files=1, value_len=40)
    kw = dict(block_size=1024, index_block_size=700, min_keys_per_index_block=4, filter_policy=1, filter_block_size=1024)
    plain = o.Sst.generate(cfg, 0, o.TableOptions(**kw))
    comp = o.Sst.build(plain.read_all(), o.TableOptions(compression=1, **kw))
    meta = comp.meta_view().tobytes()
    # the twin's index really is stored compressed: some block trailer of the metadata file carries type 1
    off, sz, enc = pkg.sst_block_handles(comp.meta_view())
    eo, es = comp.block_handles()
    assert list(off) == list(eo) and list(sz) == list(es) and len(off) > 50
    assert pkg.sst_separators(comp.meta_view()) == pkg.sst_separators(plain.meta_view())
    assert comp.read_all() == plain.read_all()
    assert len(meta) < len(plain.meta_view().tobytes())          # the index blocks shrank
    # planner and last-key helper work on it (the planner parses the metadata file; the last-key helper uncompresses the
    # last data block on the host)
    sp = pkg.plan_subcompactions([(comp.meta_view(), comp.data_view())], 4)
    assert 1 <= len(sp) <= 3 and sp == sorted(sp)
    kvs = plain.read_all()
    assert pkg.sst_last_key(comp.meta_view(), comp.data_view()) == kvs[-1][0]
    for cut in range(0, 60):                                       # a table whose LAST data block is stored compressed
        t = o.Sst.build(kvs[:len(kvs) - cut], o.TableOptions(compression=1, **kw))
        toff, tsz = t.block_handles()
        if bytes(t.data_view())[int(toff[-1]) + int(tsz[-1])] == 1:
            assert pkg.sst_last_key(t.meta_view(), t.data_view()) == kvs[len(kvs) - cut - 1][0]
            break
    else:
        raise AssertionError("no variant with a compressed last block")


def _compressible_kvs(seed, n, vmax=200):
    """Rows whose values repeat phrases (compressible), mixed with stretches of random values (blocks that stay raw)."""
    rng = random.Random(seed)
    words = [bytes(rng.randrange(32, 127) for _ in range(rng.randrange(3, 24))) for _ in range(40)]
    kvs = []
    for i in range(n):
        if (i // 500) % 4 == 3:
            v = bytes(rng.randrange(256) for _ in range(rng.randrange(1, vmax)))
        else:
            v = b" ".join(rng.choice(words) for _ in range(rng.randrange(0, vmax // 10)))
        kvs.append((o.ikey(b"user%08d/col%d" % (i // 3, i % 3), 500 + i), v))
    return kvs


@pytest.mark.parametrize("enc,filt,bs", [(1, 0, 4096), (2, 1, 2048), (1, 1, 32768)])
def test_host_table_builder_snappy_output(pkg, enc, filt, bs):
    """CompressBlock with kSnappyCompression (block_based_table_builder.cc:115-131): data blocks, index blocks and
    the filter index are stored compressed when that saves 12.5 %; the host writer and the oracle share one encoder, so
    the files are byte-identical; the oracle's reader (and so any Snappy reader) gets the same entries back."""
    kvs = _compressible_kvs(21 + enc, 6000)
    topt = dict(block_size=bs, index_block_size=1024, min_keys_per_index_block=8, key_encoding=enc, filter_policy=filt, filter_block_size=4096)
    ref = o.Sst.build(kvs, o.TableOptions(compression=1, **topt))
    plain = o.Sst.build(kvs, o.TableOptions(**topt))
    assert len(ref.data) < len(plain.data) * 0.8                   # most blocks were worth compressing ...
    b = pkg.HostTableBuilder(compression=1, **topt)
    for k, v in kvs:
        b.add(k, v)
    data, meta = b.finish()
    assert data == ref.data
    assert meta == ref.meta
    assert o.Sst.from_bytes(meta, data).read_all() == kvs
    off, sz, _ = pkg.sst_block_handles(np.frombuffer(meta, np.uint8))
    types = {data[int(a) + int(b)] for a, b in zip(off, sz)}
    assert types == {0, 1}                                          # ... and the random stretches stayed raw


@pytest.mark.parametrize("seed", range(8))
def test_host_table_builder_snappy_random_tables(pkg, seed):
    """The host writer's encoder against the oracle's over random table options and value shapes: tiny and huge blocks,
    values longer than a 64 KB fragment, long runs (chains of 64-byte copy elements), incompressible stretches."""
    rng = random.Random(1000 + seed)
    words = [bytes(rng.randrange(256) for _ in range(rng.randrange(1, 30))) for _ in range(rng.randrange(2, 40))]
    kvs = []
    for i in range(rng.randrange(50, 900)):
        shape = rng.randrange(6)
        if shape == 0:
            v = bytes(rng.randrange(256) for _ in range(rng.randrange(0, 300)))
        elif shape == 1:
            v = bytes([rng.randrange(256)]) * rng.randrange(0, 5000)
        elif shape == 2:
            v = b"".join(rng.choice(words) for _ in range(rng.randrange(0, 60)))
        elif shape == 3 and i % 40 == 0:
            v = (rng.choice(words) * 9000)[:rng.randrange(66000, 200000)]
        elif shape == 4:
            v = b""
        else:
            v = bytes(rng.choice(b"ab") for _ in range(rng.randrange(0, 400)))
        kvs.append((o.ikey(b"k%06d" % i + bytes(rng.randrange(97, 100) for _ in range(rng.randrange(0, 5))), 9000 - i), v))
    kvs.sort(key=lambda kv: (kv[0][:-8], -int.from_bytes(kv[0][-8:], "little")))
    kvs = [kv for j, kv in enumerate(kvs) if j == 0 or kvs[j - 1][0][:-8] != kv[0][:-8]]
    topt = dict(block_size=rng.choice([256, 1024, 4096, 32768, 70000]), restart_interval=rng.choice([1, 4, 16]),
                index_block_size=rng.choice([256, 4096]), min_keys_per_index_block=rng.choice([2, 100]),
                key_encoding=rng.choice([1, 2]), filter_policy=rng.randrange(2), filter_block_size=1024)
    otopt = dict(topt)
    otopt["restart"] = otopt.pop("restart_interval")
    ref = o.Sst.build(kvs, o.TableOptions(compression=1, **otopt))
    b = pkg.HostTableBuilder(compression=1, **topt)
    for k, v in kvs:
        b.add(k, v)
    data, meta = b.finish()
    assert data == ref.data and meta == ref.meta
    assert o.Sst.from_bytes(meta, data).read_all() == kvs


def test_sst_check_supported_routing_precheck(pkg):
    """Routing by job type before any upload: raw and Snappy tables are taken; a table with blocks of another
    CompressionType (here: trailers re-labelled LZ4 / ZSTD / zlib) is NotSupported with the count of such blocks; a
    handle outside the data file or an unreadable metadata file is Corruption."""
    cfg = o.GenConfig(seed=23, num_rows=3000, cols=2, versions=2, num_files=1, value_len=40)
    kvs = o.Sst.generate(cfg, 0, o.TableOptions(block_size=2048)).read_all()
    plain = o.Sst.build(kvs, o.TableOptions(block_size=2048))
    snap = o.Sst.build(kvs, o.TableOptions(block_size=2048, compression=1))
    tsp = o.Sst.build(kvs, o.TableOptions(block_size=2048, key_encoding=2))
    nb = len(plain.block_handles()[0])
    assert pkg.sst_check_supported(plain.meta_view(), plain.data_view()) == ("OK", [nb, 0, 0, 0, 0, 0, 0, 0])
    st, counts = pkg.sst_check_supported(snap.meta_view(), snap.data_view())
    assert st == "OK" and counts[1] > 0 and counts[0] + counts[1] == nb and sum(counts[2:]) == 0
    assert pkg.sst_check_supported(tsp.meta_view(), tsp.data_view())[0] == "OK"
    off, sz = plain.block_handles()
    for ctype in (2, 4, 7):                                           # kZlibCompression, kLZ4Compression, kZSTD (options.h:92-101)
        d = bytearray(plain.data)
        for b in (3, 5):
            d[int(off[b]) + int(sz[b])] = ctype
        st, counts = pkg.sst_check_supported(plain.meta_view(), bytes(d))
        assert st == "NotSupported" and counts[ctype] == 2 and counts[0] == nb - 2
    d = bytearray(plain.data)
    d[int(off[1]) + int(sz[1])] = 9
    assert pkg.sst_check_supported(plain.meta_view(), bytes(d))[0] == "Corruption"
    assert pkg.sst_check_supported(plain.meta_view(), bytes(plain.data)[:int(off[-1]) + 3])[0] == "Corruption"
    assert pkg.sst_check_supported(bytes(plain.meta)[:-7], plain.data_view())[0] == "Corruption"
