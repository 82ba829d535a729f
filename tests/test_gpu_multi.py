"""Multi-GPU paths on real GPUs (skipped on a 1-GPU box): key-range sharded compaction of one tablet
through ybgpu_compact_range_sharded (BASELINE config 5, scaled), and the key-range filter on a single GPU."""
import importlib
import os
import socket
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _ranges_worker(rank, world, uid, q, rounds, colocated):
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import oracle_py as o
    pkg = importlib.import_module("yugabyte-db_b200")
    comm = pkg.RangeComm(uid, rank, world, rank)
    if colocated:
        import workloads as w
        runs = w.random_cotable_runs(77, n_runs=6, n_tables=3, rows_per_table=400, colocated=True)
        ssts = [o.Sst.build(r, o.TableOptions(block_size=1024)) for r in runs if r]
        kw = dict(bottommost=True, cutoff_ht=o.ht_from_micros(w.BASE_US + 75, 1), other_min_ht=o.HT_MAX)
        bs = 1024
    else:
        cfg = o.GenConfig(seed=31, num_rows=60000, cols=2, versions=3, num_files=8, value_len=120, tombstone_per_1024=40)
        ssts = o.Sst.generate_all(cfg, o.TableOptions(block_size=8192))
        kw = dict(cutoff_ht=o.ht_from_micros(cfg.base_micros + 1500))
        bs = 8192
    mine = [(s.meta_view().copy(), s.data_view().copy()) for f, s in enumerate(ssts) if f % world == rank]
    data, meta, res, total = comm.compact(mine, rounds=rounds, chunk_bytes=1 << 20, block_size=bs, filter_policy=1, filter_block_size=4096,
                                          out_bytes_hint=sum(len(s.data) for s in ssts) + (1 << 20), **kw)
    piece = o.Sst.from_bytes(meta.tobytes(), data.tobytes()).read_all() if res.data_len else []
    q.put((rank, piece, int(total.num_input_records), int(res.sent_to_peers_bytes), int(res.received_bytes), res.lower, res.upper,
           res.smallest, res.largest, int(res.num_ranges)))
    comm.close()


@pytest.mark.parametrize("rounds,colocated", [(1, False), (3, False), (2, True)])
def test_key_range_sharded_compaction_two_gpus(rounds, colocated):
    """BASELINE config 5 (scaled) through the PRODUCT path: ybgpu_compact_range_sharded — C++ over NCCL behind the C ABI,
    splitters agreed through the communicator, block slices exchanged with chunked grouped ncclSend / ncclRecv, every
    rank compacting its key range(s). The ranks' tables, in rank order, hold exactly the single-job KV stream; with
    rounds > 1 a rank's table is assembled from several sequential sub-range jobs; ranges that start inside a
    colocated table receive that table's tombstones."""
    pkg = importlib.import_module("yugabyte-db_b200")
    if pkg.device_count() < 2:                     # checked without importing torch (cold import is slow)
        pytest.skip("needs 2 GPUs")
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import multiprocessing as mp
    import oracle_py as o
    world = 2
    uid = pkg.range_comm_unique_id()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_ranges_worker, args=(r, world, uid, q, rounds, colocated)) for r in range(world)]
    for p_ in procs:
        p_.start()
    got = sorted(q.get(timeout=300) for _ in range(world))
    for p_ in procs:
        p_.join(timeout=60)
        assert p_.exitcode == 0
    if colocated:
        import workloads as w
        runs = w.random_cotable_runs(77, n_runs=6, n_tables=3, rows_per_table=400, colocated=True)
        ssts = [o.Sst.build(r, o.TableOptions(block_size=1024)) for r in runs if r]
        exp = o.compact(ssts, o.CompactionParams(bottommost=True, cutoff_ht=o.ht_from_micros(w.BASE_US + 75, 1), other_min_ht=o.HT_MAX),
                        o.TableOptions(block_size=1024, filter_policy=1, filter_block_size=4096))
    else:
        cfg = o.GenConfig(seed=31, num_rows=60000, cols=2, versions=3, num_files=8, value_len=120, tombstone_per_1024=40)
        ssts = o.Sst.generate_all(cfg, o.TableOptions(block_size=8192))
        exp = o.compact(ssts, o.CompactionParams(cutoff_ht=o.ht_from_micros(cfg.base_micros + 1500)),
                        o.TableOptions(block_size=8192, filter_policy=1, filter_block_size=4096))
    ekv = exp.kv_list()
    assert [kv for g in got for kv in g[1]] == ekv
    assert sum(g[2] for g in got) == exp.stats.num_input_records
    assert all(len(g[1]) > 0 for g in got) and all(g[3] > 0 for g in got)          # both ranks work, bytes crossed NVLink
    assert got[0][5] == b"" and got[0][6] == got[1][5] and got[1][6] == b""           # [lower, upper) tile the key space
    assert got[0][7] == ekv[0][0] and got[1][8] == ekv[-1][0]
    assert got[0][9] == world * rounds


def test_key_range_filter_single_gpu():
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import oracle_py as o
    pkg = importlib.import_module("yugabyte-db_b200")
    sh = importlib.import_module("yugabyte-db_b200.sharding")
    cfg = o.GenConfig(seed=13, num_rows=20000, cols=2, versions=3, num_files=4, value_len=60, tombstone_per_1024=30)
    ssts = o.Sst.generate_all(cfg, o.TableOptions(block_size=4096))
    cutoff = o.ht_from_micros(cfg.base_micros + 1500)
    exp = o.compact(ssts, o.CompactionParams(cutoff_ht=cutoff), o.TableOptions(block_size=4096))
    keys = sorted(k[:-8] for s in ssts for k, _ in s.read_all())
    splitters = [keys[len(keys) // 3][:32], keys[2 * len(keys) // 3][:32]]       # DocKey (32 B) aligned
    out, n_in = [], 0
    for r in range(3):
        lo, hi = sh.range_of_rank(splitters, r)
        job = pkg.GpuCompactionJob(cutoff_ht=cutoff, block_size=4096, largest_user_key=keys[-1], range_lower=lo, range_upper=hi)
        for s in ssts:
            job.add_input_sst(s.meta_view(), s.data_view())
        st = job.run()
        n_in += st.num_input_records
        out += job.kv_list()
    assert out == exp.kv_list()
    assert n_in == exp.stats.num_input_records
