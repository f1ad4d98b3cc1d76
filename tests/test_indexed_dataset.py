"""``.idx`` / ``.bin`` indexed datasets (SURVEY §8f row 4): the on-disk format that feeds the loop.

* golden files written by the UNMODIFIED reference's writer (oracle/make_indexed_golden.py) are
  read back frame by frame and compared with what the reference's own reader returned for them
  (``manifest.json``); this repo's writer must reproduce the golden bytes exactly;
* the reference's own tests for this path (tests/test_indexed_dataset.py: header synthesised by
  hand with magic 0 / version 1, write->read round trip, reader survives pickling into another
  process) are restated against this repo's classes;
* writer bytes and reader frames on random frames are compared with what the reference's
  writer and reader produced for them (oracle/reference_cases.py);
* the batched path: ``host_fields`` (zero-copy [N, ...] tensors over the mapped .bin) gathered by
  the native host pool equals per-sample ``__getitem__`` + stacking.
"""
import io
import itertools
import json
import multiprocessing
import os
import pickle
from functools import reduce
from operator import mul

import numpy as np
import pytest
import torch

import frl_b200  # noqa: F401
from frl_b200 import _native
from frl_b200 import indexed_dataset as idm
from oracle import reference_cases as rc
from oracle.make_indexed_golden import FILES, frames_of

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "indexed")


def _reader(name, folder=GOLD):
    return idm.PosixIndexedDatasetReader(idxfile=os.path.join(folder, name + ".idx"),
                                         binfile=os.path.join(folder, name + ".bin"))


@pytest.mark.parametrize("name", sorted(FILES))
def test_reader_returns_what_the_reference_reader_returned(name):
    want = json.load(open(os.path.join(GOLD, "manifest.json")))[name]
    r = _reader(name)
    assert len(r) == want["len"] and str(r.dtype) == want["dtype"]
    assert r.framesize == want["framesize"] and [int(d) for d in r.size] == want["size"]
    frames = frames_of(name)                       # what was pushed into the reference's writer
    for i in range(len(r)):
        got = r[i]
        assert got.dtype == frames[i].dtype and got.shape == frames[i].shape
        assert np.array_equal(got, frames[i])
        assert float(np.asarray(got, dtype=np.float64).sum()) == want["frame_sums"][i]
        assert got.flags.writeable and got.base is None       # a private copy, not a view of the map
    assert np.asarray(r[0]).ravel().tolist() == want["first_frame"]
    with pytest.raises(AssertionError):
        r[len(r)]
    with pytest.raises(AssertionError):
        r[-1]


@pytest.mark.parametrize("name", sorted(FILES))
def test_writer_reproduces_the_reference_writers_bytes(name, tmp_path):
    with idm.IndexedDatasetWriterFactory.get(str(tmp_path / "f.idx"), str(tmp_path / "f.bin")) as w:
        for f in frames_of(name):
            w.push_back(f)
    for ext in (".idx", ".bin"):
        assert (tmp_path / ("f" + ext)).read_bytes() == open(os.path.join(GOLD, name + ext), "rb").read()


def test_writer_rejects_mixed_dtypes_and_empty_datasets():
    w = idm.IndexedDatasetWriter(idxfile=io.BytesIO(), binfile=io.BytesIO())
    with pytest.raises(AssertionError):
        w.flush()                                   # "Cannot write empty dataset"
    w.push_back(np.zeros(3, dtype=np.float32))
    with pytest.raises(AssertionError):
        w.push_back(np.zeros(3, dtype=np.float64))  # "Frames must all have same dtype"


# ---- the reference's own tests, restated (reference tests/test_indexed_dataset.py) -----------------

def _reference_test_content(type_name, num_frames, single_frame_dims, start_value=0):
    """Header synthesised as the reference's test does (:39-87): magic 0, version 1."""
    dtype = np.dtype(type_name)
    frame_dims = [single_frame_dims] * num_frames
    frame_ndims = [0] + [len(d) for d in frame_dims]
    frame_sizes = [0] + [reduce(mul, d, 1) for d in frame_dims]
    index = np.array([0, 1, idm.np_types.index(type_name) + 1, dtype.itemsize, num_frames,
                      sum(frame_ndims), *np.cumsum(frame_ndims), *np.cumsum(frame_sizes),
                      *itertools.chain.from_iterable(frame_dims)], dtype="int64")
    data = np.arange(0, np.cumsum(frame_sizes)[-1], dtype=dtype) + start_value
    return index, data


def _write_pair(folder, base, index, data):
    index.tofile(os.path.join(folder, base + ".idx"))
    data.tofile(os.path.join(folder, base + ".bin"))


def test_reading_element(tmp_path):                          # reference :110-139
    num_frames, dims = 10, (128, 128)
    _write_pair(str(tmp_path), "TEST_FILE", *_reference_test_content("float64", num_frames, dims))
    ds = idm.MultifieldIndexedDataset(str(tmp_path), fields=["TEST"], filenames=["TEST_FILE"])
    assert len(ds) == num_frames
    assert ds[0]["TEST"].shape == dims and ds[num_frames - 1]["TEST"].shape == dims
    n = dims[0] * dims[1]
    for i in (0, 3, num_frames - 1):
        assert np.array_equal(ds[i]["TEST"], i * n + np.arange(n, dtype=np.float64).reshape(dims))
    assert ds.get_raw_item(2)["TEST"].dtype == np.float64


def _mp_worker(blob, orig_len, frames):
    ds = pickle.loads(blob)
    assert orig_len == len(ds), "Dataset size must match original"
    for idx, frame in frames.items():
        assert np.array_equal(ds[idx], frame)


def test_multiprocessing(tmp_path):                          # reference :141-169
    _write_pair(str(tmp_path), "TEST_FILE", *_reference_test_content("float64", 10, (128, 128)))
    ds = _reader("TEST_FILE", str(tmp_path))
    frames = {i: ds[i] for i in (0, len(ds) - 2)}
    blob = pickle.dumps(ds)                                   # the map itself is not pickled
    assert len(blob) < 4096
    p = multiprocessing.get_context("spawn").Process(target=_mp_worker, args=(blob, len(ds), frames))
    p.start()
    p.join()
    assert p.exitcode == 0


def test_write_read(tmp_path):                               # reference :172-187
    data1 = np.arange(100).reshape(10, 5, 2)
    data2 = data1 + 1000
    idx, binf = str(tmp_path / "dataset.idx"), str(tmp_path / "dataset.bin")
    with idm.IndexedDatasetWriterFactory.get(idxfile=idx, binfile=binf) as w:
        w.push_back(data1)
        w.push_back(data2)
    r = idm.PosixIndexedDatasetReader(idxfile=idx, binfile=binf)
    assert np.array_equal(data1, r[0]) and np.array_equal(data2, r[1])


def test_multifield_dataset_checks_lengths(tmp_path):
    idm.write_fields(str(tmp_path), {"a": np.zeros((4, 3), np.float32), "b": np.zeros((5, 2), np.float32)})
    with pytest.raises(AssertionError, match="should have same number of samples"):
        idm.MultifieldIndexedDataset(str(tmp_path), fields=["a", "b"], filenames=["a", "b"])
    with pytest.raises(AssertionError):
        idm.MultifieldIndexedDataset(str(tmp_path), fields=["a"], filenames=["a", "b"])


def test_malformed_index_files_are_rejected(tmp_path):
    good = np.fromfile(os.path.join(GOLD, "pose.idx"), dtype="int64")
    r = idm.IndexedDatasetReader()
    with pytest.raises(ValueError, match="too short"):
        r._init_from_index_data(good[:4])
    with pytest.raises(ValueError, match="truncated"):
        r._init_from_index_data(good[:-3])
    bad = good.copy()
    bad[2] = 8                                               # np_types[7] is None
    with pytest.raises(AssertionError, match="unrecognized type"):
        r._init_from_index_data(bad)
    bad = good.copy()
    bad[3] = 2                                               # itemsize does not match the dtype
    with pytest.raises(AssertionError):
        r._init_from_index_data(bad)


# ---- against what the reference's writer and reader did (oracle/reference_cases.py) ----------------

def test_writer_and_reader_match_the_live_reference(tmp_path):
    want = rc.load("indexed_writer_reader")
    cases = rc.indexed_frames()
    assert len(want) == len(cases)
    for (dt, shape, frames), ref in zip(cases, want):
        mine_i, mine_b = rc.write_indexed(idm.IndexedDatasetWriter, frames)
        assert mine_i == bytes(ref["idx"].tolist()) and mine_b == bytes(ref["bin"].tolist()), (dt, shape)
        idx, binf = str(tmp_path / "x.idx"), str(tmp_path / "x.bin")
        open(idx, "wb").write(mine_i)
        open(binf, "wb").write(mine_b)
        mine = idm.PosixIndexedDatasetReader(idxfile=idx, binfile=binf)
        assert len(mine) == ref["len"] == len(frames)
        assert mine.framesize == ref["framesize"] and mine.dtype == np.dtype(ref["dtype"])
        for i in range(len(frames)):
            a, b = mine[i], ref["frames"][i].numpy()
            assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b)


# ---- batched access: mapped .bin -> native host pool ---------------------------------------------

def test_host_fields_gathered_by_the_pool_equal_per_sample_reads(tmp_path):
    rs = np.random.RandomState(3)
    n = 257
    fields = {"img": (rs.rand(n, 3, 16, 16) * 255).astype(np.uint8),
              "pose": rs.randn(n, 6).astype(np.float32),
              "label": rs.randint(0, 10, size=(n, 1)).astype(np.int64)}
    idm.write_fields(str(tmp_path), fields)
    ds = idm.MultifieldIndexedDataset(str(tmp_path), fields=list(fields), filenames=list(fields))
    host = ds.host_fields
    assert set(host) == set(fields)
    pool = _native.HostGatherPool(3)
    idx = torch.randperm(n)[:100].contiguous()
    for name, t in host.items():
        assert t.shape == fields[name].shape and not t.is_pinned()
        assert np.array_equal(t.numpy(), fields[name])                       # zero-copy view of the file
        out = torch.zeros((100,) + tuple(t.shape[1:]), dtype=t.dtype)
        pool.wait(pool.submit(t, idx, out))
        want = np.stack([ds[int(i)][name] for i in idx])                     # the per-sample path
        assert np.array_equal(out.numpy(), want)
    pool.close()


def test_batched_access_refuses_ragged_files(tmp_path):
    idx, binf = str(tmp_path / "r.idx"), str(tmp_path / "r.bin")
    with idm.IndexedDatasetWriterFactory.get(idx, binf) as w:
        w.push_back(np.zeros((2, 3), np.float32))
        w.push_back(np.zeros((4, 3), np.float32))
    r = idm.PosixIndexedDatasetReader(idxfile=idx, binfile=binf)
    assert len(r) == 2 and r[0].shape == (2, 3)               # per-sample reads keep working (frame-0 shape)
    with pytest.raises(ValueError, match="fixed-size frames"):
        r.frames_tensor()


# ---- Concat / Subset containers over indexed datasets (reference dataset.py:518-552) ---------------

def test_concat_and_subset_containers_match_the_live_reference(tmp_path):
    import frl_b200.storage_layers.dataset as my_ds
    ref = rc.load("concat_subset")
    rc.write_concat_parts(str(tmp_path))
    parts = [idm.MultifieldIndexedDataset(str(tmp_path / ("part%d" % k)), fields=["a", "b"], filenames=["a", "b"])
             for k in range(3)]
    mine = rc.concat_and_subset(my_ds.ConcatMultifieldDataset(parts), my_ds.SubsetMultifieldDataset)
    assert mine["len"] == ref["len"] == 13
    for key in ("raw", "items", "subset"):
        assert len(mine[key]) == len(ref[key])
        for a, b in zip(mine[key], ref[key]):
            assert list(a) == list(b) and all(torch.equal(a[k], b[k]) and a[k].dtype == b[k].dtype for k in a), key
    assert mine["accessor_log"] == ref["accessor_log"] == [(0, "a"), (0, "b"), (5, "a"), (5, "b"), (6, "a"), (6, "b")]
    assert mine["subset_len"] == ref["subset_len"] == 5
