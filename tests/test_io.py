"""CPU suite: the `.csr` binary format (SURVEY.md §8f row 3) — essentials_b200/io.py against the reference's own
csr_t::read_binary / write_binary (formats/csr.hxx:159-236), compiled in oracle/_ref/libref_cpu.so."""
import os

import numpy as np
import pytest
import torch

import oracle
from essentials_b200 import graphgen as gg
from essentials_b200 import io as eio

# the reference writer's bytes for _graphs() (tests/golden/make_reference_vectors.py), used without oracle/_ref
STORED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")


def _graphs():
    yield gg.rmat_csr(8, weights="hash")
    yield gg.grid_csr(7, 5)
    yield gg.rmat_csr(6, symmetric=False, weights="none")  # pattern matrix: values written as 1.0


def test_our_files_are_read_by_the_reference(tmp_path):
    """With the reference's reader, or else: our files are byte for byte the files the reference writes."""
    for i, csr in enumerate(_graphs()):
        path = str(tmp_path / f"ours_{i}.csr")
        eio.write_csr_binary(path, csr)
        if not oracle.have_ref():
            assert open(path, "rb").read() == np.load(STORED)[f"csr_file_{i}"].tobytes(), i
            continue
        off, col, val = oracle.ref_read_csr_binary(path)
        want_off, want_col, want_val = csr.host()
        assert np.array_equal(off, want_off) and np.array_equal(col, want_col)
        assert np.array_equal(val, want_val if csr.values is not None else np.ones(csr.m, np.float32))


def test_reference_files_are_read_by_us_byte_identical_writer(tmp_path):
    for i, csr in enumerate(_graphs()):
        off, col, val = csr.host()
        val = val if csr.values is not None else np.ones(csr.m, np.float32)
        ref_path, our_path = str(tmp_path / f"ref_{i}.csr"), str(tmp_path / f"ours_{i}.csr")
        if oracle.have_ref():
            oracle.ref_write_csr_binary(ref_path, off, col, val)
        else:  # the file the reference's writer produced for this graph
            np.load(STORED)[f"csr_file_{i}"].tofile(ref_path)
        eio.write_csr_binary(our_path, csr)
        assert open(ref_path, "rb").read() == open(our_path, "rb").read(), "writer must be byte-identical"
        for bits in (32, "auto"):
            back = eio.read_csr_binary(ref_path, offset_bits=bits)
            assert back.n == csr.n and back.m == csr.m and back.offsets.dtype == torch.int32
            assert np.array_equal(back.offsets.numpy(), off) and np.array_equal(back.indices.numpy(), col)
            assert np.array_equal(back.values.numpy(), val)


def test_wide_offsets_round_trip_and_errors(tmp_path):
    csr = gg.rmat_csr(7, weights="hash", offset_bits=64)
    path = str(tmp_path / "wide.csr")
    eio.write_csr_binary(path, csr)
    back = eio.read_csr_binary(path)  # auto: recognised as 64-bit from the file size
    assert back.offsets.dtype == torch.int64 and torch.equal(back.offsets, csr.offsets)
    assert torch.equal(back.indices, csr.indices) and torch.equal(back.values, csr.values)
    with pytest.raises(ValueError):
        eio.read_csr_binary(path, offset_bits=32)
    data = open(path, "rb").read()
    cut = str(tmp_path / "cut.csr")
    open(cut, "wb").write(data[:-8])
    with pytest.raises(ValueError):
        eio.read_csr_binary(cut)
    empty = gg.CSR(3, 0, torch.zeros(4, dtype=torch.int32), torch.zeros(0, dtype=torch.int32), None, "empty", True)
    p = str(tmp_path / "empty.csr")
    eio.write_csr_binary(p, empty)
    e = eio.read_csr_binary(p, offset_bits=32)
    assert e.n == 3 and e.m == 0
