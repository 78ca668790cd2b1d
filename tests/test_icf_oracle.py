"""not-gpu: the integer-coded float mapping of the CPU oracle (oracle/g4o_icf.cpp) against a numpy restatement of the same
formulas, bit for bit, and ElementSpec.int_coded_float against the range blocks of the reference's four ICF sample files.

The formulas (GvrsElementSpecificationIntCodedFloat / GvrsElementIntCodedFloat as the ICF feature request restates them;
no reference fixture pins them beyond exactly representable values):
  float -> code: NaN -> fill_int; else (int) Math.floor((double)((v - offset) * scale) + 0.5)
  code -> float: fill_int -> fill_value; else (float) code / scale + offset"""
import struct

import numpy as np
import pytest

from gvrs_common import sample_files

INT_MIN, INT_MAX = -(2 ** 31), 2 ** 31 - 1
SCALES = [1.0, 10.0, 1000.0, 3.0, np.float32(0.1), -2.0]
OFFSETS = [0.0, -11000.5]


@pytest.fixture(scope="module")
def icf_ref():
    from oracle import g4icf

    return g4icf


def np_to_int(v, scale, offset, fill_int=INT_MIN):
    v = np.asarray(v, np.float32)
    with np.errstate(all="ignore"):
        t = (v - np.float32(offset)) * np.float32(scale)       # float32, correctly rounded, not fused
        d = np.floor(t.astype(np.float64) + 0.5)               # double
        k = np.where(np.isnan(d), 0.0, np.clip(d, INT_MIN, INT_MAX)).astype(np.int32)  # Java's (int): saturating, NaN -> 0
    return np.where(np.isnan(v), np.int32(fill_int), k).astype(np.int32)


def np_to_float(k, scale, offset, fill_int=INT_MIN, fill_value=np.float32("nan")):
    k = np.asarray(k, np.int32)
    x = (k.astype(np.float32) / np.float32(scale)) + np.float32(offset)
    return np.where(k == fill_int, np.float32(fill_value), x).astype(np.float32)


def bits(u32):
    return np.array(u32, np.uint64).astype(np.uint32).view(np.float32)


def adversarial_values():
    nans = bits([0x7FC00000, 0xFFC00000, 0x7F800001, 0x7FBFFFFF, 0xFF800001, 0x7FC12345, 0xFFFFFFFF])
    special = bits([0x7F800000, 0xFF800000, 0x00000000, 0x80000000, 0x00000001, 0x80000001, 0x007FFFFF, 0x807FFFFF,
                    0x7F7FFFFF, 0xFF7FFFFF])
    ties = np.array([0.5, -0.5, 1.5, -1.5, 2.5, -2.5, 3.5, -3.5, 0.05, -0.05, 0.15, 1.25, -1.25, 8388607.5, -8388607.5,
                     np.float32(0.49999997), -np.float32(0.49999997), np.nextafter(np.float32(0.5), np.float32(1)),
                     -11000.5, -11000.0, -11001.0, -10999.5], np.float32)
    saturate = np.array([2.0 ** 31, -(2.0 ** 31), 2.0 ** 31 - 128, -(2.0 ** 31) + 128, 3e9, -3e9, 1e20, -1e20, 2147483.5,
                         -2147483.5, 214748364.0, -214748364.0, 1.0737418e9, -1.0737418e9], np.float32)
    big = np.array([16777216.0, 16777218.0, -16777218.0, 1e8, -1e8, 123456789.0], np.float32)
    return np.concatenate([nans, special, ties, saturate, big])


def adversarial_codes():
    return np.array([INT_MIN, INT_MIN + 1, INT_MAX, INT_MAX - 1, 0, 1, -1, 5, -5, 25, -25, 2 ** 24, 2 ** 24 + 1, 2 ** 24 + 3,
                     -(2 ** 24) - 1, 2 ** 25 + 1, 123456789, -123456789, 2 ** 30 + 63, -110005, -110000, 999, 1000, 1001],
                    np.int64).astype(np.int32)


def test_known_values(icf_ref):
    assert list(icf_ref.icf_to_int(np.array([-2.5, 2.5, -0.5, 0.5, np.float32(0.49999997)], np.float32), 1.0)) == [-2, 3, 0, 1, 0]
    assert list(icf_ref.icf_to_int(np.array([np.inf, -np.inf, np.nan, 3e9, -3e9], np.float32), 1.0)) == [INT_MAX, INT_MIN, INT_MIN,
                                                                                                      INT_MAX, INT_MIN]
    # above 2^24 int -> float rounds to nearest even
    assert icf_ref.icf_to_float(np.array([2 ** 24 + 1, 2 ** 24 + 3], np.int32), 1.0).tolist() == [16777216.0, 16777220.0]
    # decimetre values at scale 10: k / 10f, which can differ by one ulp from k * 0.1f
    k = np.arange(-109000, 88001, dtype=np.int32)
    v = k.astype(np.float32) * np.float32(0.1)
    assert np.array_equal(icf_ref.icf_to_int(v, 10.0), k)
    back = icf_ref.icf_to_float(k, 10.0)
    assert np.array_equal(back, k.astype(np.float32) / np.float32(10))
    ulps = np.abs(back.view(np.int32).astype(np.int64) - v.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1


@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("offset", OFFSETS)
def test_oracle_equals_numpy_on_adversarial_and_random_bits(icf_ref, scale, offset):
    v = adversarial_values()
    want = np_to_int(v, scale, offset)
    got = icf_ref.icf_to_int(v, scale, offset)
    assert np.array_equal(got, want), (v[got != want], got[got != want], want[got != want])
    k = np.concatenate([adversarial_codes(), got])
    assert np.array_equal(icf_ref.icf_to_float(k, scale, offset).view(np.uint32), np_to_float(k, scale, offset).view(np.uint32))
    rng = np.random.default_rng(abs(hash((float(scale), offset))) % 2 ** 32)
    r = rng.integers(0, 2 ** 32, 10 ** 6, dtype=np.uint64).astype(np.uint32)
    v = r.view(np.float32)
    assert np.array_equal(icf_ref.icf_to_int(v, scale, offset), np_to_int(v, scale, offset))
    k = r.view(np.int32)
    assert np.array_equal(icf_ref.icf_to_float(k, scale, offset).view(np.uint32), np_to_float(k, scale, offset).view(np.uint32))


def test_non_nan_fill(icf_ref):
    """fill -9999 at scale 10: fill_int is the fill's code; finite values with that code read back as the fill value."""
    fill_int = int(np_to_int([-9999.0], 10.0, 0.0)[0])
    assert fill_int == -99990
    v = np.array([-9999.0, -9999.04, -9998.96, np.nan, 1.0, -np.inf, np.inf], np.float32)
    k = icf_ref.icf_to_int(v, 10.0, 0.0, fill_int)
    assert np.array_equal(k, np_to_int(v, 10.0, 0.0, fill_int))
    assert k.tolist()[:4] == [fill_int] * 4
    back = icf_ref.icf_to_float(k, 10.0, 0.0, fill_int, -9999.0)
    assert np.array_equal(back.view(np.uint32), np_to_float(k, 10.0, 0.0, fill_int, -9999.0).view(np.uint32))
    assert back.tolist()[:4] == [-9999.0] * 4 and back[4] == 1.0


def test_element_spec_rebuilds_the_ICF_sample_range_blocks():
    from gridfour_b200 import gvrs

    files = sample_files()
    for name in ["Sample03_ICFNoComp.gvrs", "Sample07_ICFComp.gvrs", "Sample12_ICFNoComp.gvrs"]:
        e = gvrs.GvrsImage.parse(files[name]).spec.elements[0]
        assert e.type_code == gvrs.ELEM_INT_CODED_FLOAT
        assert gvrs.ElementSpec.int_coded_float(e.name, 1.0, 0.0, -20000.0, 20000.0).range_block == e.range_block, name
    e = gvrs.GvrsImage.parse(files["Sample14_LSOP.gvrs"]).spec.elements[0]
    again = gvrs.ElementSpec.int_coded_float(e.name, 1000.0)
    assert again.range_block == e.range_block
    assert struct.unpack_from("<ff", again.range_block, 0) == (-2147483.75, 2147483.75)
    icf = e.icf
    assert (icf.scale, icf.offset, icf.fill_int) == (1000.0, 0.0, INT_MIN) and np.isnan(icf.fill_value)
    assert gvrs.ElementSpec.integer("z").icf is None
    # a non-NaN fill is stored as its code
    e = gvrs.ElementSpec.int_coded_float("z", 10.0, 0.0, fill_value=-9999.0)
    assert struct.unpack_from("<iii", e.range_block, 20) == (INT_MIN + 1, INT_MAX, -99990) and e.fill_value == -99990
    with pytest.raises(ValueError):
        gvrs.ElementSpec.int_coded_float("z", 0.0)
