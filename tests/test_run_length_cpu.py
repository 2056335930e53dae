"""Batches of runs of different lengths, host side without a GPU: samsim_grotz_batch rejects what it cannot run
before it touches a device."""
import ctypes as C

import pytest

from samsim_b200 import api, build, grotz


@pytest.fixture(scope="module", autouse=True)
def _built():
    build.build()


def _call(members, **opt):
    L = grotz._lib()
    ms = (grotz._GrotzMember * len(members))(*[grotz._GrotzMember(tc, b"", b".", 0) for tc in members]) if members else None
    o = grotz._GrotzOptions(**opt)
    codes = (C.c_int32 * 8)()
    return L.samsim_grotz_batch(ms, len(members), C.byref(o), codes)


def test_grotz_batch_checks_before_the_device():
    assert _call([1, 101]) == -4                                        # members must share one configuration
    assert _call([101, 8]) == -4
    assert _call([1, 1], ncol=2) == -1                                  # ncol belongs to samsim_grotz
    assert _call([1], max_steps=10) == -1
    assert _call([]) == -1                                              # NULL member list


def test_grotz_batch_wrapper_raises(tmp_path):
    with pytest.raises(api.SamsimError) as e:
        grotz.grotz_batch([{"testcase": 1, "output_dir": tmp_path / "a"}, {"testcase": 101, "output_dir": tmp_path / "b"}])
    assert e.value.code == -4
    with pytest.raises(api.SamsimError) as e:
        grotz.grotz_batch([])
    assert e.value.code == -1
