"""The run-time NVRTC cache directory (runtime/jit.py): it lives under the shared temporary directory, so it is used only
when it is a private directory of the current user; a cubin planted by someone else must never be loaded."""

import os

import pytest

from pytensor_b200.runtime import jit


@pytest.fixture
def cache_dir(tmp_path, monkeypatch):
    monkeypatch.delenv("PTK_KCACHE", raising=False)
    d = tmp_path / "kcache"
    monkeypatch.setattr(jit, "CACHE_DIR", str(d))
    jit._cache_dir_ok.cache_clear()
    yield d
    jit._cache_dir_ok.cache_clear()


def test_default_cache_dir_is_created_private(cache_dir):
    assert jit._cache_dir_ok()
    assert cache_dir.is_dir() and (cache_dir.stat().st_mode & 0o777) == 0o700


@pytest.mark.parametrize("mode", [0o777, 0o770])
def test_cache_dir_writable_by_others_is_refused(cache_dir, mode):
    cache_dir.mkdir()
    os.chmod(cache_dir, mode)
    assert not jit._cache_dir_ok()


def test_cache_dir_that_is_a_link_is_refused(cache_dir, tmp_path):
    target = tmp_path / "elsewhere"
    target.mkdir(mode=0o700)
    cache_dir.symlink_to(target)
    assert not jit._cache_dir_ok()
