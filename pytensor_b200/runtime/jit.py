"""NVRTC-backed kernel cache.

The reference compiles one C++ module per Apply node with g++ and caches it on disk keyed by op/type signature
(pytensor/link/c/cmodule.py:612 ModuleCache, :1181-1260 module_from_key).  The B200 analogue: one sm_100a cubin per
generated kernel source, cached in memory per process and on disk keyed by the SHA-256 of (source, options).  On disk,
the cubins `__graft_entry__.build()` compiled into the package's `_kcache/` are read; kernels compiled at run time are
written to a per-user directory under the system's temporary directory, so that running never writes into the source
tree (which may be read-only).  `PTK_KCACHE` replaces both with one directory that is read and written (`build()` points
it at `_kcache/`).
"""

from __future__ import annotations

import ctypes
import functools
import hashlib
import os
import stat
import tempfile
import threading

from . import lib as _lib

if "PTK_KCACHE" in os.environ:
    CACHE_DIR = os.environ["PTK_KCACHE"]
    READ_DIRS: tuple[str, ...] = (CACHE_DIR,)
else:
    CACHE_DIR = os.path.join(tempfile.gettempdir(), f"ptk_kcache_{os.getuid()}")
    READ_DIRS = (os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "_kcache"), CACHE_DIR)

_lock = threading.Lock()
_cubins: dict[str, bytes] = {}
_modules: dict[str, int] = {}
_functions: dict[tuple[str, str], int] = {}
stats = {"compiled": 0, "disk_hits": 0, "mem_hits": 0, "launches": 0}


def _key(src: str, opts: tuple[str, ...]) -> str:
    h = hashlib.sha256()
    h.update(("ptk-jit-v1\0" + "\0".join(opts) + "\0").encode())
    h.update(src.encode())
    return h.hexdigest()[:32]


@functools.cache
def _cache_dir_ok() -> bool:
    """Whether CACHE_DIR may be read and written.  The default one sits in a directory where every user can create paths
    and cache keys are predictable, so a cubin another user planted there would be loaded in place of ours: it is used
    only as a real directory (not a link) that this user owns and that no one else can write to."""
    if "PTK_KCACHE" in os.environ:
        return True
    try:
        os.makedirs(CACHE_DIR, mode=0o700, exist_ok=True)
        st = os.lstat(CACHE_DIR)
    except OSError:
        return False
    return stat.S_ISDIR(st.st_mode) and st.st_uid == os.getuid() and not st.st_mode & 0o022


def compile_cubin(src: str, opts: tuple[str, ...] = ()) -> tuple[str, bytes]:
    """Source -> (key, cubin bytes). Needs no GPU (NVRTC cross-compiles), so it also runs in the CPU-only build check."""
    key = _key(src, opts)
    with _lock:
        if key in _cubins:
            stats["mem_hits"] += 1
            return key, _cubins[key]
    for d in READ_DIRS:
        cached = os.path.join(d, key + ".cubin")
        if (d != CACHE_DIR or _cache_dir_ok()) and os.path.exists(cached):
            with open(cached, "rb") as f:
                data = f.read()
            with _lock:
                _cubins[key] = data
                stats["disk_hits"] += 1
            return key, data
    path = os.path.join(CACHE_DIR, key + ".cubin")
    L = _lib.load_library()
    cubin = ctypes.c_void_p()
    size = ctypes.c_size_t()
    log = ctypes.c_void_p()
    c_opts = (ctypes.c_char_p * max(1, len(opts)))(*[o.encode() for o in opts])
    st = L.ptk_jit_compile(src.encode(), c_opts, len(opts), ctypes.byref(cubin), ctypes.byref(size), ctypes.byref(log))
    log_txt = ""
    if log.value:
        log_txt = ctypes.string_at(log.value).decode("utf-8", "replace")
        L.ptk_free(log)
    if st != 0:
        numbered = "\n".join(f"{i + 1:4d}: {line}" for i, line in enumerate(src.split("\n")))
        raise _lib.PtkError(f"NVRTC failed: {_lib.last_error()}\n{log_txt}\n--- source ---\n{numbered}")
    data = ctypes.string_at(cubin.value, size.value)
    L.ptk_free(cubin)
    try:
        if not _cache_dir_ok():
            raise OSError(f"not a private directory: {CACHE_DIR}")
        os.makedirs(CACHE_DIR, exist_ok=True)
        tmp = path + f".tmp{os.getpid()}"
        with open(tmp, "wb") as f:
            f.write(data)
        os.replace(tmp, path)
        with open(os.path.join(CACHE_DIR, key + ".cu"), "w") as f:
            f.write(src)
    except OSError:
        pass
    with _lock:
        _cubins[key] = data
        stats["compiled"] += 1
    return key, data


def get_function(src: str, name: str, opts: tuple[str, ...] = ()) -> int:
    """Source + kernel name -> CUfunction handle (loads the module on the current device on first use)."""
    key, data = compile_cubin(src, opts)
    fkey = (key, name)
    f = _functions.get(fkey)
    if f is not None:
        return f
    L = _lib.lib()
    with _lock:
        mod = _modules.get(key)
        if mod is None:
            m = ctypes.c_void_p()
            buf = ctypes.create_string_buffer(data, len(data))
            _lib.check(L.ptk_module_load(buf, len(data), ctypes.byref(m)), "ptk_module_load")
            mod = m.value
            _modules[key] = mod
        fn = ctypes.c_void_p()
        _lib.check(L.ptk_module_get_function(mod, name.encode(), ctypes.byref(fn)), f"get_function({name})")
        _functions[fkey] = fn.value
    return fn.value


def get_function_gen(gen, prefix: str, opts: tuple[str, ...] = ()):
    """`gen(kernel_name) -> source`.  The kernel is named after the hash of its own source so that the same generated
    kernel has the same name (and disk-cache key) in every process — cubins built by `build()` are hits on the GPU box.
    Returns (function handle, kernel name)."""
    placeholder = "PTKKERNELNAMEPLACEHOLDER"
    src = gen(placeholder)
    name = f"{prefix}_{hashlib.sha256(src.encode()).hexdigest()[:16]}"
    src = src.replace(placeholder, name)
    if _lib.TRACE_ONLY:
        compile_cubin(src, opts)
        return 0, name
    return get_function(src, name, opts), name


def precompile_gen(gen, prefix: str, opts: tuple[str, ...] = ()) -> str:
    """CPU-side half of get_function_gen (NVRTC only, no device): used by build() to warm the disk cache."""
    placeholder = "PTKKERNELNAMEPLACEHOLDER"
    src = gen(placeholder)
    name = f"{prefix}_{hashlib.sha256(src.encode()).hexdigest()[:16]}"
    compile_cubin(src.replace(placeholder, name), opts)
    return name


class KernelArgs:
    """Packs kernel parameters for ptk_launch: keeps the ctypes scalars alive and exposes the void*[] array."""

    __slots__ = ("_vals", "array")

    def __init__(self, vals):
        self._vals = vals
        n = len(vals)
        self.array = (ctypes.c_void_p * n)(*[ctypes.cast(ctypes.pointer(v), ctypes.c_void_p) for v in vals])


def launch(func: int, grid, block, args: KernelArgs, smem: int = 0, stream: int = 0, cooperative: bool = False,
           cluster: int = 1) -> None:
    gx, gy, gz = (tuple(grid) + (1, 1))[:3]
    bx, by, bz = (tuple(block) + (1, 1))[:3]
    stats["launches"] += 1
    if _lib.TRACE_ONLY:
        return
    _lib.check(
        _lib.lib().ptk_launch(func, gx, gy, gz, bx, by, bz, smem, stream, args.array, 1 if cooperative else 0, cluster),
        "ptk_launch",
    )
