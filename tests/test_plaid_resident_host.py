"""CPU: the compressed PLAID residency — the decode-or-keep-compressed rule, the argument validation of
flmr_corpus_create_plaid that happens before any CUDA call, and the SASS of the decoding scan kernel."""
import ctypes as C
import hashlib
import os
import re
import subprocess

import numpy as np
import pytest

from ravqa_b200 import _cabi, build
from ravqa_b200 import plaid

GiB = 1 << 30


def test_decoded_shard_bytes():
    assert plaid.decoded_shard_bytes([4, 8, 12]) == 24 * 256                 # aligned: adopted, one matrix
    assert plaid.decoded_shard_bytes([3, 5]) == (8 + 12) * 256               # ragged: decoded + padded copy
    assert plaid.decoded_shard_bytes(np.full(1_000_000, 180)) == 180_000_000 * 256


def test_keep_compressed_rule():
    free = 170 * GiB
    margin = max(plaid.DECODE_MARGIN_BYTES, int(plaid.DECODE_MARGIN_FRACTION * free))
    assert not plaid.keep_compressed(free - margin, free)                    # exactly fits after the margin
    assert plaid.keep_compressed(free - margin + 1, free)
    assert not plaid.keep_compressed(1 << 20, free)                          # small shards are decoded
    # 5M passages of 180 tokens decoded (230 GB) never fit one 180 GB device: compressed
    assert plaid.keep_compressed(plaid.decoded_shard_bytes(np.full(5_000_000, 180)), free)
    # on a small free pool the fixed margin dominates
    assert plaid.keep_compressed(GiB, 4 * GiB) and not plaid.keep_compressed(GiB, 6 * GiB)


def test_residency_override_validates_and_resets():
    with pytest.raises(ValueError):
        plaid.debug_set_residency("sometimes")
    plaid.debug_set_residency("compressed")
    try:
        assert plaid.use_compressed([4], device=None)       # forced: no device query
        plaid.debug_set_residency("decoded")
        assert not plaid.use_compressed([10 ** 9], device=None)
    finally:
        plaid.debug_set_residency("auto")


def _create(nbits=2, dim=128, doclens=(3, 5), n_centroids=16, ptr=0x1000, n_passages=None):
    L = _cabi.lib()
    dl = np.asarray(doclens, dtype=np.int32)
    out = C.c_void_p()
    rc = L.flmr_corpus_create_plaid(ptr, ptr, ptr, n_centroids, ptr, nbits, dl.ctypes.data_as(C.c_void_p),
                                    len(dl) if n_passages is None else n_passages, dim, 0, 0, C.byref(out))
    return rc, L.flmr_last_error().decode(), out


def test_create_plaid_validates_arguments_before_any_cuda_call():
    rc, msg, out = _create(nbits=3)
    assert rc == 1 and "nbits=3" in msg and not out.value
    rc, msg, _ = _create(dim=64)
    assert rc == 3 and "dim=64" in msg
    rc, msg, _ = _create(ptr=None)
    assert rc == 1 and "null" in msg
    rc, msg, _ = _create(n_centroids=0)
    assert rc == 1 and "n_centroids" in msg
    rc, msg, _ = _create(n_passages=0)
    assert rc == 1
    rc, msg, _ = _create(doclens=(4, 0, 2))
    assert rc == 1 and "length 0" in msg
    rc, msg, _ = _create(doclens=(2 ** 30,) * 2)
    assert rc == 3 and "2^31" in msg
    assert _cabi.lib().flmr_corpus_create_plaid(None, None, None, 1, None, 2, None, 1, 128, 0, 0, None) == 1


def test_decoding_scan_kernel_sass():
    """One instantiation per nbits; each issues tcgen05.mma (UTCHMMA), drains TMEM (LDTM) and streams the
    compressed tiles with bulk copies (UBLKCP) — no tensor-map loads, no older mma.sync path."""
    build.build()
    sass = subprocess.run(["cuobjdump", "-sass", build.LIB_PATH], capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    kernels = {f.split("\n", 1)[0].strip(): f for f in funcs if "flmr_scan_plaid_kernel" in f.split("\n", 1)[0]}
    assert len(kernels) == 4, sorted(kernels)
    for name, body in kernels.items():
        for mnemonic in ("UTCHMMA", "LDTM", "UBLKCP", "STS.128"):
            assert mnemonic in body, (name, mnemonic)
        assert "UTMALDG" not in body and "HMMA" not in body.replace("UTCHMMA", ""), name


def test_plaid_builder_validates_arguments_before_any_cuda_call():
    L = _cabi.lib()
    dl = np.asarray([3, 5], dtype=np.int32)
    out = C.c_void_p()
    ptr = 0x1000
    assert L.flmr_corpus_plaid_builder_create(ptr, 16, ptr, 3, dl.ctypes.data_as(C.c_void_p), 2, 128, 0, 0,
                                              C.byref(out)) == 1
    assert "nbits=3" in L.flmr_last_error().decode() and not out.value
    assert L.flmr_corpus_plaid_builder_create(ptr, 16, ptr, 2, dl.ctypes.data_as(C.c_void_p), 2, 64, 0, 0,
                                              C.byref(out)) == 3
    big = np.full(2, 2 ** 30, dtype=np.int32)
    assert L.flmr_corpus_plaid_builder_create(ptr, 16, ptr, 2, big.ctypes.data_as(C.c_void_p), 2, 128, 0, 0,
                                              C.byref(out)) == 3
    assert "2^31" in L.flmr_last_error().decode()
    assert L.flmr_corpus_plaid_builder_append(None, None, None, 1) == 1
    assert L.flmr_corpus_plaid_builder_finish(None, None) == 1
    assert L.flmr_corpus_plaid_builder_destroy(None) == 0
    assert plaid.MAX_SHARD_ROWS == 2 ** 31 - 1 - _cabi.TILE_TOKENS


# flmr_scan_plaid_kernel.cuh carries a copy of flmr_scan_kernel's MMA issuers, epilogue and reducer (the bf16 kernel
# must stay byte-identical, so the two cannot share that code).  When the bf16 kernel changes, port the change to the
# copy, then update this hash.
SCAN_KERNEL_SHA256 = "bbcd6c9d67b5eec4bd67bba1a1dab12e224e90a029ab8def8d6b9d001cfd9c82"


def test_bf16_scan_kernel_unchanged_since_the_compressed_copy():
    path = os.path.join(os.path.dirname(build.__file__), "csrc", "flmr_scan_kernel.cuh")
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()
    assert digest == SCAN_KERNEL_SHA256, (
        "flmr_scan_kernel.cuh changed: port the change to the issuers / epilogue / reducer copy in "
        "flmr_scan_plaid_kernel.cuh, then update SCAN_KERNEL_SHA256")
