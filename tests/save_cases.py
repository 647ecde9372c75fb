"""Shared pieces of the tests of blu_batch_save / blu_batch_restore (and their _dev variants): forking a lane
(copy_cases.CLane, whose oracle replays the source's history) through an image instead of blu_batch_copy, twin batches that fork one way each, and a mirror of the image layout of
blu_b200/csrc/blu_save.cuh (header fields, section offsets, checksum) so that tests can reach into an image."""
import numpy as np
import torch

from copy_cases import assert_copies, snapshot
from dev_cases import Twin

# header fields: (byte offset, numpy dtype)
HDR = dict(magic=(0, np.uint64), version=(8, np.int32), m=(12, np.int32), info_bytes=(16, np.int32), length=(24, np.int64),
           l_mem=(32, np.int64), u_mem=(40, np.int64), w_mem=(48, np.int64), l_n=(56, np.int64), u_n=(64, np.int64),
           w_n=(72, np.int64), bt_n=(80, np.int64), b_nz=(88, np.int64), checksum=(96, np.uint64))
INFO_AT = 112
# 4-byte words of the O(m) arrays of the state table (blu_slot_state.cuh), BluInfo left out (it is in the header)
STATE_WORDS = [lambda m: m + 1] + [lambda m: m] * 4 + [lambda m: 2 * m] * 2 + [lambda m: 2 * m] * 3 + \
              [lambda m: m + 1] * 8 + [lambda m: m] * 4 + [lambda m: 2 * m + 2] * 2 + [lambda m: m] * 3 + \
              [lambda m: 2 * m + 2] + [lambda m: m] * 2 + [lambda m: 4 * m + 4] + [lambda m: 2 * m] * 3


def field(img, name):
    off, dt = HDR[name]
    return img[off:off + np.dtype(dt).itemsize].view(dt)[0]


def set_field(img, name, value):
    off, dt = HDR[name]
    img[off:off + np.dtype(dt).itemsize].view(dt)[0] = value


def header_bytes(img):
    return (INFO_AT + int(field(img, "info_bytes")) + 15) & ~15


def sections(img):
    """[(name, byte offset, bytes without padding)] of the image's sections, in order"""
    m, g = int(field(img, "m")), {n: int(field(img, n)) for n in ("l_n", "u_n", "w_n", "bt_n", "b_nz")}
    sizes = [("header", header_bytes(img))]
    for st in ("l", "u", "w", "bt"):
        sizes += [(st + "_idx", 4 * g[st + "_n"]), (st + "_val", 8 * g[st + "_n"])]
    sizes += [(f"state{a}", 4 * w(m)) for a, w in enumerate(STATE_WORDS)]
    sizes += [("b_len", 8 * m), ("b_i", 8 * g["b_nz"]), ("b_x", 8 * g["b_nz"])]
    out, off = [], 0
    for name, n in sizes:
        out.append((name, off, n))
        off += (n + 15) & ~15
    assert off == int(field(img, "length")), (off, int(field(img, "length")))
    return out


def checksum(img):
    """the image checksum of blu_save.cuh: sum mod 2^64 of splitmix64's finalizer of (word index << 32 | word)"""
    w = img[:int(field(img, "length"))].view(np.uint32).astype(np.uint64)
    ck = HDR["checksum"][0] // 4
    w[ck] = 0
    w[ck + 1] = 0
    with np.errstate(over="ignore"):
        x = (np.arange(len(w), dtype=np.uint64) << np.uint64(32)) | w
        x ^= x >> np.uint64(30); x *= np.uint64(0xbf58476d1ce4e5b9)
        x ^= x >> np.uint64(27); x *= np.uint64(0x94d049bb133111eb)
        x ^= x >> np.uint64(31)
        return np.uint64(x.sum(dtype=np.uint64))


def reseal(img):
    """a copy of img with one header field changed by the caller already, its checksum made valid again"""
    set_field(img, "checksum", checksum(img))
    return img


def restore_fork(b, dst, src, mode):
    """basis dst[r] becomes basis src[r] through images: every distinct source is saved once and its image restored into
    all its destinations (fan-out of one image).  mode: 'host' (save / restore), 'dev' (save_dev / restore_dev) or
    'cross' (save by the host, restore_dev of the bytes moved to the device)."""
    u = sorted(set(src))
    if mode == "dev":
        imgs = b.save_dev(u)
    else:
        imgs = b.save(u)
        if mode == "cross":
            imgs = [torch.as_tensor(a).to(b._torch_device()) for a in imgs]
    pick = [imgs[u.index(s)] for s in src]
    return b.restore_dev(dst, pick) if mode in ("dev", "cross") else b.restore(dst, pick)


def fork(b, lanes, dst, src, mode="dev"):
    """restore_fork on the batch and the lanes (copy_cases.fork's counterpart)"""
    st = b.copy(dst, src) if isinstance(b, SaveTwin) else restore_fork(b, dst, src, mode)
    assert st == 0, st
    for d, s in zip(dst, src):
        if d < len(lanes):
            lanes[d].adopt(lanes[s])


def fork_and_check(b, lanes, dst, src, seed, mode="dev"):
    fork(b, lanes, dst, src, mode)
    ks = sorted(set(dst) | set(src))
    assert_copies(snapshot(b, ks, seed=seed, lanes=lanes), dst, src)


class SaveTwin(Twin):
    """twin batches: `h` forks through blu_batch_copy, `d` through images (restore_fork with `mode`); every other call
    runs as Twin runs it, and the two are compared after each"""

    def __init__(self, make, dev, mode):
        super().__init__(make, dev)
        self.mode = mode

    def copy(self, dst, src):
        st = self.h.copy(dst, src)
        assert restore_fork(self.d, dst, src, self.mode) == st
        self.assert_state()
        return st
