"""Shared generators and comparison helpers for the parity tests (SURVEY.md section 8d inputs)."""
import numpy as np


def random_boxes(n, seed, width=1000, height=600, smin=16, smax=512, integer=False):
    """centres uniform, sizes log-uniform [smin, smax], clipped to the image."""
    rng = np.random.default_rng(seed)
    cx = rng.uniform(0, width, n)
    cy = rng.uniform(0, height, n)
    w = np.exp(rng.uniform(np.log(smin), np.log(smax), n))
    h = np.exp(rng.uniform(np.log(smin), np.log(smax), n))
    b = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], axis=1)
    b[:, 0::2] = np.clip(b[:, 0::2], 0, width - 1)
    b[:, 1::2] = np.clip(b[:, 1::2], 0, height - 1)
    if integer:
        b = np.round(b)
    return b.astype(np.float32)


def tie_free_scores(n, seed, lo=0.001, hi=0.999):
    rng = np.random.default_rng(seed)
    return rng.permutation(np.linspace(lo, hi, n)).astype(np.float32)


def iou_matrix64(b):
    """float64 IoU (+1 convention) of every pair, for margin checks."""
    b = b.astype(np.float64)
    area = (b[:, 2] - b[:, 0] + 1) * (b[:, 3] - b[:, 1] + 1)
    iw = np.minimum(b[:, None, 2], b[None, :, 2]) - np.maximum(b[:, None, 0], b[None, :, 0]) + 1
    ih = np.minimum(b[:, None, 3], b[None, :, 3]) - np.maximum(b[:, None, 1], b[None, :, 1]) + 1
    inter = np.clip(iw, 0, None) * np.clip(ih, 0, None)
    return inter / (area[:, None] + area[None, :] - inter)


def nudge_off_threshold(boxes, thresh, margin=1e-5, max_rounds=20, seed=0):
    """Perturb boxes until no pair's IoU lies within `margin` of `thresh`, so that fp32 rounding /
    FMA-contraction differences between implementations cannot flip a comparison."""
    rng = np.random.default_rng(seed)
    b = boxes.copy()
    for _ in range(max_rounds):
        iou = iou_matrix64(b)
        np.fill_diagonal(iou, 0)
        bad = np.where(np.abs(iou - thresh) < margin)
        if bad[0].size == 0:
            return b
        idx = np.unique(bad[0])
        b[idx, 2] += rng.uniform(0.25, 0.75, idx.size).astype(np.float32)
    raise AssertionError("could not separate IoUs from threshold")


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    denom = max(np.abs(b).max(), 1e-30)
    return np.abs(a - b).max() / denom


def digest(a):
    """sha256 of an array's shape and values: for NaN-free arrays, equal digests <=> np.array_equal
    (floats are hashed as float64 with -0.0 folded into +0.0, integers as int64)."""
    import hashlib
    a = np.asarray(a)
    if a.dtype.kind == "f":
        a = a.astype(np.float64) + 0.0
    else:
        a = a.astype(np.int64)
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(str(a.shape).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_idx(size, n=1024, seed=0):
    """A fixed sample of n flat indices into an array of `size` elements (all of them if fewer)."""
    if size <= n:
        return np.arange(size)
    return np.sort(np.random.default_rng(seed).choice(size, n, replace=False))


# ---------------------------------------------------------------------------------------------
# Test-only HDF5 assembler (superblock v0, old-style groups, contiguous float32 datasets): builds
# files with NESTED groups and multi-node group B-trees byte by byte from the file-format
# specification, to exercise mnc_b200/hdf5_min.py beyond the flat files the reference ships.
def write_h5_tree(path, tree):
    """tree: {name: ndarray | subtree}.  Datasets are written as contiguous little-endian float32."""
    import struct
    UNDEF = 0xFFFFFFFFFFFFFFFF
    buf = bytearray(b"\x00" * 96)          # superblock v0 (56 bytes) + root symbol-table entry (40)

    def alloc(n):
        while len(buf) % 8:
            buf.append(0)
        off = len(buf)
        buf.extend(b"\x00" * n)
        return off

    def put(off, data):
        buf[off:off + len(data)] = data

    def msg(mtype, body):
        body = bytes(body) + b"\x00" * (-len(body) % 8)
        return struct.pack("<HHB3x", mtype, len(body), 0) + body

    def header(msgs):
        body = b"".join(msgs)
        off = alloc(16 + len(body))
        put(off, struct.pack("<BBHII4x", 1, 0, len(msgs), 1, len(body)) + body)
        return off

    def dataset(arr):
        arr = np.ascontiguousarray(arr, dtype="<f4")
        data_off = alloc(arr.nbytes)
        put(data_off, arr.tobytes())
        space = struct.pack("<BBB5x", 1, arr.ndim, 0) + b"".join(struct.pack("<Q", d) for d in arr.shape)
        dtype = struct.pack("<BBBBI", 0x11, 0x20, 0x1F, 0x00, 4) + struct.pack("<HHBBBBI", 0, 32, 23, 8, 0, 23, 127)
        layout = struct.pack("<BBQQ", 3, 1, data_off, arr.nbytes)
        return header([msg(0x01, space), msg(0x03, dtype), msg(0x08, layout)])

    def group(sub):
        children = []
        for name in sorted(sub):           # group B-trees keep names in order
            v = sub[name]
            children.append((name, group(v)[0] if isinstance(v, dict) else dataset(v)))
        heap_data = bytearray(b"\x00" * 8)
        name_off = {}
        for name, _ in children:
            name_off[name] = len(heap_data)
            raw = name.encode() + b"\x00"
            heap_data.extend(raw + b"\x00" * (-len(raw) % 8))
        hd = alloc(len(heap_data))
        put(hd, heap_data)
        heap = alloc(32)
        put(heap, b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap_data), UNDEF, hd))
        snods = []
        for s in range(0, max(len(children), 1), 8):       # 2 * leaf K = 8 symbols per node
            part = children[s:s + 8]
            node = alloc(8 + 8 * 40)
            ent = b"".join(struct.pack("<QQII16x", name_off[n], a, 0, 0) for n, a in part)
            put(node, b"SNOD" + struct.pack("<BBH", 1, 0, len(part)) + ent)
            snods.append((node, name_off[part[-1][0]] if part else 0))
        tree_off = alloc(24 + (2 * 32 + 1) * 8 + 2 * 32 * 8)
        body = b"TREE" + struct.pack("<BBHQQ", 0, 0, len(snods), UNDEF, UNDEF) + struct.pack("<Q", 0)
        for node, last_name in snods:
            body += struct.pack("<QQ", node, last_name)
        put(tree_off, body)
        return header([msg(0x11, struct.pack("<QQ", tree_off, heap))]), tree_off, heap

    root, btree, heap = group(tree)
    put(0, b"\x89HDF\r\n\x1a\n" + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0) +
        struct.pack("<QQQQ", 0, UNDEF, len(buf), UNDEF) +
        struct.pack("<QQII", 0, root, 1, 0) + struct.pack("<QQ", btree, heap))
    with open(path, "wb") as f:
        f.write(bytes(buf))
