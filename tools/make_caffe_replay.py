"""Converts ONE iteration of the reference's Caffe CIFAR export
(``tests/functional/data/cifar_export.tar.xz`` of the reference tree: text dumps of every layer's
blobs before/after its forward and backward pass, batch 3) into compact ``.npz`` files that travel
with the repo, one per layer and direction (the tarball is 65 MB of text).
Arrays are NHWC float32; weights keep Caffe's [F][C][ky][kx] order.

    python tools/make_caffe_replay.py <reference tree> [iteration]
"""
import collections
import os
import sys
import tarfile

import numpy

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                   "caffe_cifar_iter%d")


def parse(text):
    blobs = {}
    lines = text.split("\n")
    i = 0
    while i < len(lines):
        parts = lines[i].rstrip().split("\t")
        if len(parts) >= 5 and parts[1].startswith("num:"):
            name = parts[0]
            d = dict(p.split(":") for p in parts[1:])
            n, c, h, w = int(d["num"]), int(d["channels"]), int(d["height"]), int(d["width"])
            arr = numpy.zeros((n, c, h, w), numpy.float32)
            i += 1
            for a in range(n):
                assert lines[i].strip() == "num:%d" % a, lines[i]
                i += 1
                for b in range(c):
                    assert lines[i].strip() == "channels:%d" % b, lines[i]
                    i += 1
                    for y in range(h):
                        arr[a, b, y] = numpy.array(lines[i].split(), dtype=numpy.float64)
                        i += 1
            blobs[name] = arr
        else:
            i += 1
    return blobs


def main(ref_tree, iteration=0):
    out = {}
    src = os.path.join(ref_tree, "tests", "functional", "data", "cifar_export.tar.xz")
    with tarfile.open(src, "r:xz") as tar:
        for m in tar.getmembers():
            parts = m.name.split("/")
            if len(parts) != 3 or parts[1] != str(iteration):
                continue
            kind, layer, direction, when, _ts = parts[2].split(".")
            if when != "after":
                continue
            blobs = parse(tar.extractfile(m).read().decode())
            for name, arr in blobs.items():
                if name.startswith("blob_"):
                    if direction != "forward":
                        continue
                    val = arr                                   # weights: Caffe order
                else:
                    val = numpy.ascontiguousarray(arr.transpose(0, 2, 3, 1))   # NCHW -> NHWC
                out["%s/%s/%s" % (layer, direction, name)] = val.astype(numpy.float32)
    parts = collections.defaultdict(dict)
    for key, val in out.items():
        layer, direction, _ = key.split("/")
        parts[layer + "." + direction][key] = val
    path = OUT % iteration
    os.makedirs(path, exist_ok=True)
    for name, arrays in sorted(parts.items()):
        numpy.savez_compressed(os.path.join(path, name + ".npz"), **arrays)
    print(path, len(parts), "files", len(out), "arrays")


if __name__ == "__main__":
    main(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 0)
