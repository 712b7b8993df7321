"""The `run_editing_*` entry-point plumbing on the CPU: dataset schema, RLE mask decoding (against the reference's own
function, recorded in tests/golden/reference_cli.npz), output layout, skip-if-exists, and the image-parallel split of the
work list."""
import ast
import json
import os

import numpy as np
import pytest

from pnpinversion_b200 import cli
from pnpinversion_b200.parallel import shard_sizes
from oracle import ref_shim
from tests.reference_golden import recorded_fixture

golden = recorded_fixture("cli")


def _reference_mask_decode():
    path = os.path.join(ref_shim.REF, "run_editing_p2p.py")
    with open(path) as f:
        tree = ast.parse(f.read(), filename=path)
    tree.body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "mask_decode"]
    ns = {"np": np}
    exec(compile(tree, path, "exec"), ns)
    return ns["mask_decode"]


def test_mask_decode_matches_the_reference_function(golden):
    ref = _reference_mask_decode() if golden.recording else None
    rng = np.random.RandomState(0)
    for i in range(5):
        starts = np.sort(rng.choice(512 * 512 - 600, size=40, replace=False))
        rle = []
        for s in starts:
            rle += [int(s), int(rng.randint(1, 500))]
        rle += [512 * 512 - 10, 500]  # a run that overshoots the image: clipped (run_editing_p2p.py:16)
        assert golden.equal(f"mask_decode/{i}", cli.mask_decode(rle), lambda: ref(rle))
    assert golden.equal("mask_decode/empty", cli.mask_decode([]), lambda: ref([]))


def test_mask_round_trip_and_border():
    m = np.zeros((512, 512), np.uint8)
    m[100:200, 50:300] = 1
    dec = cli.mask_decode(cli.mask_encode(m))
    assert dec[150, 100] == 1 and dec[300, 300] == 0
    assert dec[0].all() and dec[-1].all() and dec[:, 0].all() and dec[:, -1].all()  # forced border
    inner = dec[1:-1, 1:-1]
    assert np.array_equal(inner, m[1:-1, 1:-1])


def _args(data, out, methods, **kw):
    import argparse

    p = argparse.ArgumentParser()
    cli.add_common_args(p, methods)
    a = p.parse_args(["--data_path", data, "--output_path", out])
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_sweep_layout_skip_and_sharding(tmp_path, monkeypatch):
    from PIL import Image

    data = str(tmp_path / "data")
    out = str(tmp_path / "out")
    cli.write_synthetic_dataset(data, n_items=13, size=64)
    items = cli.read_items(data, cli.CATEGORIES)
    assert len(items) == 13 and items[0]["prompt_src"] == "a cat sitting on a table with a green eyes"  # brackets stripped
    assert items[0]["blended_word"] == ["cat", "dog"] and cli.mask_decode(items[0]["mask"], (64, 64)).shape == (64, 64)
    assert len(cli.read_items(data, ["3"])) == 1  # editing_type_id filter (run_editing_p2p.py:101-102)
    calls = []

    def edit_one(method, item):
        calls.append((method, item["key"]))
        return Image.new("RGB", (2048, 512))

    # two ranks: contiguous uneven split 7 / 6, every item edited exactly once
    for rank in range(2):
        monkeypatch.setenv("RANK", str(rank))
        monkeypatch.setenv("WORLD_SIZE", "2")
        st = cli.sweep(_args(data, out, ["directinversion+p2p"]), ("directinversion+p2p",), edit_one)
        assert st["items"] == (7 if rank == 0 else 6) and st["edited"] == st["items"]
    assert sorted(k for _, k in calls) == sorted(it["key"] for it in items)
    first = items[0]
    dst = cli.out_path(first, data, out, "directinversion+p2p")
    assert dst == first["image_path"].replace(data, os.path.join(out, "directinversion+p2p")) and os.path.exists(dst)
    assert Image.open(dst).size == (2048, 512)
    # second run: everything is skipped unless --rerun_exist_images
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("WORLD_SIZE", "1")
    n = len(calls)
    st = cli.sweep(_args(data, out, ["directinversion+p2p"]), ("directinversion+p2p",), edit_one)
    assert st["skipped"] == 13 and st["edited"] == 0 and len(calls) == n
    st = cli.sweep(_args(data, out, ["directinversion+p2p"], rerun_exist_images=True), ("directinversion+p2p",), edit_one)
    assert st["edited"] == 13
    # batching: edit_many receives chunks of --batch items
    chunks = []

    def edit_many(method, its):
        chunks.append(len(its))
        return [Image.new("RGB", (2048, 512)) for _ in its]

    cli.sweep(_args(data, out, ["directinversion+p2p"], rerun_exist_images=True, batch=4), ("directinversion+p2p",),
              edit_one, edit_many)
    assert chunks == [4, 4, 4]  # the last chunk of one goes through edit_one
    with pytest.raises(NotImplementedError):
        cli.sweep(_args(data, out, ["no-such-method"]), ("directinversion+p2p",), edit_one)


def test_pie_bench_split_sizes():
    assert shard_sizes(700, 8) == [88, 88, 88, 88, 87, 87, 87, 87]
