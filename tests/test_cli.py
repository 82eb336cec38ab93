"""The reference's process-level seam: `VoxelRaymarcher <scale> <hashtable|vcs> <original|longestaxis>` (Main.cu:176-229)."""
import os
import struct
import subprocess

import numpy as np
import pytest

from tests.common import ROOT, scenes
from voxelraymarcher_b200 import api

CLI = os.path.join(ROOT, "voxelraymarcher_b200", "VoxelRaymarcher")


def test_cli_requires_a_scale():
    p = subprocess.run([CLI], stdout=subprocess.PIPE, text=True)
    assert p.returncode == 1                                  # Main.cu:181-185
    assert p.stdout.strip() == "You need to provide a voxel scale"


@pytest.mark.skipif(api.device_available(), reason="CPU-only tier check")
def test_cli_fails_loudly_without_a_gpu(tmp_path):
    p = subprocess.run([CLI, "8", "hashtable", "original"], stdout=subprocess.PIPE, text=True, cwd=tmp_path)
    assert p.returncode != 0
    assert "Storage Type: Cuckoo Hash Table" in p.stdout and "Raymarching Algorithm: Original" in p.stdout
    assert "Device Count: 0" in p.stdout and "ERROR" in p.stdout


def _run_cli(tmp_path, args):
    p = subprocess.run([CLI, *args], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=tmp_path)
    assert p.returncode == 0, p.stdout
    from PIL import Image
    return p.stdout, np.asarray(Image.open(os.path.join(tmp_path, "output.png")).convert("RGB"))


@pytest.mark.gpu
@pytest.mark.parametrize("argv,storage,algo", [(["8", "hashtable", "original"], "hashtable", "original"), (["8"], "vcs", "longestaxis"),
                                               (["8", "vcs", "bogus"], "vcs", "longestaxis")])
def test_cli_matches_api_on_csv_scene(tmp_path, argv, storage, algo):
    xyz, rgb = scenes.probe_scene()
    os.makedirs(tmp_path / "resources")
    scenes.write_csv(str(tmp_path / "resources" / "scene.vox"), xyz, rgb)
    out, img = _run_cli(tmp_path, argv)
    for line in ("Device Count:", "regions that are filled", "Storage Structures Generated", "Execution Time for Ray Marching Algorithm is:"):
        assert line in out
    assert "There are : 13/125 regions that are filled" in out
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene(storage)
    want = s.render(1920, 1080, algo, api.Camera.reference_default(), scale=8)["rgb"]
    assert img.shape == (1080, 1920, 3)
    assert np.array_equal(img, want)


@pytest.mark.gpu
def test_cli_reads_magicavoxel(tmp_path):
    rng = np.random.default_rng(3)
    pts = np.unique(rng.integers(0, 40, size=(3000, 3)), axis=0).astype(np.uint8)
    idx = rng.integers(1, 256, size=pts.shape[0]).astype(np.uint8)
    palette = rng.integers(0, 256, size=(256, 4)).astype(np.uint8)

    def chunk(cid, body, children=b""):
        return cid + struct.pack("<II", len(body), len(children)) + body + children
    xyzi = struct.pack("<I", pts.shape[0]) + np.concatenate([pts, idx[:, None]], 1).tobytes()
    kids = chunk(b"SIZE", struct.pack("<III", 40, 40, 40)) + chunk(b"XYZI", xyzi) + chunk(b"RGBA", palette.tobytes())
    os.makedirs(tmp_path / "resources")
    with open(tmp_path / "resources" / "scene.vox", "wb") as f:
        f.write(b"VOX " + struct.pack("<I", 150) + chunk(b"MAIN", b"", kids))
    _, img = _run_cli(tmp_path, ["1", "vcs", "original", "--width", "640", "--height", "360"])
    xyz = np.stack([pts[:, 0], pts[:, 2], pts[:, 1]], 1).astype(np.int32)      # z-up -> y-up
    pal = palette[idx.astype(np.int32) - 1].astype(np.uint32)                  # palette entry i is stored at i-1
    rgb = (pal[:, 0] << 16) | (pal[:, 1] << 8) | pal[:, 2]
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene("vcs")
    cam = api.Camera((6.0, 2.0, 6.0), (0.0, 0.0, -1.0), (0.0, 1.0, 0.0), 60.0, np.float32(640) / np.float32(360))
    want = s.render(640, 360, "original", cam, scale=1, want_hits=True)
    assert np.array_equal(img, want["rgb"])
    assert want["hits"][..., 3].sum() > 1000


# ---- scene loaders, checked without a GPU through `--dump-voxels` -------------------------------------------------------------------
def _dump(tmp_path, scene_bytes):
    os.makedirs(tmp_path / "resources", exist_ok=True)
    with open(tmp_path / "resources" / "scene.vox", "wb") as f:
        f.write(scene_bytes)
    out = tmp_path / "dump.csv"
    p = subprocess.run([CLI, "1", "vcs", "original", "--dump-voxels", str(out)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=tmp_path)
    if p.returncode != 0:
        return None, p.stdout
    rows = [tuple(int(v) for v in line.split(",")) for line in open(out).read().splitlines() if line]
    return rows, p.stdout


def test_csv_reader_matches_the_reference_reader(tmp_path):
    """geometry/VoxelFile.cuh:9-35 through the reference's OWN reader (oracle host build) on a file full of its quirks: empty fields do
    not count, lines with fewer than four fields are skipped, extra fields ignored, std::stoi number syntax (white space, signs,
    trailing text), CRLF line ends, duplicates (last wins), negative coordinates, no newline at the end."""
    from tests.common import po
    rng = np.random.default_rng(11)
    lines = ["1,2,3,255", "4,,5,,6,,1193046", ",,7,8,9,65280,", "10,11,12", "", ",,,", " 13, 14,\t15, 16711680", "-70,-3,-129,4660",
             "+5,6,7,99 trailing", "20,21,22,23,24,25", "1,2,3,128\r", "3,2,1,77\r", "1e2,5,5,5", "0x10,9,9,9", "64,64,64,16777215", "-1,-1,-1,1"]
    for _ in range(300):
        x, y, z = (int(v) for v in rng.integers(-150, 150, 3))
        sep = rng.choice([",", ",,", ", "])
        lines.append(sep.join(str(v) for v in (x, y, z, int(rng.integers(1, 1 << 24)))))
    text = "\n".join(lines)            # no trailing newline
    rows, out = _dump(tmp_path, text.encode())
    assert rows is not None, out
    assert (1, 2, 3, 255) in rows and (4, 5, 6, 1193046) in rows and (7, 8, 9, 65280) in rows and (13, 14, 15, 16711680) in rows
    assert (5, 6, 7, 99) in rows and (20, 21, 22, 23) in rows and (1, 5, 5, 5) in rows and (0, 9, 9, 9) in rows
    assert not any(r[:3] == (10, 11, 12) for r in rows)
    if not po.available("refh"):
        pytest.skip("the reference's own reader needs a build of the original project in oracle/_ref (oracle/Makefile, from a reference checkout that is not part of this repository)")
    ref = po.OracleScene("refh")
    ref.load_file(str(tmp_path))
    ref.build("hashtable")
    mine = po.OracleScene("refh")
    mine.add_voxels(np.array([r[:3] for r in rows], np.int32), np.array([r[3] for r in rows], np.uint32))
    mine.build("hashtable")
    assert ref.info() == mine.info()
    q = np.concatenate([np.array([r[:3] for r in rows], np.int32), rng.integers(-160, 160, size=(4000, 3)).astype(np.int32)])
    a, _ = ref.lookup(q)
    b, _ = mine.lookup(q)
    assert np.array_equal(a, b) and (a != po.EMPTY).sum() >= len(set(r[:3] for r in rows))
    ref.close(); mine.close()


def test_csv_reader_reports_a_field_that_is_not_a_number(tmp_path):
    rows, out = _dump(tmp_path, b"1,2,3,4\n5,x,7,8\n")
    assert rows is None and "line 2" in out and "field 2" in out          # (the reference dies there with an uncaught std::invalid_argument)


def _vox_chunk(cid, body, children=b""):
    return cid + struct.pack("<II", len(body), len(children)) + body + children


def _vox_dict(d):
    out = struct.pack("<I", len(d))
    for k, v in d.items():
        out += struct.pack("<I", len(k)) + k.encode() + struct.pack("<I", len(v)) + v.encode()
    return out


def test_magicavoxel_scene_graph_places_models(tmp_path):
    """nTRN / nGRP / nSHP: two models, three instances -- translated, translated + rotated, and nested under a translated group -- each
    placed about the model's centre floor(size / 2) the way MagicaVoxel does; z-up -> y-up; palette colours."""
    rng = np.random.default_rng(5)
    sizes = [(5, 4, 3), (2, 6, 2)]
    models = []
    for sx, sy, sz in sizes:
        pts = np.unique(np.stack([rng.integers(0, sx, 30), rng.integers(0, sy, 30), rng.integers(0, sz, 30)], 1), axis=0).astype(np.uint8)
        idx = rng.integers(1, 256, size=pts.shape[0]).astype(np.uint8)
        models.append((pts, idx))
    palette = rng.integers(0, 256, size=(256, 4)).astype(np.uint8)
    kids = b""
    for (sx, sy, sz), (pts, idx) in zip(sizes, models):
        kids += _vox_chunk(b"SIZE", struct.pack("<III", sx, sy, sz))
        kids += _vox_chunk(b"XYZI", struct.pack("<I", pts.shape[0]) + np.concatenate([pts, idx[:, None]], 1).tobytes())

    def trn(node, child, frame):
        return _vox_chunk(b"nTRN", struct.pack("<I", node) + _vox_dict({}) + struct.pack("<IiiI", child, -1, 0, 1) + _vox_dict(frame))

    def grp(node, children):
        return _vox_chunk(b"nGRP", struct.pack("<I", node) + _vox_dict({}) + struct.pack("<I", len(children)) + b"".join(struct.pack("<I", c) for c in children))

    def shp(node, model):
        return _vox_chunk(b"nSHP", struct.pack("<I", node) + _vox_dict({}) + struct.pack("<I", 1) + struct.pack("<I", model) + _vox_dict({}))
    rot = 1 | (0 << 2) | (1 << 4)            # rows: (0,-1,0), (1,0,0), (0,0,1) -> first row picks column 1 negated, second row column 0
    kids += trn(0, 1, {}) + grp(1, [2, 4, 6])
    kids += trn(2, 3, {"_t": "10 -20 7"}) + shp(3, 0)
    kids += trn(4, 5, {"_t": "-30 5 -4", "_r": str(rot)}) + shp(5, 1)
    kids += trn(6, 7, {"_t": "100 0 0"}) + grp(7, [8]) + trn(8, 9, {"_t": "0 50 1"}) + shp(9, 0)
    kids += _vox_chunk(b"RGBA", palette.tobytes())
    rows, out = _dump(tmp_path, b"VOX " + struct.pack("<I", 200) + _vox_chunk(b"MAIN", b"", kids))
    assert rows is not None, out

    def place(m, r, t):
        pts, idx = models[m]
        size = np.array(sizes[m], np.int64)
        c2 = 2 * pts.astype(np.int64) + 1 - size
        w = np.floor_divide(c2 @ np.array(r, np.int64).T, 2) + np.array(t, np.int64)
        pal = palette[idx.astype(np.int32) - 1].astype(np.int64)
        col = (pal[:, 0] << 16) | (pal[:, 1] << 8) | pal[:, 2]
        return [(int(a[0]), int(a[2]), int(a[1]), int(c)) for a, c in zip(w, col)]
    eye = [[1, 0, 0], [0, 1, 0], [0, 0, 1]]
    want = place(0, eye, (10, -20, 7)) + place(1, [[0, -1, 0], [1, 0, 0], [0, 0, 1]], (-30, 5, -4)) + place(0, eye, (100, 50, 1))
    assert sorted(rows) == sorted(want)
    assert rows[:len(models[0][0])] == want[:len(models[0][0])]             # load order: depth first from the root
