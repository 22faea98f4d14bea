"""SURVEY §8 row f4: the DTU on-disk formats and the checkpoint dictionary (mvs_b200/dtu.py) against what the UNMODIFIED reference
reads from the same files (tests/golden/dtu/ + tests/golden/dtu_formats.npz, written by oracle/make_golden_dtu.py) -- bit-exact,
the reference's quirks included."""
import os
import random

import numpy as np
import pytest
import torch

from mvs_b200 import dtu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = os.path.join(ROOT, "tests", "golden", "dtu")
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "dtu_formats.npz"))


@pytest.mark.parametrize("tag,cams", [("all", [0, 1, 2, 3]), ("sub02", [0, 2]), ("sub03", [0, 3])])
def test_camera_files_and_pairs(tag, cams):
    c = dtu.read_cameras(BASE, cams)
    for key in ("K", "R", "T", "d", "d_int"):
        got = np.stack(c[key])
        assert got.dtype == np.float64 and np.array_equal(got, GOLD[f"{tag}_{key}"]), key
    # pair.txt: the reference's control flow decides what is found (a view outside cam_list leaves its score line to be parsed as
    # a view line -- "sub03" pins that: the score lines start with 3, which IS in the list, and an empty pair array results)
    assert len(c["pairs"]) == int(GOLD[f"{tag}_n_pairs"])
    for k, p in enumerate(c["pairs"]):
        assert p.dtype == np.int64 and np.array_equal(p, GOLD[f"{tag}_pair{k}"])
    if tag == "all":
        assert [list(p) for p in c["pairs"]] == [[1, 2, 3], [0, 2, 3], [0, 1, 3], [0, 1, 2]]


def test_pfm_reader_matches_the_reference_including_its_endianness_rule():
    dep = os.path.join(BASE, "Depths", "scan1_train")
    for name in ("depth_map_0000.pfm", "depth_map_0001.pfm", "colour_0000.pfm"):
        got = dtu.load_pfm(os.path.join(dep, name))
        want = GOLD["pfm_" + name]
        assert got.shape == want.shape and got.dtype.kind == "f"
        assert np.array_equal(np.ascontiguousarray(got).view(np.uint32), want.view(np.uint32))      # bit-exact
    first = dtu.load_pfm(os.path.join(dep, "depth_map_0000.pfm"))
    assert first.shape == (5, 7) and np.all(first[0, :2] == 0) and 425 <= first[1:].min() <= first.max() <= 475
    # the same little-endian bytes under scale -1 are read BIG-endian by the reference (reversed PFM convention): not a depth map
    second = dtu.load_pfm(os.path.join(dep, "depth_map_0001.pfm"))
    assert not (425 <= float(np.nanmax(np.abs(second[1:]))) <= 475)
    names = dtu.depth_file_names(BASE, [0, 1], [1])
    assert [os.path.relpath(p, BASE) for p in names[0]] == list(GOLD["depth_file_names"])


def test_pfm_round_trip(tmp_path):
    g = np.random.default_rng(3)
    for shape, scale in (((6, 9), 1.0), ((4, 5, 3), -2.0), ((1, 1), 1.0)):
        img = g.random(shape).astype(np.float32)
        p = str(tmp_path / "x.pfm")
        dtu.write_pfm(p, img, scale)
        back = dtu.load_pfm(p)
        assert np.array_equal(back.reshape(img.shape), img)
    with open(str(tmp_path / "bad.pfm"), "wb") as f:
        f.write(b"P6\n2 2\n1.0\n" + b"\0" * 16)
    with pytest.raises(Exception, match="Invalid Header"):
        dtu.load_pfm(str(tmp_path / "bad.pfm"))


def test_resumable_sampler():
    random.seed(1234)
    items = list(range(40))
    s = dtu.ResumableSampler(items, i=2, batch_size=7)
    assert list(s) == list(GOLD["sampler_seq"]) and len(s) == int(GOLD["sampler_len"])
    assert items == list(GOLD["sampler_items_after"])                # the data list is shuffled in place, as the reference does
    assert list(dtu.ResumableSampler(list(range(10)), i=0, batch_size=14)) == list(range(10))
    assert len(dtu.ResumableSampler(list(range(10)), i=1, batch_size=14)) == 0


def test_checkpoint_dictionary_round_trip(tmp_path):
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 3), torch.nn.BatchNorm2d(4))
    opt = torch.optim.Adam(model.parameters(), lr=0.005)
    sch = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, mode="min", factor=0.8, patience=2, cooldown=4, min_lr=0.0001)
    model(torch.randn(2, 3, 8, 8)).sum().backward()
    opt.step()
    ck = dtu.checkpoint_dict(3, 99, model, opt, sch, [1.0, 0.5], [0.3], [0.2])
    assert tuple(ck) == dtu.CHECKPOINT_KEYS                          # train.py:111-121: same keys, same order
    path = dtu.checkpoint_name(str(tmp_path), "run", 3, 99)
    assert os.path.basename(path) == "run_3_99"
    torch.save(ck, path)
    model2 = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 3), torch.nn.BatchNorm2d(4))
    opt2 = torch.optim.Adam(model2.parameters(), lr=0.1)
    sch2 = torch.optim.lr_scheduler.ReduceLROnPlateau(opt2, mode="min", factor=0.8, patience=2, cooldown=4, min_lr=0.0001)
    start, b_idx, loss, a1, a2 = dtu.load_checkpoint(path, model2, opt2, sch2, epochs=10)
    assert (start, b_idx, loss, a1, a2) == (4, 99, [1.0, 0.5], [0.3], [0.2])
    for k, v in model.state_dict().items():
        assert torch.equal(v, model2.state_dict()[k])
    assert opt2.state_dict()["param_groups"][0]["lr"] == 0.005
    with pytest.raises(ValueError, match="epochs completed in ckpt: 4"):
        dtu.load_checkpoint(path, model2, opt2, sch2, epochs=4)      # train.py:172-175


def test_native_regulariser_loads_a_reference_shaped_checkpoint():
    """The model_state_dict of a reference checkpoint carries cost_volume_reg.* keys with the reference's shapes
    (model.py:68-98): they load into the drop-in CostVolumeReg unchanged."""
    import mvs_b200
    reg = mvs_b200.CostVolumeReg(device="cpu")
    shapes = {"conv_0_0.weight": (8, 32, 3, 3, 3), "conv_3_0.weight": (64, 32, 3, 3, 3), "deconv_3_0.weight": (64, 32, 3, 3, 3),
              "deconv_1_0.weight": (16, 8, 3, 3, 3), "conv_out.weight": (1, 8, 3, 3, 3), "BN_2.running_var": (32,)}
    sd = reg.state_dict()
    for k, shp in shapes.items():
        assert tuple(sd[k].shape) == shp
    other = mvs_b200.CostVolumeReg(device="cpu")
    other.load_state_dict({k: v.clone() + 1 for k, v in sd.items()}, strict=True)
    assert torch.equal(other.conv_2_1.weight, reg.conv_2_1.weight + 1)


def test_against_the_recorded_reference():
    """What the reference's data.py (`Cameras`, `load_depth`) returned for tests/golden/dtu, as oracle/make_golden_dtu.py recorded
    it in dtu_formats.npz: the same per-camera arrays, pairs and depth map, element for element."""
    mine = dtu.read_cameras(BASE, [0, 1, 2, 3])
    for key in ("K", "R", "T", "d", "d_int"):
        want = GOLD[f"all_{key}"]
        assert len(mine[key]) == len(want) and all(np.array_equal(a, b) for a, b in zip(want, mine[key])), key
    assert len(mine["pairs"]) == int(GOLD["all_n_pairs"])
    assert all(np.array_equal(GOLD[f"all_pair{k}"], p) for k, p in enumerate(mine["pairs"]))
    p = os.path.join(BASE, "Depths", "scan1_train", "depth_map_0000.pfm")
    assert np.array_equal(GOLD["pfm_depth_map_0000.pfm"], dtu.load_pfm(p))
