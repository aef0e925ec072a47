"""ObservationToArray / ObservationToFeatureArray (campx/rendering.py:461-712).

CPU: the numpy oracle against the reference-recorded fixture tests/golden/observation_arrays.json (made by
oracle/gen_golden_arrays.py), live against the reference where CAMPX_REFERENCE_ROOT names a checkout of it, and the constructor
errors of the host classes.  GPU: `campx_b200.rendering` (one `cx_board_mapper_apply` launch) against the
fixture, against the oracle on random boards of many geometries / dtypes / permutations, through real engine
observations, and at 2^20 boards through size-independent properties.
"""
import itertools
import json
import os

import numpy as np
import pytest

from oracle import campx_oracle as O
from oracle import shim


@pytest.fixture(scope="module")
def fixture(golden_dir):
    with open(os.path.join(golden_dir, "observation_arrays.json")) as f:
        return json.load(f)


def spec_mapping(spec):
    return {ch: (tuple(v) if isinstance(v, list) else v) for ch, v in spec["mapping"].items()}


def oracle_convert(spec, board, characters):
    if spec["kind"] == "array":
        dtype = None if spec["dtype"] is None else np.dtype(spec["dtype"])
        return O.observation_to_array(board, spec_mapping(spec), dtype=dtype, permute=spec["permute"])
    return O.observation_to_feature_array(board, characters, spec["layers"], permute=spec["permute"])


def frame_board(case, frame):
    return np.frombuffer(frame["board"].encode("latin-1"), dtype=np.uint8).reshape(case["rows"], case["cols"])


def test_oracle_matches_reference_fixture(fixture):
    n = 0
    for case in fixture["cases"]:
        for frame in case["frames"]:
            got = oracle_convert(case["spec"], frame_board(case, frame), case["characters"])
            assert list(got.shape) == frame["shape"], case["spec"]
            assert got.dtype.name == frame["dtype"], case["spec"]
            assert got.reshape(-1).tolist() == frame["values"], case["spec"]
            n += 1
    assert n == 150


def test_oracle_errors_match_reference_fixture(fixture):
    board = np.frombuffer(b"######A> ##^#v## < ######", dtype=np.uint8).reshape(5, 5)
    for rec in fixture["errors"]:
        exc = {"RuntimeError": RuntimeError, "ValueError": ValueError}[rec["error"]["type"]]
        with pytest.raises(exc) as ei:
            oracle_convert(rec["spec"], board, " #<>A^v")
        if exc is RuntimeError:
            assert str(ei.value) == rec["error"]["message"]


def test_host_classes_constructor_errors(fixture):
    """Same exception classes and messages as the reference's constructors (no GPU needed)."""
    from campx_b200 import rendering as R
    for rec in fixture["errors"]:
        if not rec["what"].startswith("bad_permute"):
            continue
        spec = rec["spec"]
        with pytest.raises(ValueError) as ei:
            if spec["kind"] == "array":
                R.ObservationToArray(spec_mapping(spec), permute=spec["permute"])
            else:
                R.ObservationToFeatureArray(spec["layers"], permute=spec["permute"])
        assert str(ei.value) == rec["error"]["message"]


@pytest.mark.skipif(not shim.reference_available(),
                    reason="needs a checkout of the original CampX (set CAMPX_REFERENCE_ROOT)")
def test_oracle_matches_live_reference():
    from oracle import gen_golden as gg
    from oracle import gen_golden_arrays as ga
    from campx import rendering as rr
    game, obs, _, _ = gg.make_ref_game("hello")
    rng = np.random.Generator(np.random.PCG64(5))
    for _ in range(6):
        obs, _, _ = game.play(int(rng.integers(0, 4)))
    board = np.asarray(obs.board)
    for spec in ga.converter_specs(ga.HELLO_CHARS):
        want = np.array(ga.build(rr, spec)(obs))
        got = oracle_convert(spec, board, "".join(sorted(obs.layers.keys())))
        assert got.dtype == want.dtype and got.shape == want.shape and (got == want).all(), spec


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------

def build_host(spec, **kw):
    from campx_b200 import rendering as R
    if spec["kind"] == "array":
        dtype = None if spec["dtype"] is None else np.dtype(spec["dtype"])
        return R.ObservationToArray(spec_mapping(spec), dtype=dtype, permute=spec["permute"], **kw)
    return R.ObservationToFeatureArray(spec["layers"], permute=spec["permute"])


class FakeObservation(object):
    def __init__(self, board, characters):
        self.board, self.characters = board, characters


@pytest.mark.gpu
def test_gpu_matches_reference_fixture(fixture):
    """All frames of a case form one batch [frames, rows, cols]; every element must equal the reference's."""
    import torch
    for case in fixture["cases"]:
        boards = np.stack([frame_board(case, f) for f in case["frames"]])
        obs = FakeObservation(torch.from_numpy(boards).cuda(), case["characters"])
        got = build_host(case["spec"])(obs)
        want_dtype = case["frames"][0]["dtype"]
        assert str(got.dtype) == "torch." + want_dtype, case["spec"]
        got = got.cpu().numpy()
        for k, frame in enumerate(case["frames"]):
            assert list(got[k].shape) == frame["shape"], case["spec"]
            assert got[k].reshape(-1).tolist() == frame["values"], (case["spec"], k)


@pytest.mark.gpu
def test_gpu_errors_match_reference_fixture(fixture):
    import torch
    board = torch.from_numpy(np.frombuffer(b"######A> ##^#v## < ######", dtype=np.uint8).reshape(1, 5, 5).copy()).cuda()
    obs = FakeObservation(board, " #<>A^v")
    for rec in fixture["errors"]:
        if rec["error"]["type"] != "RuntimeError":
            continue
        with pytest.raises(RuntimeError) as ei:
            build_host(rec["spec"])(obs)
        assert str(ei.value) == rec["error"]["message"]
    # check=False: no host synchronisation, no exception; known cells are still mapped
    conv = build_host({"kind": "array", "mapping": {"#": 1.0}, "dtype": None, "permute": None}, check=False)
    out = conv(obs).cpu().numpy()
    assert out.dtype == np.float64 and (out[0] == (board[0].cpu().numpy() == ord("#"))).all()


GEOMETRIES = [(1, 1), (1, 3), (2, 2), (5, 5), (3, 7), (13, 36), (16, 16), (9, 31), (64, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", GEOMETRIES)
def test_gpu_matches_oracle_on_random_boards(rows, cols):
    """Ragged batch sizes (CTA tile tails, unaligned tails), every permutation, element sizes 1/2/4/8."""
    import torch
    rng = np.random.Generator(np.random.PCG64(rows * 100 + cols))
    chars = " #A>@x"
    codes = np.frombuffer(chars.encode(), dtype=np.uint8)
    for n in (1, 3, 17, 272 if rows * cols <= 512 else 33):
        boards = codes[rng.integers(0, len(chars), size=(n, rows, cols))]
        d_boards = torch.from_numpy(boards).cuda()
        specs = []
        for dtype, depth in (("uint8", 3), ("int16", 2), ("float32", 5), ("float64", 1), ("int64", 2), ("bool", 1)):
            mapping = {}
            for i, ch in enumerate(chars):
                v = [(7 * i + 3 * k) % 2 if dtype == "bool" else (i + 1) * (k + 2) + (0 if dtype == "uint8" else -4)
                     for k in range(depth)]
                mapping[ch] = v
            for permute in list(itertools.permutations(range(3)))[:: (1 if n <= 3 else 2)] + [None]:
                specs.append({"kind": "array", "mapping": mapping, "dtype": dtype,
                              "permute": None if permute is None else list(permute)})
        specs.append({"kind": "array", "mapping": {ch: float(ord(ch)) / 3 for ch in chars}, "dtype": "float32",
                      "permute": [1, 0]})
        specs.append({"kind": "features", "layers": "A?@ ", "permute": [1, 2, 0]})
        specs.append({"kind": "features", "layers": "#x", "permute": None})
        for spec in specs:
            got = build_host(spec)(FakeObservation(d_boards, chars)).cpu().numpy()
            for k in (0, n // 2, n - 1):
                want = oracle_convert(spec, boards[k], chars)
                assert got[k].dtype == want.dtype and got[k].shape == want.shape, spec
                assert (got[k] == want).all(), (spec, n, k)


@pytest.mark.gpu
def test_gpu_engine_observations_and_single_env_shapes():
    """Through real engines: batched boat_race / Hello World observations and a num_envs=None engine."""
    import torch
    from campx_b200 import rendering as R
    from examples.worlds import make_world
    rgb = {ch: (i, 2 * i, 255 - i) for i, ch in enumerate(" #<>A^v")}
    game = make_world("boat_race", num_envs=64)
    obs, _, _ = game.its_showtime()
    to_rgb = R.ObservationToArray(rgb, dtype=np.uint8, permute=(1, 2, 0))
    feats = R.ObservationToFeatureArray("A#?", permute=None)
    rng = np.random.Generator(np.random.PCG64(3))
    for _ in range(5):
        obs, _, _ = game.play(torch.from_numpy(rng.integers(0, 5, size=64).astype(np.uint8)).cuda())
        img = to_rgb(obs).cpu().numpy()
        f = feats(obs)
        assert img.shape == (64, 5, 5, 3) and tuple(f.shape) == (64, 3, 5, 5) and f.dtype == torch.float32
        boards = obs.board.cpu().numpy()
        for k in (0, 31, 63):
            assert (img[k] == O.observation_to_array(boards[k], rgb, dtype=np.uint8, permute=(1, 2, 0))).all()
            assert (f[k].cpu().numpy() == O.observation_to_feature_array(boards[k], " #<>A^v", "A#?")).all()
        # the feature planes of game characters are the float layers of the observation
        assert torch.equal(f[:, 0], obs.layers["A"].float()) and torch.equal(f[:, 1], obs.layers["#"].float())
        assert float(f[:, 2].abs().sum()) == 0.0
    single = make_world("boat_race")
    obs, _, _ = single.its_showtime()
    assert tuple(to_rgb(obs).shape) == (5, 5, 3)
    assert tuple(R.ObservationToArray({ch: ord(ch) for ch in " #<>A^v"})(obs).shape) == (5, 5)
    with pytest.raises(RuntimeError):
        R.ObservationToFeatureArray("xyz")(obs)


@pytest.mark.gpu
def test_gpu_full_size_properties():
    """2^20 boat_race boards: RGB image is a per-cell function of the board; planes partition the board."""
    import torch
    from campx_b200 import rendering as R
    from examples.worlds import make_world
    n = 1 << 20
    game = make_world("boat_race", num_envs=n)
    game.its_showtime()
    acts = game.native.fill_actions(3, seed=9)
    for t in range(3):
        obs, _, _ = game.play(acts[t])
    chars = " #<>A^v"
    lut = torch.zeros((256, 3), dtype=torch.uint8, device="cuda")
    rgb = {}
    for i, ch in enumerate(chars):
        rgb[ch] = (10 * i + 1, 20 * i + 2, 30 * i + 3)
        lut[ord(ch)] = torch.tensor(rgb[ch], dtype=torch.uint8)
    img = R.ObservationToArray(rgb, dtype=np.uint8, permute=(1, 2, 0))(obs)
    assert tuple(img.shape) == (n, 5, 5, 3)
    assert torch.equal(img, lut[obs.board.long()])
    planes = R.ObservationToFeatureArray(chars)(obs)
    assert tuple(planes.shape) == (n, 7, 5, 5)
    assert torch.equal(planes.sum(dim=1), torch.ones((n, 5, 5), device="cuda"))
    assert torch.equal(planes, obs.layered_board_as(torch.float32))
