"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/observation_arrays.json from the UNMODIFIED reference.

    CAMPX_REFERENCE_ROOT=<checkout of the original CampX> python oracle/gen_golden_arrays.py

Runs the reference's `ObservationToArray` and `ObservationToFeatureArray` (campx/rendering.py:461-712) on
observations produced by the reference engine (boat_race and Hello World, under `oracle/shim.py`) for a
set of value mappings, dtypes and `permute` arguments, and records inputs (board) and outputs (shape, dtype,
flattened values), plus the exception class and message of the error cases.  Nothing is copied from the
reference; the fixture is what `tests/` checks the numpy oracle and the CUDA board mapper against.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import gen_golden as gg  # noqa: E402  (installs the shim)

BOAT_CHARS = " #<>A^v"
HELLO_CHARS = " #1234@"


def converter_specs(chars):
    rgb = {ch: [(37 * i) % 256, (91 * i + 5) % 256, 255 - 20 * i] for i, ch in enumerate(chars)}
    specs = []
    for permute in (None, [1, 2, 0], [2, 1, 0], [0, 2, 1], [2, 0, 1], [1, 0, 2]):
        specs.append({"kind": "array", "mapping": rgb, "dtype": "uint8", "permute": permute})
    specs.append({"kind": "array", "mapping": {ch: ord(ch) + 1 for ch in chars}, "dtype": None, "permute": None})
    specs.append({"kind": "array", "mapping": {ch: ord(ch) + 1 for ch in chars}, "dtype": None, "permute": [1, 0]})
    specs.append({"kind": "array", "mapping": {ch: 0.5 * i - 1.0 for i, ch in enumerate(chars)}, "dtype": None,
                  "permute": None})
    specs.append({"kind": "array", "mapping": {ch: [0.25 * i, -3.0 * i] for i, ch in enumerate(chars)},
                  "dtype": "float32", "permute": [1, 2, 0]})
    specs.append({"kind": "array", "mapping": {ch: [i, -i, 1000 * i, 7] for i, ch in enumerate(chars)},
                  "dtype": "int16", "permute": None})
    for permute in (None, [1, 2, 0], [2, 0, 1]):
        specs.append({"kind": "features", "layers": chars[4] + "#z" + chars[3], "permute": permute})
    specs.append({"kind": "features", "layers": chars, "permute": None})
    return specs


def build(rr, spec):
    if spec["kind"] == "array":
        mapping = {ch: (tuple(v) if isinstance(v, list) else v) for ch, v in spec["mapping"].items()}
        dtype = None if spec["dtype"] is None else np.dtype(spec["dtype"])
        return rr.ObservationToArray(mapping, dtype=dtype, permute=spec["permute"])
    return rr.ObservationToFeatureArray(spec["layers"], permute=spec["permute"])


def error_record(fn):
    try:
        fn()
    except Exception as e:      # noqa: BLE001  (the class and message are what is recorded)
        return {"type": type(e).__name__, "message": str(e)}
    return None


def main():
    from campx import rendering as rr
    cases = []
    for world, chars, actions in (("boat_race", BOAT_CHARS, [1, 1, 3, 3, 0]), ("hello", HELLO_CHARS, [0, 3, 1])):
        game, obs, _, _ = gg.make_ref_game(world)
        observations = [(obs.board + 0, {k: v + 0 for k, v in obs.layers.items()})]
        for a in actions:
            obs, _, _ = game.play(gg.encode_action(world, a))
            observations.append((obs.board + 0, {k: v + 0 for k, v in obs.layers.items()}))
        for spec in converter_specs(chars):
            conv = build(rr, spec)
            frames = []
            for board, layers in observations:
                out = np.array(conv(rr.Observation(board=board, layers=layers, layered_board=None)))
                frames.append({"board": "".join(chr(int(v)) for v in board.reshape(-1).tolist()),
                               "shape": list(out.shape), "dtype": out.dtype.name,
                               "values": out.reshape(-1).tolist()})
            cases.append({"world": world, "rows": int(board.shape[0]), "cols": int(board.shape[1]),
                          "characters": "".join(sorted(layers.keys())), "actions": actions, "spec": spec,
                          "frames": frames})
    game, obs, _, _ = gg.make_ref_game("boat_race")
    errors = [
        {"what": "unknown_character", "spec": {"kind": "array", "mapping": {"#": 1.0}, "dtype": None, "permute": None},
         "error": error_record(lambda: rr.ObservationToArray({"#": 1.0})(obs))},
        {"what": "no_such_feature", "spec": {"kind": "features", "layers": "xyz", "permute": None},
         "error": error_record(lambda: rr.ObservationToFeatureArray("xyz")(obs))},
        {"what": "bad_permute_3d", "spec": {"kind": "array", "mapping": {"#": [1, 2]}, "dtype": None, "permute": [0, 1]},
         "error": error_record(lambda: rr.ObservationToArray({"#": (1, 2)}, permute=(0, 1)))},
        {"what": "bad_permute_2d", "spec": {"kind": "array", "mapping": {"#": 1}, "dtype": None, "permute": [0, 1, 2]},
         "error": error_record(lambda: rr.ObservationToArray({"#": 1}, permute=(0, 1, 2)))},
        {"what": "bad_permute_features", "spec": {"kind": "features", "layers": "#", "permute": [0, 1]},
         "error": error_record(lambda: rr.ObservationToFeatureArray("#", permute=(0, 1)))},
    ]
    assert all(e["error"] is not None for e in errors)
    fx = {"source": "reference@%s campx/rendering.py ObservationToArray / ObservationToFeatureArray executed under "
                    "oracle/shim.py" % gg.REF_COMMIT,
          "generator": "oracle/gen_golden_arrays.py", "cases": cases, "errors": errors}
    path = os.path.join(gg.GOLDEN_DIR, "observation_arrays.json")
    with open(path, "w") as f:
        json.dump(fx, f, separators=(",", ":"))
    print(path, os.path.getsize(path), "bytes;", len(cases), "cases;", sum(len(c["frames"]) for c in cases), "frames")
    for e in errors:
        print(e["what"], e["error"]["type"])


if __name__ == "__main__":
    main()
