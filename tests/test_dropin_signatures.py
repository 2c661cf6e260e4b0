"""Drop-in boundary (SURVEY.md §8b): every function, class and method of the reference's modules
exists in sift-based-od_b200/ under the same name with the same parameter list (extra parameters
must be optional and come last).  Compared on the syntax trees, so nothing is imported or run; the
reference side is the snapshot of its signatures below (the reference itself is not part of this
repository)."""
import ast
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
OURS = ROOT / "sift-based-od_b200"
MODULES = ["main", "PoseBin", "AffineParameters", "HoughTransform", "HoughTransformHelperFunctions",
           "PostProcessing", "SiftHelperFunctions", "VisualHelperFunctions", "GenerateDatabaseInfo"]

# name -> parameter list, as in the reference (file:line in SURVEY.md §8b)
SNAPSHOT = {
    "main": {"Main.__init__": "self", "Main.get_query_features": "self, path", "Main.run_matcher": "self",
             "Main.apply_hough_transform": "self, bins=15", "Main.get_valid_bins": "self, threshold=5",
             "Main.update_keypoint_pairs": "self", "Main.apply_affine_parameters": "self, threshold",
             "Main.post_process": "self", "Main.plot": "self"},
    "HoughTransform": {"perform_hough_transform":
                       "matching_keypoints, image_query, bin_x=15, bin_y=15, bin_theta=15, bin_sigma=15"},
    "HoughTransformHelperFunctions": {"estimate_object_pose": "data",
                                      "calculate_bin_index": "object_pose, bins, query_image_shape"},
    "AffineParameters": {"Gen_A": "x, y, votes", "Gen_b": "b_x, b_y, votes", "Calc_x": "A, b", "Ext_Params": "x",
                         "AffineParameters": "posebin",
                         "remove_outliers": "posebin, image_query_size, x_factor=8, y_factor=8"},
    "GenerateDatabaseInfo": {"save_object": "obj, filename"},
    "SiftHelperFunctions": {"get_centroid": "kp", "make_temp_kp": "kp", "unpack_sift_octave": "kpt", "make_kp": "temp_kp"},
}


def api(path: Path) -> dict[str, str]:
    out = {}
    for node in ast.parse(path.read_text()).body:
        if isinstance(node, ast.FunctionDef):
            out[node.name] = ast.unparse(node.args)
        elif isinstance(node, ast.ClassDef):
            for n in node.body:
                if isinstance(n, ast.FunctionDef):
                    out[f"{node.name}.{n.name}"] = ast.unparse(n.args)
    return out


def compatible(ref_args: str, our_args: str) -> bool:
    if ref_args == our_args:
        return True
    extra = our_args[len(ref_args):]
    return our_args.startswith(ref_args) and all("=" in p for p in extra.strip(", ").split(", ") if p)


@pytest.mark.parametrize("module", MODULES)
def test_same_names_and_parameters(module):
    ref = SNAPSHOT.get(module, {})
    ours = api(OURS / f"{module}.py")
    assert ref or module in ("VisualHelperFunctions", "PoseBin", "PostProcessing"), module
    for name, args in ref.items():
        assert name in ours, f"{module}.{name} is missing from the drop-in"
        assert compatible(args, ours[name]), f"{module}.{name}({ours[name]}) != reference ({args})"
