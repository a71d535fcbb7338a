#!/usr/bin/env python
"""Position error of meshes against a ground-truth mesh, on the GPU: the two-sided distance report of
``dual_dmp_b200.distance.hausdorff`` (vertex sampling; values also relative to the ground truth's bounding-box
diagonal, the figure upstream check/hausdorff_checker.py prints with MeshLab) for each mesh, one JSON line per file,
plus the mean angular difference of the face normals (``Loss.mad``, degrees) when the face counts match.

  python scripts/mesh_distance.py --gt X_gt.obj out/*.obj

OBJ files are read with ``Mesh.fill_from_file``'s parser without building the mesh graph, so non-manifold scans are
accepted.  The ground truth's BVH is built once and reused for every file.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from dual_dmp_b200 import synth  # noqa: E402
from dual_dmp_b200.distance import MeshBVH, hausdorff  # noqa: E402
from dual_dmp_b200.util import loss as L  # noqa: E402
from dual_dmp_b200.util.mesh import Mesh  # noqa: E402


def load_obj(path):
    """(vs float64 [V,3], faces int64 [F,3]) from an OBJ file"""
    return Mesh.fill_from_file(Mesh.__new__(Mesh), path)


def main(argv=None) -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--gt", required=True, help="ground-truth OBJ")
    ap.add_argument("meshes", nargs="+", help="OBJ files to measure against the ground truth")
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args(argv)
    gt_vs, gt_faces = load_obj(args.gt)
    gt = MeshBVH(gt_vs, gt_faces, args.device)
    gt_fn = None
    for path in args.meshes:
        vs, faces = load_obj(path)
        rep = {"file": path, **hausdorff((vs, faces), gt)}
        if len(faces) == len(gt_faces):
            if gt_fn is None:
                gt_fn = synth.face_normals_areas(gt_vs, gt_faces)[0]
            rep["mad"] = float(L.mad(synth.face_normals_areas(vs, faces)[0], gt_fn))
        print(json.dumps(rep), flush=True)


if __name__ == "__main__":
    main()
