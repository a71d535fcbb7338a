#!/usr/bin/env python
"""Position error of meshes against a ground-truth mesh, on the GPU: the two-sided distance report of
``dual_dmp_b200.distance.hausdorff`` (vertex sampling; values also relative to the ground truth's bounding-box
diagonal, the figure upstream check/hausdorff_checker.py prints with MeshLab) for each mesh, one JSON line per file,
plus the mean angular difference of the face normals (``Loss.mad``, degrees) when the face counts match.

  python scripts/mesh_distance.py --gt X_gt.obj out/*.obj
  python scripts/mesh_distance.py --gt X_gt.obj --samples 1000000 [--seed S] out/*.obj

With ``--samples N`` each line also carries ``"surface"``: the report of ``dual_dmp_b200.distance.surface_distance``
with N area-weighted surface samples per mesh (distances that do not depend on either triangulation, and the normal
error across the nearest-face correspondence), for every file whatever its face count.

OBJ files are read with ``Mesh.fill_from_file``'s parser without building the mesh graph, so non-manifold scans are
accepted.  The ground truth's BVH (and its sampling prefix) is built once and reused for every file.
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
from dual_dmp_b200.distance import MeshBVH, hausdorff, surface_distance  # noqa: E402
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
    ap.add_argument("--samples", type=int, default=None, help="surface samples per mesh: adds \"surface\"")
    ap.add_argument("--seed", type=int, default=0, help="seed of the surface samples")
    args = ap.parse_args(argv)
    if args.samples is not None and not 1 <= args.samples < 1 << 31:
        ap.error(f"--samples must lie in [1, 2^31), got {args.samples}")
    if args.seed < 0:
        ap.error(f"--seed must be non-negative, got {args.seed}")
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
        if args.samples is not None:
            rep["surface"] = surface_distance((vs, faces), gt, args.samples, args.seed)
        print(json.dumps(rep), flush=True)


if __name__ == "__main__":
    main()
