"""Driver for real scans of the upstream Dual-DMP project (astaka-pe/Dual-DMP ``main4real.py``), restated for the tests.

The upstream script is not part of this repository.  This restatement makes the calls its loop makes through the same
``util`` modules (SURVEY.md §3.3): the loop of tests/drivers/main.py without ground truth, so no MAD and no viewer,
with the CAD-style defaults k = 3, 0, 3, 4, 2 and bnfloop = 5 (main4real.py:18-24), and ``Mesh.save`` of the
prediction every 10 epochs into ``<input>/output/<epoch>_ddmp.obj`` (:80-83).  It imports nothing from the project
except the ``util`` modules.
"""
import argparse
import os

import torch
from tqdm import tqdm

import util.datamaker as Datamaker
import util.loss as Loss
import util.models as Models  # noqa: F401
from util.mesh import Mesh
from util.networks import NormalNet, PosNet


def get_parser():
    parser = argparse.ArgumentParser(description="Dual Deep Mesh Prior for real scans")
    parser.add_argument("-i", "--input", type=str, required=True)
    parser.add_argument("--pos_lr", type=float, default=0.01)
    parser.add_argument("--norm_lr", type=float, default=0.01)
    parser.add_argument("--iter", type=int, default=100)
    parser.add_argument("--k1", type=float, default=3.0)
    parser.add_argument("--k2", type=float, default=0.0)
    parser.add_argument("--k3", type=float, default=3.0)
    parser.add_argument("--k4", type=float, default=4.0)
    parser.add_argument("--k5", type=float, default=2.0)
    parser.add_argument("--grad_crip", type=float, default=0.8)
    parser.add_argument("--bnfloop", type=int, default=5)
    parser.add_argument("--gpu", type=int, default=0)
    args = parser.parse_args()
    for k, v in vars(args).items():
        print("{:12s}: {}".format(k, v))
    return args


def main():
    args = get_parser()
    mesh_dic, dataset = Datamaker.create_dataset(args.input)
    n_mesh, o1_mesh = mesh_dic["n_mesh"], mesh_dic["o1_mesh"]
    out_dir = os.path.join(args.input, "output")
    os.makedirs(out_dir, exist_ok=True)

    device = torch.device("cuda:" + str(args.gpu) if torch.cuda.is_available() else "cpu")
    posnet = PosNet(device).to(device)
    normnet = NormalNet(device).to(device)
    optimizer_pos = torch.optim.Adam(posnet.parameters(), lr=args.pos_lr)
    optimizer_norm = torch.optim.Adam(normnet.parameters(), lr=args.norm_lr)

    for epoch in tqdm(range(1, args.iter + 1)):
        posnet.train()
        normnet.train()
        optimizer_pos.zero_grad()
        optimizer_norm.zero_grad()

        pos = posnet(dataset)
        loss_pos1 = Loss.pos_rec_loss(pos, n_mesh.vs)
        loss_pos2 = Loss.mesh_laplacian_loss(pos, n_mesh)

        norm = normnet(dataset)
        loss_norm1 = Loss.norm_rec_loss(norm, n_mesh.fn)
        loss_norm2, _ = Loss.fn_bnf_loss(pos, norm, n_mesh, loop=args.bnfloop)
        if epoch <= 100:
            loss_norm2 = loss_norm2 * 0.0

        loss_pos3 = Loss.pos_norm_loss(pos, norm, n_mesh)

        loss = (args.k1 * loss_pos1 + args.k2 * loss_pos2 + args.k3 * loss_norm1 + args.k4 * loss_norm2
                + args.k5 * loss_pos3)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(normnet.parameters(), args.grad_crip)
        optimizer_pos.step()
        optimizer_norm.step()

        if epoch % 10 == 0:
            o1_mesh.vs = pos.to("cpu").detach().numpy().copy()
            Mesh.compute_face_normals(o1_mesh)
            Mesh.compute_vert_normals(o1_mesh)
            Mesh.save(o1_mesh, os.path.join(out_dir, "{}_ddmp.obj".format(epoch)))


if __name__ == "__main__":
    main()
