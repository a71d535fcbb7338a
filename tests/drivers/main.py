"""Training driver of the upstream Dual-DMP project (astaka-pe/Dual-DMP ``main.py``), restated for the tests.

The upstream script is not part of this repository.  This restatement makes the calls its loop makes, in the same
order and through the same ``util`` modules, so that with ``dual_dmp_b200/dropin`` first on the path it exercises
the drop-in boundary the way the upstream driver does (SURVEY.md §3.1, INTEGRATION.md §2): flags (main.py:15-37), a
``viser`` server (:42-43, stubbed in tests/stubs), ``Datamaker.create_dataset`` (:46), ``PosNet(device).to(device)``
/ ``NormalNet`` with two ``torch.optim.Adam`` (:51-55), numpy ``Loss.mad`` (:60), the loop body (:87-110), every 10
epochs ``Mesh.compute_face_normals`` / ``compute_vert_normals`` through the class and ``Loss.mad`` (:117-123), every
100 epochs ``Mesh.save`` into ``<input>/output/<epoch>_ddmp=<mad>.obj`` (:125-127), and the final MAD (:149).
It imports nothing from the project except the ``util`` modules.
"""
import argparse
import os

import numpy as np
import torch
import viser
import viser.transforms  # noqa: F401
from tqdm import tqdm

import util.datamaker as Datamaker
import util.loss as Loss
import util.models as Models  # noqa: F401
from util.mesh import Mesh
from util.networks import NormalNet, PosNet


def get_parser():
    parser = argparse.ArgumentParser(description="Dual Deep Mesh Prior")
    parser.add_argument("-i", "--input", type=str, required=True)
    parser.add_argument("--pos_lr", type=float, default=0.01)
    parser.add_argument("--norm_lr", type=float, default=0.01)
    parser.add_argument("--norm_optim", type=str, default="Adam")
    parser.add_argument("--iter", type=int, default=1000)
    parser.add_argument("--k1", type=float, default=3.0)
    parser.add_argument("--k2", type=float, default=4.0)
    parser.add_argument("--k3", type=float, default=4.0)
    parser.add_argument("--k4", type=float, default=4.0)
    parser.add_argument("--k5", type=float, default=1.0)
    parser.add_argument("--grad_crip", type=float, default=0.8)
    parser.add_argument("--bnfloop", type=int, default=1)
    parser.add_argument("--gpu", type=int, default=0)
    parser.add_argument("--viewer", action="store_true", default=True)
    parser.add_argument("--port", type=int, default=8080)
    args = parser.parse_args()
    for k, v in vars(args).items():
        print("{:12s}: {}".format(k, v))
    return args


def main():
    args = get_parser()
    server = viser.ViserServer(port=args.port)

    mesh_dic, dataset = Datamaker.create_dataset(args.input)
    gt_mesh, n_mesh, o1_mesh = mesh_dic["gt_mesh"], mesh_dic["n_mesh"], mesh_dic["o1_mesh"]
    out_dir = os.path.join(args.input, "output")
    os.makedirs(out_dir, exist_ok=True)

    device = torch.device("cuda:" + str(args.gpu) if torch.cuda.is_available() else "cpu")
    posnet = PosNet(device).to(device)
    normnet = NormalNet(device).to(device)
    optimizer_pos = torch.optim.Adam(posnet.parameters(), lr=args.pos_lr)
    optimizer_norm = torch.optim.Adam(normnet.parameters(), lr=args.norm_lr)

    init_mad = Loss.mad(n_mesh.fn, gt_mesh.fn)
    print("initial_mad: {:.3f}".format(init_mad))

    with server.gui.add_folder("Training"):
        gui_mad = server.gui.add_number("MAD", initial_value=init_mad, disabled=True)
    server.scene.add_mesh_simple("/noisy", vertices=n_mesh.vs.astype(np.float32), faces=n_mesh.faces)

    mad_value = init_mad
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
            mad_value = Loss.mad(o1_mesh.fn, gt_mesh.fn)
            gui_mad.value = mad_value
            server.scene.add_mesh_simple("/output", vertices=o1_mesh.vs.astype(np.float32), faces=o1_mesh.faces)

        if epoch % 100 == 0:
            Mesh.save(o1_mesh, os.path.join(out_dir, "{}_ddmp={:.3f}.obj".format(epoch, mad_value)))

    print("final_mad: {:.3f}".format(mad_value))


if __name__ == "__main__":
    main()
