"""CPU, world size 2 over gloo: the sharded upload of the view-split path carries a paged scan's texture pages, the page
of every triangle and the page table (each rank uploads its slice of every array and the slices are all-gathered)."""
import multiprocessing as mp
import os
import socket

import numpy as np
import torch
import torch.distributed as dist


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    from mvlm_b200 import synth
    from mvlm_b200.io_obj import Mesh
    from mvlm_b200.sharding import upload_mesh_sharded
    from mvlm_b200.utils.render3d import ObjRenderer3D, page_table

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    v, uv, t = synth.face_mesh(grid=30, seed=1)
    tri_page = (np.arange(len(t)) % 3 - 1).astype(np.int32)
    pages = [synth.face_texture(s, seed=s) for s in (17, 32)]
    mesh = Mesh(verts=v, tris=t, uvs=uv, texture=None, pages=pages, tri_page=tri_page)
    d = upload_mesh_sharded(ObjRenderer3D(device="cpu"), mesh)
    ok = all(np.array_equal(a.numpy(), b) for a, b in ((d.verts, v), (d.tris, t), (d.uvs, uv), (d.tri_page, tri_page),
                                                        (d.page_table, page_table(pages))))
    ok = ok and len(d.pages) == 2 and all(np.array_equal(a.numpy(), b) for a, b in zip(d.pages, pages))
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_sharded_upload_carries_pages_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)], res
