"""Host-side logic that needs no GPU: adjacency builders vs the reference's own adj_init output,
CSR/transposes, OBJ i/o, parameter layout and initialisation, sharding arithmetic."""
import types

import numpy as np
import pytest
import torch

import ptk_b200
from ptk_b200.graph import Graph


@pytest.mark.parametrize("tag,use_touch,finger", [("v", False, False), ("p", True, True), ("g", True, False)])
def test_adj_init_matches_reference(golden, objects_dir, tag, use_touch, finger):
    adj = golden("adjacency")
    args = types.SimpleNamespace(use_touch=use_touch, finger=finger, num_grasps=5)
    info, verts = ptk_b200.utils.load_mesh_vision(args, objects_dir + "/vision_charts.obj", device="cpu")
    assert verts.shape == (1824, 3)
    for which in ("origional", "adj"):
        g = Graph.from_dense(info[which])
        assert np.array_equal(g.host["rowptr"], adj[f"{tag}_{which}_rowptr"])
        assert np.array_equal(g.host["col"], adj[f"{tag}_{which}_col"])
        deg = np.diff(g.host["rowptr"])
        assert np.array_equal(g.host["val"], np.repeat(np.float32(1) / deg.astype(np.float32), deg))
    assert np.array_equal(info["faces"].numpy(), adj[f"{tag}_faces"])


def test_expected_graph_sizes(golden):
    adj = golden("adjacency")
    assert len(adj["p_adj_rowptr"]) - 1 == 1949 and len(adj["p_adj_col"]) == 24291
    assert len(adj["g_adj_rowptr"]) - 1 == 2324 and len(adj["g_adj_col"]) == 60726
    assert len(adj["v_adj_col"]) == 9888
    g = Graph.from_csr(adj["p_adj_rowptr"], adj["p_adj_col"], "cpu")
    assert g.n_hubs == 5 and g.n_hubs_t == 5
    assert list(g.hubs.numpy()) == [1824 + 25 * i + 4 for i in range(5)]


def test_transpose_csr(golden):
    adj = golden("adjacency")
    g = Graph.from_csr(adj["g_adj_rowptr"], adj["g_adj_col"], "cpu")
    d = g.dense()
    gt = Graph.from_dense(d.t().contiguous())
    assert np.array_equal(g.host["rowptr_t"], gt.host["rowptr"])
    assert np.array_equal(g.host["col_t"], gt.host["col"])
    assert np.array_equal(g.host["val_t"], gt.host["val"])


def test_graph_cache_keyed_on_version():
    a = torch.eye(4)
    g1 = ptk_b200.graph.graph_of(a)
    assert ptk_b200.graph.graph_of(a) is g1
    a[0, 1] = 0.5
    g2 = ptk_b200.graph.graph_of(a)
    assert g2 is not g1 and g2.nnz == 5


def test_obj_roundtrip(tmp_path, golden):
    m = golden("meshes")
    v, f = torch.from_numpy(m["touch_verts"]), torch.from_numpy(m["touch_faces"].astype(np.int64))
    p = tmp_path / "t.obj"
    ptk_b200.obj_io.save_obj(str(p), v, f)
    v2, faces, _ = ptk_b200.obj_io.load_obj(str(p))
    assert torch.equal(faces.verts_idx, f) and torch.allclose(v2, v, atol=1e-6)
    (tmp_path / "q.obj").write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nf 1/1/1 2/2/2 3/3/3 4/4/4\nf -1 -2 -3\n")
    _, faces, _ = ptk_b200.obj_io.load_obj(str(tmp_path / "q.obj"))
    assert faces.verts_idx.tolist() == [[0, 1, 2], [0, 2, 3], [3, 2, 1]]


def test_gcn_state_dict_layout_and_init(golden):
    torch.manual_seed(1234)
    args = types.SimpleNamespace(num_GCN_layers=20, hidden_GCN_size=300, cut=0.33)
    net = ptk_b200.GCN(50, args)
    sd = net.state_dict()
    assert sd["layers.0.weight"].shape == (1, 50, 300) and sd["layers.19.weight"].shape == (1, 300, 3)
    assert sd["layers.7.bias"].shape == (300,)
    assert net.layers[0].propagated() == 99 and net.layers[19].propagated() == 3
    # same RNG consumption as the reference's reset_parameters => same weights under the same seed
    g = golden("gcn")
    assert abs(net.layers[5].weight.double().sum().item() - g["p_default_w5_sum"][0]) < 1e-9


def test_shard_bounds_cover_everything():
    for n in (1, 7, 16, 1600):
        for w in (1, 2, 3, 8):
            spans = [ptk_b200.dist.shard_bounds(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_install_patches_reference_module():
    fake = types.SimpleNamespace()
    fake_model = types.SimpleNamespace(GCN=None, GCN_layer=None)
    try:
        ptk_b200.install(fake, [fake_model])
        assert fake.chamfer_distance is ptk_b200.utils.chamfer_distance
        assert fake.batch_sample is ptk_b200.utils.batch_sample
        assert fake_model.GCN is ptk_b200.GCN and fake_model.GCN_layer is ptk_b200.GCN_layer
        assert not hasattr(fake_model, "Encoder") and not hasattr(fake_model, "Graph_Model")
        # the autoencoder / DDQN modules: their GCN consumers and the Positional_Encoder copies are replaced too
        ae = types.SimpleNamespace(GCN_layer=None, Encoder=None, AutoEncoder=None, Positional_Encoder=None)
        ddqn = types.SimpleNamespace(GCN_layer=None, Graph_Model=None, Positional_Encoder=None, Encoder=None)
        ptk_b200.install(fake, [ae, ddqn])
        assert ae.Encoder is ptk_b200.model.Encoder and ae.Positional_Encoder is ptk_b200.Positional_Encoder
        assert ddqn.Graph_Model is ptk_b200.model.Graph_Model and ddqn.GCN_layer is ptk_b200.GCN_layer
        assert ddqn.Encoder is None  # an unrelated class called Encoder (no AutoEncoder beside it) is left alone
    finally:
        ptk_b200.uninstall()  # install() also switched ptk_b200.utils.face_draw; later tests expect the default
    assert ptk_b200.utils.face_draw == "uniform"


def test_encoder_mirrors_state_dict_layout():
    """Positional_Encoder / Mask_Encoder / Encoder / Graph_Model keep the reference's parameter names
    (vision/model.py:367-414, autoencoder/model.py:45-92, DDQN/model.py:65-101)."""
    pe, me = ptk_b200.Positional_Encoder(48), ptk_b200.Mask_Encoder(48)
    assert list(pe.state_dict()) == ["model.0.weight", "model.0.bias", "model.2.weight", "model.2.bias",
                                     "model.4.weight", "model.4.bias"]
    assert pe.model[0].weight.shape == (12, 63) and pe.model[4].weight.shape == (48, 24)
    assert list(me.state_dict()) == ["model.0.weight"] and me.model[0].weight.shape == (4, 48)
    enc = ptk_b200.model.Encoder(50, types.SimpleNamespace(num_GCN_layers=3, hidden_GCN_size=40, cut=0.33,
                                                           encoding_size=20))
    keys = list(enc.state_dict())
    assert keys[:6] == ["layers.0.weight", "layers.0.bias", "layers.1.weight", "layers.1.bias", "layers.2.weight",
                        "layers.2.bias"]
    assert keys[6:] == [f"mlp.{i}.0.{w}" for i in range(4) for w in ("weight", "bias")]
    assert enc.layers[2].do_cut is False and enc.layers[2].propagated() == 40 and enc.layers[0].propagated() == 13
    gm = ptk_b200.model.Graph_Model(types.SimpleNamespace(layers=2, hidden_dim=100, num_actions=50, cut=0.33),
                                    {"adj": torch.eye(3)})
    assert [tuple(l.weight.shape) for l in gm.layers] == [(1, 300, 100), (1, 100, 50)]
    assert "positional_embedding.model.4.weight" in gm.state_dict() and "mask_embedding.model.0.weight" in gm.state_dict()


def test_pytorch3d_shim_imports():
    ptk_b200.install_pytorch3d_shim()
    from pytorch3d.loss import chamfer_distance  # noqa: F401
    from pytorch3d.ops.mesh_face_areas_normals import mesh_face_areas_normals  # noqa: F401
    from pytorch3d.ops.sample_points_from_meshes import _rand_barycentric_coords
    from pytorch3d.io.obj_io import load_obj, save_obj  # noqa: F401
    w0, w1, w2 = _rand_barycentric_coords(2, 5, torch.float32, "cpu")
    assert torch.allclose(w0 + w1 + w2, torch.ones(2, 5))


def test_factor_hubs_is_exact_on_the_real_graphs_and_falls_back_otherwise(golden):
    """graph.factor_hubs: the reduced CSR + alpha * w on the common set reproduces the adjacency exactly for the
    fused touch graphs (forward and transpose), leaves hub-free graphs alone, and refuses non-rank-1 hub rows."""
    import numpy as np
    from ptk_b200.graph import Graph, factor_hubs
    adj = golden("adjacency")

    def dense(rowptr, col, val, n):
        a = np.zeros((n, n), np.float64)
        a[np.repeat(np.arange(n), np.diff(rowptr)), col] = val
        return a

    for tag, n_hubs in (("p", 5), ("g", 20)):
        g = Graph.from_csr(adj[f"{tag}_adj_rowptr"], adj[f"{tag}_adj_col"], "cpu")
        h = g.host
        for rp, col, val in ((h["rowptr"], h["col"], h["val"]), (h["rowptr_t"], h["col_t"], h["val_t"])):
            f = factor_hubs(rp, col, val, g.n)
            assert len(f["hubs"]) == n_hubs and len(f["common_col"]) > 1000
            assert f["row_skip"].sum() == n_hubs and (np.diff(f["rowptr"])[f["hubs"]] < 64).all()
            rec = dense(f["rowptr"], f["col"], f["val"], g.n)
            for hub, a in zip(f["hubs"], f["alpha"]):
                rec[hub, f["common_col"]] += np.float64(a) * f["common_w"].astype(np.float64)
            assert np.array_equal(rec.astype(np.float32), dense(rp, col, val, g.n).astype(np.float32))
    g0 = Graph.from_csr(adj["p_origional_rowptr"], adj["p_origional_col"], "cpu")
    assert g0.fwd_k.n_common == 0 and g0.fwd_k.n_hubs == 0
    # hub rows whose weights are not rank-1 on the shared columns must not be factored
    rng = np.random.default_rng(0)
    n = 400
    rows = [np.unique(np.append(rng.integers(0, n, 5), i)) for i in range(n)]
    shared = np.arange(100, 300)
    for hub in (3, 50):
        rows[hub] = np.unique(np.concatenate([rows[hub], shared]))
    rowptr = np.zeros(n + 1, np.int32)
    rowptr[1:] = np.cumsum([len(r) for r in rows])
    col = np.concatenate(rows).astype(np.int32)
    f = factor_hubs(rowptr, col, rng.random(len(col)).astype(np.float32), n)
    assert f["common_col"] is None and len(f["hubs"]) == 2


def test_faces_cache_never_serves_a_stale_copy_and_checks_the_id_range():
    """ADVICE r1 (high): a faces tensor freed and replaced by another one at the same address must not get the old
    int32 copy; ids outside [0, V) raise like torch indexing would instead of reading out of bounds."""
    import gc
    from ptk_b200.utils import _faces_i32
    g = torch.Generator().manual_seed(0)
    for _ in range(40):
        f = torch.randint(0, 50, (64, 3), generator=g)
        got = _faces_i32(f, 50)
        assert got.dtype == torch.int32 and torch.equal(got.long(), f)
        del f, got
        gc.collect()
    f = torch.randint(0, 50, (64, 3), generator=g)
    a = _faces_i32(f, 50)
    assert _faces_i32(f, 50) is a  # same live tensor, same version: cached
    f[0, 0] = 49  # in-place edit bumps the version
    assert _faces_i32(f, 50)[0, 0] == 49
    with pytest.raises(IndexError):
        _faces_i32(f, 49)
    with pytest.raises(IndexError):
        _faces_i32(torch.tensor([[0, 1, -1]]), 5)
    with pytest.raises(ValueError):
        _faces_i32(torch.zeros(4, 2, dtype=torch.int64), 5)


def test_tile_unions_index_every_entry_of_the_kernel_csr(golden):
    """graph.tile_unions (host side of ptk_gcn_aggregate_tiled): per tile of 8 rows the union is the sorted set of the
    non-hub rows' columns, every CSR entry's local index points back at its column, hub rows are left out, and the
    union is 2-3x smaller than the sum of the degrees on the real graphs (what the dense-tile kernel lives on)."""
    from ptk_b200 import graph as G
    adj = golden("adjacency")
    for name in ("p_adj", "g_adj", "p_origional"):
        rp, col = adj[name + "_rowptr"], adj[name + "_col"]
        n = len(rp) - 1
        deg = np.diff(rp)
        val = np.repeat((1.0 / deg).astype(np.float32), deg)
        f = G.factor_hubs(rp, col, val, n)
        skip = f["row_skip"] if f["row_skip"] is not None else (np.diff(f["rowptr"]) > G.HUB_DEG)
        uptr, ucol, lidx, max_union = G.tile_unions(f["rowptr"], f["col"], skip, n)
        krp, kcol = f["rowptr"], f["col"]
        n_tiles = (n + G.TILE_ROWS - 1) // G.TILE_ROWS
        assert len(uptr) == n_tiles + 1 and uptr[-1] == len(ucol) and max_union == np.diff(uptr).max() <= 256
        total_deg = 0
        for t in range(n_tiles):
            u = ucol[uptr[t]:uptr[t + 1]]
            assert np.all(np.diff(u) > 0)                                   # sorted, unique
            want = set()
            for i in range(t * G.TILE_ROWS, min(n, (t + 1) * G.TILE_ROWS)):
                if skip[i]:
                    continue
                c = kcol[krp[i]:krp[i + 1]]
                assert np.array_equal(u[lidx[krp[i]:krp[i + 1]]], c)        # local index -> the entry's column
                want.update(c.tolist())
                total_deg += len(c)
            assert set(u.tolist()) == want
        assert 2.0 < total_deg / len(ucol) < 3.5, (name, total_deg / len(ucol))
