"""Host-side logic that needs no GPU: checkpoint format bridge (SURVEY section 5 / 8f-3)."""
def test_checkpoint_format_round_trip(tmp_path):
    """scripts/train.py:207-212 dictionary: written by learn.save_checkpoint, read by learn.load_or_initialize_model, and
    its model_state_dict has the reference's 104 tensors (SURVEY section 5) — CPU only, no kernels involved."""
    import torch
    from knightvision_b200 import learn as LR
    from knightvision_b200.model import ChessNet
    torch.manual_seed(0)
    net = ChessNet()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    p = str(tmp_path / "best_model.pth")
    LR.save_checkpoint(p, net, opt, epoch=3, loss=1.25)
    ck = torch.load(p, map_location="cpu")
    assert set(ck) == {"epoch", "model_state_dict", "optimizer_state_dict", "loss"} and ck["epoch"] == 3
    keys = list(ck["model_state_dict"])
    assert len(keys) == 104 and keys[0] == "conv1.weight" and "res_blocks.4.bn2.running_var" in keys
    assert sum(v.numel() for k, v in ck["model_state_dict"].items() if not k.endswith("num_batches_tracked")
               and "running" not in k) == 25381642                          # the reference's parameter count
    net2, opt2, ep = LR.load_or_initialize_model(p, "cpu")
    assert ep == 3 and all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), net2.state_dict().values()))
    torch.save({"module." + k: v for k, v in net.state_dict().items()}, str(tmp_path / "bare.pth"))   # DataParallel-style
    net3, _, ep3 = LR.load_or_initialize_model(str(tmp_path / "bare.pth"), "cpu")
    assert ep3 == 0 and torch.equal(net3.conv2.weight, net.conv2.weight)
    _, _, ep4 = LR.load_or_initialize_model(str(tmp_path / "missing.pth"), "cpu")
    assert ep4 == 0



def test_whole_tower_task_order():
    """kv_tower_order.h (the schedule of tower_umma2_kernel): every (layer, board tile, channel tile) exactly once; a tile
    comes after the tiles it reads — (l-1, m, *) — by at least a round of the 74 CTA pairs (or the 4-CTA clusters) whenever
    a chunk is large enough, so the dependency waits of the kernel do not spin; chunks are contiguous and differ by at
    most one board tile."""
    import numpy as np
    from simt_emu import emu
    cases = [(1024, 2, 11, 74, 74), (508, 2, 11, 74, 74), (1, 2, 11, 74, 74), (75, 2, 3, 74, 74), (149, 1, 40, 148, 74),
             (300, 1, 40, 148, 74), (7, 2, 11, 1, 74), (1024, 2, 11, 0, 74), (223, 2, 11, 74, 74), (625, 2, 11, 74, 74)]
    # what tests/test_gpu_shapes.py runs: 1, 5, 130 and 1 201 boards (1, 2, 33, 301 board tiles), towers of 1-5 layers,
    # 256 or 512 channels, KV_TOWER_CHUNK 1, 2, 3 and the defaults (74 tiles at 512 channels, 148 at 256) ...
    cases += [(M, NT, nl, ct, 74) for M in (1, 2, 33, 301) for NT in (1, 2) for nl in (1, 2, 3, 5)
              for ct in (1, 2, 3, 74, 148)]
    # ... and the 4-CTA-cluster kernel at the default chunk: tiles in pairs (1, 17, 151, and the hybrid launch's slice
    # of 268 tiles = 134 pairs), half the chunk, a round of at most 37 clusters
    cases += [(M, NT, nl, ct, 37) for M in (1, 17, 134, 151) for NT in (1, 2) for nl in (1, 2, 3, 5) for ct in (37, 74)]
    for M, NT, nl, ct, rnd in cases:
        o = emu.tower_order(M, NT, nl, ct)
        assert len(o) == nl * M * NT
        key = (o[:, 0].astype(np.int64) * M + o[:, 1]) * NT + o[:, 2]
        assert len(np.unique(key)) == len(key) and key.min() == 0 and key.max() == len(key) - 1
        pos = np.empty(len(key), np.int64)
        pos[key] = np.arange(len(key))
        m = np.arange(M)
        dmin = None
        for l in range(1, nl):
            for n in range(NT):
                for n2 in range(NT):
                    d = (pos[(l * M + m) * NT + n] - pos[((l - 1) * M + m) * NT + n2]).min()
                    dmin = d if dmin is None else min(dmin, d)
        assert dmin is None or dmin > 0
        if dmin is not None and ct * NT >= rnd and M >= ct:
            assert dmin >= rnd            # inputs finished at least one full round of the CTA pairs (clusters) earlier
        if ct > 0 and M >= 2 * ct:        # depth-first: the layer-0 tasks of a chunk are contiguous, chunks are balanced
            idx = np.flatnonzero(o[:, 0] == 0)
            cuts = np.flatnonzero(np.diff(idx) > 1)
            sizes = np.diff(np.concatenate([[0], cuts + 1, [len(idx)]])) // NT
            assert sizes.max() - sizes.min() <= 1 and sizes.min() >= ct and sizes.sum() == M


def test_hybrid_tower_slices_partition_the_board_tiles():
    """The two kernels of the hybrid tower launch split the board tiles without gap or overlap; the cluster kernel's share
    is even (it takes tiles in pairs) and proportional to its SMs."""
    from simt_emu import emu
    for M in (0, 1, 2, 3, 37, 132, 133, 625, 1024, 4097):
        assert emu.tower_slice(0, 132, 148, M) == (0, M)
        o1, c1 = emu.tower_slice(1, 132, 148, M)
        o2, c2 = emu.tower_slice(2, 132, 148, M)
        assert o1 == 0 and c1 % 2 == 0 and o2 == c1 and c1 + c2 == M
        assert abs(c1 - M * 132 / 148) < 2


def test_float64_network_reference_matches_golden():
    """The float64 graph of tests/test_gpu_shapes.py (the network reference of its per-layer and schedule tests)
    reproduces tests/golden/net_wide.npz, the UNMODIFIED reference ChessNet in fp32: the reference architecture with
    BatchNorm statistics (ref_bnrand_*) and the 20 x 256 tower (t20_*), within 2e-4 — CPU only."""
    import numpy as np
    import torch
    import helpers as H
    from oracle import kv_oracle as O
    from netref import Fp64Net, bnrand_net
    g = np.load(H.GOLDEN + "/net_wide.npz")
    for prefix, kw in (("ref_bnrand", {}), ("t20", dict(stem=256, tower=256, blocks=20, conv2=False))):
        n = 8
        net = bnrand_net(seed=2 if kw else 0, **kw)
        with torch.no_grad():
            p, v = Fp64Net(net, "cpu").forward(torch.from_numpy(O.encode(g["lines"][:n])))
        p, v = p.numpy(), v.numpy()
        d_cols = np.abs(np.take_along_axis(p, g["cols"][:n].astype(np.int64), axis=1) - g[prefix + "_cols"][:n]).max()
        d_top = np.abs(np.take_along_axis(p, g[prefix + "_top_idx"][:n].astype(np.int64), axis=1)
                       - g[prefix + "_top_val"][:n]).max()
        d_val = np.abs(v - g[prefix + "_value"][:n]).max()
        assert max(d_cols, d_top, d_val) < 2e-4, (prefix, d_cols, d_top, d_val)
