"""Host-side logic that needs no GPU (and no compute call into the C-ABI library)."""


def test_plan_lanes_and_sync_marks():
    """Two-lane plan bookkeeping (engine.Plan): lane of every step and the fork / join edges, no GPU needed."""
    from rdfc_gan_b200.engine import Plan
    p = Plan()

    def add(name):
        p.steps.append(lambda s: None)
        p.names.append(name)

    add('stems')
    p.fork()
    p.lane(0); add('r.en2'); add('r.en3')
    p.lane(1); add('d.en2'); add('d.en3')
    p.join()
    p.fork()
    add('fuse1'); add('r.de5')
    p.lane(1); add('d.de5')
    p.join()
    add('fuse_depth')
    assert p.lanes() == [0, 0, 0, 1, 1, 0, 0, 1, 0]
    assert p.sync == {1: ['fork'], 5: ['join', 'fork'], 8: ['join']}


def test_umma_filter_packing_layout():
    """engine.pack_weight(umma=True), the filter layout of the tensor-core conv (train_ops.conv2d_nhwc packs with it too):
    [tap][Cin/8][CoutP][8] (bf16), padded to 16 output rows; host-side only (no kernel launch)."""
    import torch
    from rdfc_gan_b200.engine import pack_weight
    w = torch.randn(40, 64, 3, 3)
    p = pack_weight(w, umma=True)
    assert p.dtype == torch.bfloat16 and tuple(p.shape) == (9, 8, 48, 8)
    for tap, chunk, co, e in ((0, 0, 0, 0), (4, 3, 17, 5), (8, 7, 39, 7)):
        assert p[tap, chunk, co, e] == w[co, chunk * 8 + e, tap // 3, tap % 3].bfloat16()
    assert (p[:, :, 40:, :] == 0).all()
