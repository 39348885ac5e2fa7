"""Device BVH build (SURVEY.md section 8(f) row 4, mesh_desc_t::use_fast_bvh_build): structural validity of the radix tree
rc_build_lbvh returns, and bitwise parity of the image rendered over the acceleration structure built from it."""
import time

import numpy as np
import pytest

from ray_b200 import capi, cuda, host, scenes
from common import STORED, maybe_oracle

pytestmark = pytest.mark.gpu


def _random_boxes(n, seed, degenerate=False):
    rng = np.random.default_rng(seed)
    c = rng.random((n, 3), dtype=np.float32) * 20.0 - 10.0
    if degenerate:  # many identical centroids: equal Morton codes, the (code, rank) tie-break must keep the tree valid
        c[: n // 2] = c[0]
    e = rng.random((n, 3), dtype=np.float32) * 0.3
    return np.concatenate([c - e, c + e], axis=1).astype(np.float32)


@pytest.mark.parametrize("n,degenerate", [(2, False), (3, False), (1000, False), (1000, True), (300000, False)])
def test_radix_tree_is_a_valid_bvh(n, degenerate):
    boxes = _random_boxes(n, 7 + n, degenerate)
    ctx = cuda.Context()
    nodes, order = ctx.build_lbvh(boxes)
    ctx.close()
    assert np.array_equal(np.sort(order), np.arange(n, dtype=np.uint32))
    internal, leaves = nodes[: n - 1], nodes[n - 1:]
    assert (internal["count"] == 0).all() and (leaves["count"] == 1).all()
    assert np.array_equal(leaves["first"], np.arange(n, dtype=np.uint32))
    assert np.array_equal(leaves["mn"], boxes[order, :3]) and np.array_equal(leaves["mx"], boxes[order, 3:])
    # every node but the root is referenced exactly once
    refs = np.bincount(np.concatenate([internal["left"], internal["right"]]), minlength=2 * n - 1)
    assert refs[0] == 0 and (refs[1:] == 1).all()
    # boxes are the exact union of the children's boxes
    l, r = nodes[internal["left"]], nodes[internal["right"]]
    assert np.array_equal(internal["mn"], np.minimum(l["mn"], r["mn"]))
    assert np.array_equal(internal["mx"], np.maximum(l["mx"], r["mx"]))
    # reachable from the root: depth-first walk visits all 2n-1 nodes, leaf ranks in order (contiguous subtree ranges)
    seen, stack, ranks = 0, [0], []
    while stack:
        i = stack.pop()
        seen += 1
        if nodes["count"][i]:
            ranks.append(int(nodes["first"][i]))
        else:
            stack.append(int(nodes["right"][i]))
            stack.append(int(nodes["left"][i]))
    assert seen == 2 * n - 1 and ranks == list(range(n))


def _camera_only(desc):
    import copy
    d = copy.copy(desc)
    d.meshes, d.instances, d.lights, d.textures, d.materials = [], [], [], [], []
    d.env_map = d.back_map = capi.RS_INVALID
    return d


def _fast(desc):
    for m in desc.meshes:
        m.use_fast_bvh_build = True
    return desc


def test_fast_build_renders_bit_identically_to_the_reference_over_the_same_arrays():
    """hall-250k: meshes built on the device, image == the reference's stage functions over those arrays (bitwise; without
    the oracle library: the built-in sampler table and the stored digest); and the first-hit AOV equals the one of the
    SAH-built scene (same geometry, whatever the tree)."""
    o = maybe_oracle()
    w, h, spp = 960, 540, 2
    r = host.Renderer(w, h)
    if o is not None:
        r.set_sampler_table(o.pmj_table())
    t0 = time.time()
    s = scenes.build(_fast(scenes.hall("principled", w, h)), r.create_scene())
    t_fast = time.time() - t0
    assert r.render(s, (0, 0, w, h), 0, spp) == spp
    raw, dn = r.pixels(host.RAW), r.pixels(host.DEPTH_NORMALS)
    c = r.counters()
    if o is None:
        STORED.check("lbvh/fast_build_hall", raw, np.asarray([c["primary_rays"], c["secondary_rays"], c["shadow_rays"]]))
    else:
        cam_scene = scenes.build(_camera_only(scenes.hall("principled", w, h)), o.Scene(wide=True))
        ref, n_rays, n_shadow = o.view_render(s.view(), s.camera(), cam_scene, w, h, spp)
        assert c["primary_rays"] + c["secondary_rays"] == n_rays and c["shadow_rays"] == n_shadow
        assert np.array_equal(raw.view(np.uint32), ref.view(np.uint32))
        cam_scene.close()
    fast_nodes = s.node_count()
    s.close()

    t0 = time.time()
    s2 = scenes.build(scenes.hall("principled", w, h), r.create_scene())
    t_sah = time.time() - t0
    r.clear()
    assert r.render(s2, (0, 0, w, h), 0, spp) == spp
    dn2 = r.pixels(host.DEPTH_NORMALS)
    rel = np.abs(dn[..., 3] - dn2[..., 3]) / np.maximum(np.abs(dn2[..., 3]), 1e-3)
    assert float((rel > 1e-4).mean()) < 2e-3  # exact-t ties between coplanar neighbours may resolve differently
    print(f"scene build: fast {t_fast:.2f} s ({fast_nodes} nodes) vs SAH {t_sah:.2f} s ({s2.node_count()} nodes)")
    s2.close()
    r.close()
