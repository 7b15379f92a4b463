"""Shared helpers for the tests: fixture loading and a Gmsh 2.2 ASCII writer."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MESHES = ["one_wall", "sphere", "cylinder", "pore_small", "pore", "pore_without_dna"]
# mesh fixture -> config that goes with it
CASES = {"one_wall": "one_wall", "sphere": "sphere", "cylinder": "cylinder", "pore_small": "pore", "pore": "pore",
         "pore_without_dna": "pore_without_dna"}  # (generated mesh: scripts/make_pore_without_dna_mesh.py)


def load_mesh_arrays(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in ("x", "y", "tri", "ba", "bb", "bphys")}


def cfg_path(name):
    return os.path.join(GOLDEN, CASES.get(name, name) + ".cfg")


def hub_mesh(spokes, rings, boundary=False, hub_at="first", seed=0):
    """A polar mesh around one hub vertex of `spokes` triangles: a full disc (closed fan, valence `spokes`) or, with
    `boundary`, a half disc with the hub on the straight edge (open fan, valence spokes + 1).  Rings of vertices at radii
    1..rings; each quad between two rings is split along a random diagonal, so other vertices have valences 3 to 8.
    `hub_at` ("first", "middle", "last") places the hub's vertex index and its fan's block of triangles, i.e. its row in
    vertex order and in first-touch order.  Every triangle's corners are rotated at random and its orientation is
    flipped with probability 1/2; every boundary segment is reversed with probability 1/2.  Physical tags come in runs
    of two segments and cycle through shape_cfg's four surfaces as 0, 2, 1, 3, so that a vertex inside a run touches one
    surface and a vertex between runs two: two Dirichlet surfaces, a Dirichlet and a Neumann one, or two Neumann ones.  The two segments at a boundary hub are tagged 1 (Neumann).  y > 0 everywhere."""
    rng = np.random.RandomState(seed)
    n = spokes + 1 if boundary else spokes                   # vertices per ring
    th = (np.pi if boundary else 2.0 * np.pi) * np.arange(n) / spokes
    r = np.repeat(np.arange(1, rings + 1, dtype=np.float64), n)
    x = np.concatenate([[0.0], r * np.cos(np.tile(th, rings))])
    y = np.concatenate([[0.0], r * np.sin(np.tile(th, rings))]) + (1.0 if boundary else rings + 1.0)
    ring = lambda j, k: 1 + j * n + k % n                     # noqa: E731 -- vertex k of ring j (0 = innermost)
    fan = [(0, ring(0, k), ring(0, k + 1)) for k in range(spokes)]
    quads = []
    for j in range(rings - 1):
        for k in range(spokes):
            a0, a1, b0, b1 = ring(j, k), ring(j, k + 1), ring(j + 1, k), ring(j + 1, k + 1)
            quads += [(a0, a1, b1), (a0, b1, b0)] if rng.rand() < 0.5 else [(a0, a1, b0), (a1, b1, b0)]
    cut = {"first": 0, "middle": len(quads) // 2, "last": len(quads)}[hub_at]
    tri = np.array(quads[:cut] + fan + quads[cut:], dtype=np.int64)
    tri = np.stack([np.roll(t, rng.randint(3)) for t in tri])
    flip = rng.rand(len(tri)) < 0.5
    tri[flip] = tri[flip][:, ::-1]
    seg = [(ring(rings - 1, k), ring(rings - 1, k + 1)) for k in range(spokes)]
    if boundary:  # the straight edge, through the hub
        line = [ring(j, spokes) for j in range(rings - 1, -1, -1)] + [0] + [ring(j, 0) for j in range(rings)]
        seg += list(zip(line[:-1], line[1:]))
    seg = np.array(seg, dtype=np.int64)
    rev = rng.rand(len(seg)) < 0.5
    seg[rev] = seg[rev][:, ::-1]
    # the hub's vertex index: first, middle or last
    nv = len(x)
    pos = {"first": 0, "middle": nv // 2, "last": nv - 1}[hub_at]
    new = np.concatenate([[pos], np.arange(nv - 1) + (np.arange(nv - 1) >= pos)])  # old index -> new index
    old = np.empty(nv, dtype=np.int64)
    old[new] = np.arange(nv)
    bphys = np.array([0, 2, 1, 3])[(np.arange(len(seg)) // 2) % 4]
    if boundary:
        bphys[spokes + rings - 1:spokes + rings + 1] = 1
    return dict(x=x[old], y=y[old], tri=new[tri].astype(np.int32), ba=new[seg[:, 0]].astype(np.int32),
                bb=new[seg[:, 1]].astype(np.int32), bphys=bphys.astype(np.int32))


# Meshes that reach the kernels' capacity fallbacks and mixed orientations (tests/test_host_mesh_shapes.py states which
# shape reaches which fallback): name -> (hub_mesh arguments, refinement levels).
SHAPES = {
    "hub9": (dict(spokes=9, rings=3, boundary=False, hub_at="first", seed=1), 0),
    "hub16": (dict(spokes=16, rings=9, boundary=False, hub_at="middle", seed=2), 0),
    "hub17": (dict(spokes=17, rings=9, boundary=False, hub_at="last", seed=3), 0),
    "hub16_open": (dict(spokes=16, rings=5, boundary=True, hub_at="middle", seed=4), 0),
    "hub600": (dict(spokes=600, rings=3, boundary=False, hub_at="first", seed=5), 0),
    "hub600_open": (dict(spokes=600, rings=3, boundary=True, hub_at="middle", seed=6), 0),
    "hub636_last": (dict(spokes=636, rings=3, boundary=False, hub_at="last", seed=7), 0),
    "hub600_ref2": (dict(spokes=600, rings=5, boundary=False, hub_at="middle", seed=8), 2),
}


def shape_arrays(name):
    """the unrefined arrays of SHAPES[name] and its refinement levels"""
    kw, levels = SHAPES[name]
    return hub_mesh(**kw), levels


def shape_cfg(path, cylindrical=1):
    """A config for the hub meshes: Dirichlet surfaces 0 and 2, Neumann surfaces 1 and 3 with non-zero fluxes of the
    potential and of both concentrations (each surface has the same type for all three components)."""
    surf = [("0", "0", "0.06", "0.06"), ("1", "0.3", "0.02", "-0.015"), ("0", "1.5", "0.05", "0.07"),
            ("1", "-0.2", "0.01", "0.03")]
    text = ("[system]\nn_surfaces=4\nverbosity=0\ncylindrical=%d\nl_b=1\nlinearSolverIterations=5000\n"
            "newtonReassembleThreshold=0.0\nnewtonReduction=1e-08\nnewtonMinLinearReduction=1e-08\nnewtonMaxIterations=50\n"
            "newtonLineSearchMaxIteration=500\nc0=0.06\ntau=0.1\nprintStiffnessMatrix=0\noutputFreq=1\nnSteps=1\n"
            "potentialUpdateFreq=1\n\n[mesh]\nfilename=hub.msh\n" % cylindrical)
    for s, (bt, phi, cp, cm) in enumerate(surf):
        if bt == "0":
            text += ("\n[surface_%d]\ncoulombBtype=0\ncoulombPotential=%s\nplusDiffusionBtype=0\nplusDiffusionConcentration=%s\n"
                     "minusDiffusionBtype=0\nminusDiffusionConcentration=%s\n" % (s, phi, cp, cm))
        else:
            text += ("\n[surface_%d]\ncoulombBtype=1\ncoulombFlux=%s\nplusDiffusionBtype=1\nplusDiffusionFlux=%s\n"
                     "minusDiffusionBtype=1\nminusDiffusionFlux=%s\n" % (s, phi, cp, cm))
    with open(path, "w") as f:
        f.write(text)
    return path


def write_gmsh(path, a, node_id_offset=1, shuffle_nodes=False, extra_nodes=0):
    """Writes mesh arrays as Gmsh 2.2 ASCII: line elements first (file order = boundary segment order),
    then triangles.  Node ids are 1-based; `extra_nodes` appends unused nodes (the reader must skip them)."""
    nv = len(a["x"])
    ids = np.arange(nv) + node_id_offset
    with open(path, "w") as f:
        f.write("$MeshFormat\n2.2 0 8\n$EndMeshFormat\n$Nodes\n%d\n" % (nv + extra_nodes))
        order = np.arange(nv)
        if shuffle_nodes:
            order = np.random.RandomState(0).permutation(nv)
        for i in order:
            f.write("%d %.17g %.17g 0\n" % (ids[i], a["x"][i], a["y"][i]))
        for k in range(extra_nodes):
            f.write("%d 99 99 0\n" % (nv + node_id_offset + k))
        f.write("$EndNodes\n$Elements\n%d\n" % (len(a["ba"]) + len(a["tri"])))
        eid = 1
        for s in range(len(a["ba"])):
            f.write("%d 1 2 %d %d %d %d\n" % (eid, a["bphys"][s], 100 + a["bphys"][s], ids[a["ba"][s]], ids[a["bb"][s]]))
            eid += 1
        for t in a["tri"]:
            f.write("%d 2 2 7 8 %d %d %d\n" % (eid, ids[t[0]], ids[t[1]], ids[t[2]]))
            eid += 1
        f.write("$EndElements\n")
