"""Loaders for the reference's on-disk formats (raceline CSV, ROS map yaml + image)."""
import numpy as np

from f1tenth_planning_b200 import io


def test_map_round_trip(tmp_path):
    from PIL import Image
    rng = np.random.default_rng(0)
    img = rng.choice([0, 205, 254], size=(40, 60), p=[0.2, 0.1, 0.7]).astype(np.uint8)
    Image.fromarray(img).save(tmp_path / "m.pgm")
    (tmp_path / "m.yaml").write_text("image: m.pgm\nresolution: 0.05\norigin: [-1.5, 2.0, 0.0]\n"
                                     "negate: 0\noccupied_thresh: 0.65\nfree_thresh: 0.196\n")
    occ, origin, res = io.load_map(str(tmp_path / "m.yaml"))
    assert occ.shape == (40, 60) and origin == (-1.5, 2.0) and res == 0.05
    # black (0) occupied, 254 free, 205 unknown -> occupied; row 0 is the bottom image row
    assert np.array_equal(occ, (img[::-1] != 254).astype(np.uint8))
    (tmp_path / "n.yaml").write_text("image: m.pgm\nresolution: 0.05\norigin: [0, 0, 0]\nnegate: 1\n"
                                     "occupied_thresh: 0.65\nfree_thresh: 0.196\n")
    occ_n, _, _ = io.load_map(str(tmp_path / "n.yaml"))
    assert np.array_equal(occ_n, (img[::-1] != 0).astype(np.uint8))


def test_raceline_layouts(tmp_path):
    a = np.arange(15, dtype=np.float64).reshape(3, 5)
    p5 = tmp_path / "a.csv"
    p5.write_text("#x_m ; y_m ; vx_mps ; psi_rad ; kappa_radpm\n" +
                  "\n".join(";".join("%.7f" % v for v in r) for r in a))
    assert np.array_equal(io.load_raceline(str(p5)), a)
    b = np.arange(21, dtype=np.float64).reshape(3, 7)
    p7 = tmp_path / "b.csv"
    p7.write_text("# id\n# hash\n# s_m; x_m; y_m; psi_rad; kappa_radpm; vx_mps; ax_mps2\n" +
                  "\n".join("; ".join("%.7f" % v for v in r) for r in b))
    assert np.array_equal(io.load_raceline(str(p7)), b[:, [1, 2, 5, 3, 4]])
