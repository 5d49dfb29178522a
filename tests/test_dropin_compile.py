"""Drop-in check of the scene-construction API (SURVEY.md §8 b1): the reference's OWN main.cpp — its nine scene builders,
`color()`, `de_nan()` and the sample loop with `cam.get_ray(u, v)` — is compiled, unchanged, against this repo's headers
(host/compat/*.h are one-line stand-ins for the reference's header names, host/rtnw/scene.hpp has the classes) and linked
with librtnw_host.so.  The builders taken from the reference's text are then run and flattened, and the tables must be
byte-identical to the ones the named scenes of the host library produce, i.e. what the GPU renders is the same.  Needs
a checkout of the reference project named by RTNW_REFERENCE; nothing from it is copied into the repo."""
import ctypes as C
import importlib
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "peter-shirley-ray-tracing-the-next-week_b200"
REF = Path(os.environ["RTNW_REFERENCE"]) / "Peter-Shirley-Project Code" if os.environ.get("RTNW_REFERENCE") else None
sys.path.insert(0, str(ROOT))
rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")

DRIVER = r'''
#define main reference_main            // keep the reference's main() (its sample loop must compile) but do not run it
#include "main.cpp"
#undef main
#include <cstdio>
#include "rtnw/flatten.hpp"
static void dump(FILE* f, const void* p, size_t n) { fwrite(&n, sizeof n, 1, f); if (n) fwrite(p, 1, n, f); }
int main(int argc, char** argv) {
    struct { const char* name; hitable* (*build)(); } scenes[] = {
        {"cornell_box", cornell_box}, {"cornell_smoke", cornell_smoke}, {"final", final}, {"simple_light", simple_light},
        {"two_spheres", two_spheres}, {"random_scene", random_scene}, {"test", test}};
    std::cout.setstate(std::ios_base::failbit);   // final() prints every box
    for (auto& s : scenes) {
        srand48(0x1234ABCD);                       // the never-seeded drand48 state, then the tables drawn before main()
        perlin::regenerate();
        hitable* world = s.build();
        rtnw::flat_scene flat;
        if (rtnw::flatten(world, flat) != 0) { fprintf(stderr, "flatten %s: %s\n", s.name, flat.error.c_str()); return 1; }
        const rtnw_scene_desc d = flat.desc();
        FILE* f = fopen((std::string(argv[1]) + "/" + s.name + ".bin").c_str(), "wb");
        dump(f, d.items, sizeof(rtnw_item) * d.n_items);
        dump(f, d.nodes, sizeof(rtnw_bvh_node) * d.n_nodes);
        dump(f, d.prims, sizeof(rtnw_prim) * d.n_prim_slots);
        dump(f, d.xforms, sizeof(rtnw_xform_op) * d.n_xform_ops);
        dump(f, d.materials, sizeof(rtnw_material) * d.n_materials);
        dump(f, d.textures, sizeof(rtnw_texture) * d.n_textures);
        fclose(f);
    }
    return 0;
}
'''


def _tables(d):
    def blob(ptr, n, size):
        return C.string_at(ptr, n * size) if n else b""
    parts = [blob(d.items, d.n_items, C.sizeof(rtnw.Item)), blob(d.nodes, d.n_nodes, C.sizeof(rtnw.BvhNode)),
             blob(d.prims, d.n_prim_slots, C.sizeof(rtnw.Prim)), blob(d.xforms, d.n_xform_ops, C.sizeof(rtnw.XformOp)),
             blob(d.materials, d.n_materials, C.sizeof(rtnw.Material)), blob(d.textures, d.n_textures, C.sizeof(rtnw.Texture))]
    return b"".join(len(p).to_bytes(8, "little") + p for p in parts)


@pytest.mark.skipif(REF is None or not (REF / "main.cpp").exists(), reason="RTNW_REFERENCE does not name a checkout of the reference project")
def test_reference_main_cpp_compiles_unchanged_and_builds_the_same_scenes(tmp_path):
    (tmp_path / "driver.cpp").write_text(DRIVER)
    exe = tmp_path / "driver"
    cmd = ["g++", "-std=gnu++14", "-O1", "-ffp-contract=off", "-w", f"-I{PKG / 'host' / 'compat'}", f"-I{PKG / 'host'}",
           f"-I{ROOT / 'include'}", f"-iquote{REF}", f"-I{tmp_path}", "-o", str(exe), str(tmp_path / "driver.cpp"),
           f"-L{PKG / 'lib'}", "-lrtnw_host", f"-Wl,-rpath,{PKG / 'lib'}"]
    # the reference's main.cpp is found through -iquote ONLY for the `#include "main.cpp"` line: its own `#include "sphere.h"`
    # etc. would also resolve there, so the file is compiled from a directory that holds nothing else
    ref_copy = tmp_path / "ref"
    ref_copy.mkdir()
    (ref_copy / "main.cpp").write_bytes((REF / "main.cpp").read_bytes())   # temp dir only, removed with it
    cmd[cmd.index(f"-iquote{REF}")] = f"-I{ref_copy}"
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([str(exe), str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    for name in ["cornell_box", "cornell_smoke", "final", "simple_light", "two_spheres", "random_scene", "test"]:
        hs = rtnw.HostScene(name)
        assert (out / f"{name}.bin").read_bytes() == _tables(hs.desc), f"{name}: tables differ from the named scene"
