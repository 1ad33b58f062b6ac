"""Launch geometry of the fused kernels, restated from their launchers, and a guard that reads the geometry a call really launched
from a torch.profiler trace.

The parity tests that use these pick their batch sizes from the mirror below, so that they run the kernels at the games per CTA,
warps per CTA, groups per warp and shared-memory padding that bench.py and the training loops launch.  The guard then asserts that
the call launched exactly that: when a launcher changes its rules, the tests fail and say so instead of quietly testing a smaller
geometry.  Every function cites the launcher it restates."""
import json
import os
import subprocess
import sys
from collections import namedtuple

import torch

from tron_b200 import abi

Launch = namedtuple("Launch", "name args grid block smem")
Geometry = namedtuple("Geometry", "kernel args G grid block smem")

KB = 1024


def sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _ceil(a, b):
    return -(-a // b)


def _r16(x):
    return (x + 15) & ~15


def _es(dt):
    return abi.dtype_size(dt)


def _lp_cp(enc):
    """step_dispatch.cuh:17-28 (dispatch_obs): enc -> (lut planes, const plane)"""
    return {abi.ENC_LUT1: (1, False), abi.ENC_POPUP3: (3, False), abi.ENC_POPUP3_CONST: (3, True)}[enc]


def _b(v):
    return "true" if v else "false"


def smem_for_ctas_per_sm(smem, cap):
    """step_dispatch.cuh:47-50: dynamic shared memory that leaves room for `cap` resident CTAs per SM"""
    want = (228 * KB) // (cap + 1) - KB + 256
    return want if smem < want <= 200 * KB else smem


# ------------------------------------------------------------------ games per CTA of the 10x10 and bit-plane kernels
def small_grid_G(n, sms):
    """step_c144.cu:6-13 (tile_envs_small_grid): ceil(n / (8 * SMs)) rounded up to a multiple of 16, clamped to [16, 128]"""
    g = _ceil(n, 8 * sms)
    g = (g + 15) & ~15
    return min(128, max(16, g))


def _ragged(n, G):
    while n % G == 0:
        n += 1
    return n


def n_for_small_grid(G, sms, ragged, capped=False):
    """smallest batch with tile_envs_small_grid == G, plus `ragged` games (more if needed so that the last CTA is partial).
    capped: also more than 8 CTAs per SM, the only case in which the launchers pad shared memory (step_bits.cu:352,
    step_dispatch.cuh:67); that takes G == 128 and n > 128 * 8 * SMs."""
    slots = 8 * sms
    n = (G - 16) * slots + 1 if G > 16 else 1  # ceil(n / slots) == G - 15 rounds up to G
    if capped:
        assert G == 128
        n = max(n, G * slots + 1)
    n = _ragged(n + ragged, G)
    assert small_grid_G(n, sms) == G and (not capped or _ceil(n, G) > slots)
    return n


def bits_staging_G(W, H):
    """step_bits.cu:387-389: games per CTA that ~18 KB of int8 staging holds on a board other than 10x10"""
    g = 18432 // abi.cells_per_env(W, H)
    g -= g % 16
    return min(128, max(16, g))


def bits_G(n, W, H, sms):
    """step_bits.cu:381-394 (launch_step_bits): 10x10 boards use tile_envs_small_grid; other boards cap it at ~18 KB of staging"""
    if W == 10 and H == 10:
        return small_grid_G(n, sms)
    return min(small_grid_G(n, sms), bits_staging_G(W, H))


def n_for_bits_capped(W, H, sms, ragged):
    """smallest batch at which a board other than 10x10 runs its largest G with more than 8 CTAs per SM, plus `ragged` games"""
    g = bits_staging_G(W, H)
    n = _ragged(g * 8 * sms + 1 + ragged, g)
    assert bits_G(n, W, H, sms) == g and _ceil(n, g) > 8 * sms
    return n


def bits_geometry(n, W, H, layout, dt, enc, prev, sms, slide=False, cap_opt=0):
    """step_bits.cu:338-367 (bits_smem, launch_bits_one) for a MODE_STEP call of T == 1.  prev: the caller hands back the buffer
    the env wrote last (tron_step_args.obs_prev), which takes the delta instantiation for bf16 / f32 on 10x10 boards."""
    lp, cp = _lp_cp(enc)
    C = abi.cells_per_env(W, H)
    G = bits_G(n, W, H, sms)
    w_t = 10 if (W == 10 and H == 10) else 0
    delta = prev and w_t == 10 and dt != abi.I8  # DeltaObs::kOn
    grid = _ceil(n, G)
    smem = _r16(G * C) + _r16(G) + 6 * 16  # bits_smem
    if delta:
        upp = 144 // (32 // _es(dt))  # units of 32 bytes per plane
        smem += 4 * 4 + G * 2 * lp * upp * 2
    if grid > 8 * sms:
        slide_plane = layout == "bits"
        cap = cap_opt or ((32 if lp == 1 else 5) if dt == abi.I8 else 5 if (slide_plane or delta) else 4)
        smem = smem_for_ctas_per_sm(smem, cap)
    ch8 = 8 if w_t == 10 else (4 if C % 4 == 0 else 1)  # step_bits.cu:379, 385, 392-393
    ch = 4 if (dt == abi.F32 and ch8 == 8) else ch8  # step_dispatch.cuh:42 (obs_ch)
    args = (_b(layout == "bits"), str(w_t), str(dt), str(lp), _b(cp), str(ch), "0", _b(delta))
    return Geometry("step_bits_kernel", args, G, grid, 128, smem)


# ------------------------------------------------------------------ int8-grid kernels (layout tile8)
def tile_G(n, W, H, sms):
    """step_c144.cu:14-17 for 10x10; step_generic.cu:8-16 (tile_envs_generic, TRON_OPT_TILE_BYTES at its default 18432) otherwise"""
    C = abi.cells_per_env(W, H)
    if C == 144:
        return small_grid_G(n, sms)
    g = min(128, max(1, 18432 // C))
    need = 1 if C % 16 == 0 else 2 if C % 8 == 0 else 4 if C % 4 == 0 else 8 if C % 2 == 0 else 16
    if g >= need:
        g -= g % need
    return g


def tile_geometry(n, W, H, dt, enc, sms, cap_opt=0):
    """step_dispatch.cuh:52-71 (tile_smem_bytes, launch_one) for a MODE_STEP call"""
    lp, cp = _lp_cp(enc)
    C = abi.cells_per_env(W, H)
    G = tile_G(n, W, H, sms)
    grid = _ceil(n, G)
    smem = _r16(G * C) + _r16(C) + G * 4 + G + 8 + 16 + 16 + 6 * 16
    cap = cap_opt or (5 if C == 144 else 6 if C >= 2048 else 32)  # default_tile_ctas
    if cap < 32 and grid > 8 * sms:
        smem = smem_for_ctas_per_sm(smem, cap)
    c_t, ch = (144, 8) if C == 144 else (0, 4 if C % 4 == 0 else 1)
    ch = 4 if (dt == abi.F32 and ch == 8) else ch
    args = (str(c_t), "128", str(dt), str(lp), _b(cp), str(ch), "0")
    return Geometry("step_tile_kernel", args, G, grid, 128, smem)


# ------------------------------------------------------------------ trail layout
def trail_bulk_geometry(n, W, H, dt, enc, sms):
    """step_trail.cu:632-658 (launch_trail_obs_one, bulk-store branch) -> Geometry plus (grp, nwarp, gpw): games per group, warps
    per CTA, games per warp.  A warp renders gpw / grp groups."""
    lp, cp = _lp_cp(enc)
    row = 2 * abi.enc_planes(enc) * abi.cells_per_env(W, H) * _es(dt)
    grp = 1
    while (grp * row) % 16:
        grp *= 2
    while grp < 16 and grp * row < 8192:
        grp *= 2
    wbytes = _r16(grp * row)
    assert wbytes <= 200 * KB
    nwarp = min(4, (200 * KB) // wbytes)
    smem = nwarp * wbytes
    ctas = max(1, min(6, (227 * KB) // (smem + KB)))
    gpw = n // ((8 if row >= 8192 else 3) * ctas * sms * nwarp)
    gpw = min(32, gpw)
    gpw = max(grp, gpw // grp * grp)
    G = nwarp * gpw
    geo = Geometry("step_trail_obs_bulk_kernel", (str(dt), str(lp), _b(cp), "0"), G, _ceil(n, G), 32 * nwarp, smem)
    return geo, grp, nwarp, gpw


def n_for_trail_groups(W, H, dt, enc, sms, groups, ragged):
    """smallest batch at which every warp of the bulk-store kernel renders `groups` groups, plus `ragged` games"""
    _, grp, nwarp, _ = trail_bulk_geometry(1, W, H, dt, enc, sms)
    row = 2 * abi.enc_planes(enc) * abi.cells_per_env(W, H) * _es(dt)
    smem = nwarp * _r16(grp * row)
    ctas = max(1, min(6, (227 * KB) // (smem + KB)))
    n = groups * grp * (8 if row >= 8192 else 3) * ctas * sms * nwarp + ragged
    geo, grp2, nwarp2, gpw = trail_bulk_geometry(n, W, H, dt, enc, sms)
    assert (grp2, nwarp2, gpw) == (grp, nwarp, groups * grp), (grp2, nwarp2, gpw)
    return n


def trail_fallback_geometry(n, W, H, dt, enc, sms):
    """step_trail.cu:660-669 (the element-store kernel, TRON_OPT_ENCODE_VARIANT 32): 4 warps, gpw games per warp"""
    lp, cp = _lp_cp(enc)
    C = abi.cells_per_env(W, H)
    gpw = min(32, max(1, n // (6 * 4 * sms * 4)))
    G = 4 * gpw
    args = (str(dt), str(lp), _b(cp), "4" if C % 4 == 0 else "1", "0")
    return Geometry("step_trail_obs_kernel", args, G, _ceil(n, G), 128, _r16(C)), gpw


# ------------------------------------------------------------------ state replay ring
def replay_states_geometry(k, W, H, layout, sms):
    """step_bits.cu:545-556 (launch_replay_states): G = min(32, ceil(k / (2 * SMs))) transitions per CTA"""
    G = min(32, max(1, _ceil(k, 2 * sms)))
    C = abi.cells_per_env(W, H)
    smem = 6 * 16 + _r16(G) + G * 2 * _r16(C)
    w_t = 10 if (W == 10 and H == 10) else 0
    return Geometry("replay_states_kernel", (_b(layout == "bits"), str(w_t)), G, _ceil(k, G), 128, smem)


# ------------------------------------------------------------------ the guard
def _split(name):
    """'void tron::step_bits_kernel<false, 10, 3, 1, false, 8, 0, true>(tron::StepParams)' -> ('step_bits_kernel', ('false', ...))"""
    head = name.split("(", 1)[0] if "<" not in name else name[:name.rindex(">") + 1]
    if "<" not in head:
        return head.split("::")[-1].split()[-1], ()
    base, args = head.split("<", 1)
    return base.split("::")[-1].split()[-1], tuple(a.strip() for a in args[:-1].split(","))


def launches(fn, tmp_path):
    """run fn() under torch.profiler with CUDA activity -> (fn's result, [Launch]) of the kernels it launched, from the exported
    trace's "grid", "block" and "shared memory" fields"""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    launches.n = getattr(launches, "n", 0) + 1
    path = tmp_path / ("launches_%d.json" % launches.n)
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    path.unlink()
    got = []
    launches.categories = sorted({str(e.get("cat")) for e in events})  # for the failure message of a trace without kernels
    for e in events:
        if e.get("cat") != "kernel":
            continue
        a = e["args"]
        base, targs = _split(e["name"])
        got.append(Launch(base, targs, tuple(a["grid"]), tuple(a["block"]), int(a["shared memory"])))
    return out, got


def assert_geometry(got, want, what=""):
    """exactly one launch of want.kernel, with want's template arguments, grid, block and dynamic shared memory"""
    mine = [x for x in got if x.name == want.kernel]
    assert len(mine) == 1, "%s: expected one launch of %s, got %s (trace event categories %s)" % (
        what, want.kernel, got, getattr(launches, "categories", None))
    x = mine[0]
    assert x.args == want.args, "%s: %s launched as <%s>, expected <%s>" % (what, x.name, ", ".join(x.args), ", ".join(want.args))
    assert x.grid == (want.grid, 1, 1) and x.block == (want.block, 1, 1), "%s: %s grid %s block %s, expected grid %d block %d (G = %d)" % (
        what, x.name, x.grid, x.block, want.grid, want.block, want.G)
    assert x.smem == want.smem, "%s: %s has %d B of shared memory, expected %d" % (what, x.name, x.smem, want.smem)
    return x


def guarded(fn, tmp_path, want, what=""):
    """fn() under the guard: returns fn's result after asserting the launch geometry"""
    out, got = launches(fn, tmp_path)
    assert_geometry(got, want, what)
    return out


# ------------------------------------------------------------------ the guard, in a fresh process
_PROBE = r"""
import json, pathlib, sys, tempfile
import torch
import _geometry as geo
from tron_b200 import _lib
from tron_b200.batch_env import BatchedTron
L = _lib.load()
out = []
with tempfile.TemporaryDirectory() as tmp:
    for c in json.loads(sys.argv[1]):
        for opt, val in c["options"]:
            _lib.check(L.tron_set_option(opt, val))
        env = BatchedTron(**dict(c["env"], obs_dtype=getattr(torch, c["env"]["obs_dtype"])))
        env.reset()
        _, got = geo.launches(env.step, pathlib.Path(tmp))
        out.append([list(x) for x in got])
        for opt, _ in c["options"]:
            _lib.check(L.tron_set_option(opt, 0))
print(json.dumps(out))
"""


def step_launches_in_fresh_process(configs):
    """[Launch] of one BatchedTron.step() per config ({"env": BatchedTron kwargs with obs_dtype as a torch dtype name, "options":
    [(TRON_OPT_*, value)]}), each of a freshly reset env, profiled in a new Python process.  The geometry of a step depends only on
    the configuration, the options and the batch size, so this checks the launches of an env built the same way in a process
    whose profiler has recorded nothing before.  (Late in a long test process, a torch.profiler session has been seen to record
    the launch calls but none of the kernels.)"""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([here, os.path.dirname(here)] + [p for p in [os.environ.get("PYTHONPATH")] if p]))
    r = subprocess.run([sys.executable, "-c", _PROBE, json.dumps(configs)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    return [[Launch(x[0], tuple(x[1]), tuple(x[2]), tuple(x[3]), int(x[4])) for x in got] for got in res]
